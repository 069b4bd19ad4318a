"""Training-set generation from meshes (pcgc_mesh_parse, pcgc_mesh_sample, python -m pcgcv1_b200.dataset), one JSON line (DESIGN.md
section 7, "dataset preparation" row).

    python tools/bench_dataset.py [--reps 5] [--out DIR]

On a subdivided unit icosphere of 1.31 M faces (level 8), randomly rotated:
  - sample[n, R]: for n = 10^6 / 10^7 samples on an R = 256 / 1024 grid, call_ms = one whole Codec.sample_mesh call (CUDA events
    around --reps calls after one warm-up call; it ends in the call's own synchronisation), the per-phase times of the library's
    profiler (weight / scan / sample / sort), oracle_s = oracle/meshsample.py on the host (one run), and equal = the device's
    points, samples and faces equal the oracle's bit for bit;
  - read_s: load_mesh of the mesh written as OBJ (mean of 3 reads after one);
  - cli_s_per_mesh: `python -m pcgcv1_b200.dataset` with its defaults (10^6 points, 256^3, 64^3 cubes) on 8 meshes of 50 k faces
    (a level-6 icosphere cut to 50 000 faces, each copy scaled differently), wall time of the fresh process over 8 (interpreter
    start, reading, sampling, partitioning and writing included).
The card's name and power limit are read in the same run.  Nothing is written in the repository (files go to a temporary directory)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60)
        limit = r.stdout.strip().split(",")[-1].strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def _write_obj(path, v, f):
    with open(path, "w") as fh:
        fh.write("".join("v %r %r %r\n" % tuple(p) for p in v.tolist()))
        fh.write("".join("f %d %d %d\n" % tuple(t) for t in (f + 1).tolist()))


def bench_sample(codec, v, f, n, R, rot, reps):
    import torch
    from oracle import meshsample as om
    dv, df = codec.to_device(v, torch.float64), codec.to_device(f, torch.int32)
    codec.sample_mesh(dv, df, n, 1, R, rot)
    codec.profile(True)
    for _ in range(reps):
        codec.sample_mesh(dv, df, n, 1, R, rot)
    prof = {r["tag"]: r for r in codec.profile_report()}
    codec.profile(False)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        codec.sample_mesh(dv, df, n, 1, R, rot)
    ev1.record()
    ev1.synchronize()
    call_ms = ev0.elapsed_time(ev1) / reps
    pts, samples, faces = codec.sample_mesh(dv, df, n, 1, R, rot, return_samples=True)
    t0 = time.perf_counter()
    opts, osamples, ofaces, _ = om.sample_mesh(v, f, n, 1, R, rot)
    oracle_s = time.perf_counter() - t0
    equal = bool(np.array_equal(pts.cpu().numpy(), opts) and np.array_equal(faces.cpu().numpy(), ofaces)
                 and np.array_equal(samples.cpu().numpy().view(np.uint64), osamples.view(np.uint64)))
    out = {"n": n, "resolution": R, "unique_points": int(len(opts)), "call_ms": round(call_ms, 3), "oracle_s": round(oracle_s, 3),
           "speedup_vs_oracle": round(oracle_s * 1000.0 / call_ms, 1), "equal": equal}
    for tag in ("mesh_weight", "mesh_scan", "mesh_sample", "mesh_sort"):
        out[tag + "_ms"] = round(prof[tag]["ms"] / prof[tag]["count"], 3)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="", help="also write the JSON line to DIR/bench_dataset.json")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_dataset needs a CUDA device (B200)")
    from oracle import meshsample as om
    from pcgcv1_b200 import dataset as ds, runtime
    card, limit = _card()
    res = {"card": card, "power_limit": limit, "cpu_threads": os.cpu_count()}
    codec = runtime.get_codec("voxception", "")
    v, f = om.icosphere(8)
    res["faces"] = int(len(f))
    rot = ds.random_rotation(1)
    res["sample"] = [bench_sample(codec, v, f, n, R, rot, args.reps) for n in (10 ** 6, 10 ** 7) for R in (256, 1024)]
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "ico8.obj")
        _write_obj(obj, v, f)
        ds.load_mesh(obj)
        t0 = time.perf_counter()
        for _ in range(3):
            ds.load_mesh(obj)
        res["read_s"] = round((time.perf_counter() - t0) / 3, 3)
        res["obj_mb"] = round(os.path.getsize(obj) / 1e6, 1)
        v6, f6 = om.icosphere(6)
        f6 = f6[:50_000]
        src = os.path.join(tmp, "meshes")
        os.makedirs(src)
        for k in range(8):
            _write_obj(os.path.join(src, "m%d.obj" % k), v6 * [1.0, 1.0 + 0.1 * k, 1.0 - 0.05 * k], f6)
        t0 = time.perf_counter()
        subprocess.run([sys.executable, "-m", "pcgcv1_b200.dataset", os.path.join(src, "*.obj"), os.path.join(tmp, "cubes")], cwd=ROOT,
                       check=True, stdout=subprocess.DEVNULL)
        res["cli_s_per_mesh"] = round((time.perf_counter() - t0) / 8, 3)
        res["cli_cubes"] = len([p for p in os.listdir(os.path.join(tmp, "cubes")) if p.endswith(".npy")])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_dataset.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
