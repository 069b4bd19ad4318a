"""D1 / D2 metric on the GPU against the CPU built-in, one JSON line (DESIGN.md section 7, "D1 / D2 metric" row).

    python tools/bench_metrics.py [--reps 10] [--out DIR]

For the synthetic vox10 (789 k points) and vox12 (1.78 M points) clouds: the codec compresses and decodes the cloud, the rho = 1.0
reconstruction is the B set, seeded unit normals stand in for the normals file.  Reported per cloud:
  - grid_ms / query_ms: the device metric's two phases (CUDA events of the library's profiler, mean over --reps calls after two
    warm-up calls; grids of both sets, then both directions' queries and sums);
  - call_ms: one whole pcgc_geometry_sums call (CUDA events around --reps calls);
  - candidate_ms: one candidate of the GPU-resident rho search (top-k, extraction, metric, figures to the host; host clock after a
    synchronise, mean over five candidates);
  - cpu_candidate_s: the CPU built-in on the same pair as the file-based search runs it (reconstruction written as .ply, then
    pc_error: three files read back, two k-d trees), one call;
  - speedup = cpu_candidate_s / candidate_ms.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


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


def _write_normals(path, pts, normals):
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
                "property float nx\nproperty float ny\nproperty float nz\nend_header\n" % len(pts))
        f.write("".join("%d %d %d %r %r %r\n" % (p[0], p[1], p[2], n[0], n[1], n[2]) for p, n in zip(pts.tolist(), normals.tolist())))


def bench_cloud(name, pts, reps, tmp):
    import torch
    from pcgcv1_b200 import runtime, transform
    from pcgcv1_b200.dataprocess import inout_points as iop
    from pcgcv1_b200.eval_ablation_studies import DeviceRhoSearch
    from pcgcv1_b200.models import model_voxception
    from pcgcv1_b200.myutils import pc_error_wrapper as pw
    from pcgcv1_b200.process import preprocess
    codec = runtime.get_codec("voxception", "")
    src, srcn, rec = (os.path.join(tmp, name + s) for s in (".ply", "_n.ply", "_rec.ply"))
    iop.write_ply_data(src, pts)
    rng = np.random.default_rng(0)
    normals = rng.normal(size=pts.shape)
    normals /= np.linalg.norm(normals, axis=1, keepdims=True)
    _write_normals(srcn, pts, normals)
    cubes, pos, nums = preprocess(src, 1, 64, 64, codec=codec)
    out = transform.compress_hyper(cubes, model_voxception, "")
    logits = codec.to_device(transform.decompress_hyper(*[o.numpy() for o in out], model_voxception, ""))
    search = DeviceRhoSearch(src, srcn, codec=codec)
    search.post(rec, logits, nums, pos, 1, 64, 1.0)
    a, b, n = search.input, search.points, search.normals

    for _ in range(2):
        codec.geometry_sums(a, b, n)
    torch.cuda.synchronize()
    codec.profile(True)
    for _ in range(reps):
        codec.geometry_sums(a, b, n)
    prof = {r["tag"]: r for r in codec.profile_report()}
    codec.profile(False)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        codec.geometry_sums(a, b, n)
    ev1.record()
    ev1.synchronize()
    call_ms = ev0.elapsed_time(ev1) / reps

    rhos = [0.9, 1.0, 1.05, 1.1, 1.2]
    search.post(rec, logits, nums, pos, 1, 64, rhos[0])
    search.metric(src, rec, srcn, 1024)                         # warm-up of the candidate's shapes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for rho in rhos:
        search.post(rec, logits, nums, pos, 1, 64, rho)
        search.metric(src, rec, srcn, 1024)
    candidate_ms = (time.perf_counter() - t0) * 1000.0 / len(rhos)

    search.post(rec, logits, nums, pos, 1, 64, 1.0)
    dev = search.metric(src, rec, srcn, 1024)
    t0 = time.perf_counter()
    search.write(rec)
    row = pw.pc_error(src, rec, srcn, 1024)
    cpu_s = time.perf_counter() - t0
    same_d1 = float(row["mseF,PSNR (p2point)"].iloc[0]) == dev["mseF,PSNR (p2point)"]
    return {"points_a": int(len(a)), "points_b": int(len(b)),
            "grid_ms": round(prof["geometry_grid"]["ms"] / prof["geometry_grid"]["count"], 3),
            "query_ms": round(prof["geometry_query"]["ms"] / prof["geometry_query"]["count"], 3),
            "call_ms": round(call_ms, 3), "candidate_ms": round(candidate_ms, 3), "cpu_candidate_s": round(cpu_s, 3),
            "speedup": round(cpu_s * 1000.0 / candidate_ms, 1), "d1_psnr_equal_cpu": bool(same_d1),
            "d1_psnr": dev["mseF,PSNR (p2point)"], "d2_psnr": dev["mseF,PSNR (p2plane)"]}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="", help="also write the JSON line to DIR/bench_metrics.json")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics needs a CUDA device (B200)")
    from pcgcv1_b200 import synthetic
    card, limit = _card()
    res = {"card": card, "power_limit": limit, "cpu_threads": os.cpu_count()}
    with tempfile.TemporaryDirectory() as tmp:
        res["vox10"] = bench_cloud("vox10", synthetic.cloud_vox10(0), args.reps, tmp)
        res["vox12"] = bench_cloud("vox12", synthetic.cloud_vox12(0), args.reps, tmp)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_metrics.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
