"""Point normals on the GPU (pcgc_estimate_normals) against the CPU oracle, one JSON line (DESIGN.md section 7, "point normals" row).

    python tools/bench_normals.py [--knn 30] [--reps 10] [--out DIR]

For the synthetic vox10 (789 k points) and vox12 (1.78 M points) clouds, reported per cloud:
  - grid_ms / query_ms: the two phases (CUDA events of the library's profiler, mean over --reps calls after two warm-up calls);
  - call_ms: one whole Codec.estimate_normals call (CUDA events around --reps calls);
  - cpu_s: the oracle of tests/test_gpu_normals.py on the host: cKDTree with all threads, the lowest index at the k-th distance,
    the same two-pass covariance and numpy.linalg.eigh (one run);
  - cli_s: `python -m pcgcv1_b200.normals` from .ply to _n.ply in a fresh process (interpreter start and file I/O included);
  - share_within_1e-8_rad: points whose GPU normal is within 1e-8 rad of the CPU eigenvector (up to sign);
    worst_angle_clear_rad: the largest such angle among points whose eigen-gap clears lambda1 - lambda0 > 1e-6 lambda2;
    knn_equal: the neighbour indices equal the oracle's, index for index.
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


def _sq(e):
    return (e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]


def cpu_oracle(pts, k):
    """(knn [n,m], normals [n,3], eigenvalues [n,3], eigenvectors [n,3,3]) with the kernel's neighbourhood rule and covariance."""
    from scipy.spatial import cKDTree
    n = len(pts)
    m = min(k, n)
    tree = cKDTree(pts)
    wide = min(n, 2 * m + 8)                 # enough candidates to hold every tie at the k-th distance on most points
    _, cand = tree.query(pts, k=wide, workers=-1)
    cand = cand.reshape(n, wide)
    d2 = _sq(pts[:, None, :] - pts[cand])
    order = np.lexsort((cand, d2), axis=-1)
    knn = np.take_along_axis(cand, order[:, :m], 1)
    kth = np.take_along_axis(d2, order[:, m - 1:m], 1)[:, 0]
    short = np.flatnonzero(~((d2.max(1) > kth * (1 + 1e-9) + 1e-12) | (wide == n)))
    if len(short):                           # ties run past the candidates: radius query at the k-th distance
        r = np.sqrt(kth[short]) * (1 + 1e-9) + 1e-9
        for qi, c in zip(short, tree.query_ball_point(pts[short], r, workers=-1)):
            c = np.asarray(c, np.int64)
            knn[qi] = c[np.lexsort((c, _sq(pts[qi] - pts[c])))[:m]]
    normals = np.empty((n, 3))
    w_all, v_all = np.empty((n, 3)), np.empty((n, 3, 3))
    for a in range(0, n, 200_000):
        sl = slice(a, min(a + 200_000, n))
        U = pts[knn[sl]] - pts[sl][:, None, :]
        mu = np.zeros((U.shape[0], 3))
        for j in range(m):
            mu = mu + U[:, j]
        mu = mu / m
        C = np.zeros((U.shape[0], 3, 3))
        for j in range(m):
            e = U[:, j] - mu
            C = C + e[:, :, None] * e[:, None, :]
        C = C / m
        w, v = np.linalg.eigh(C)
        w_all[sl], v_all[sl], normals[sl] = w, v, v[:, :, 0]
    return knn, normals, w_all, v_all


def bench_cloud(name, pts, k, reps, tmp):
    import torch
    from pcgcv1_b200 import runtime
    from pcgcv1_b200.dataprocess import inout_points as iop
    codec = runtime.get_codec("voxception", "")
    pts = np.ascontiguousarray(pts, np.float64)
    t = codec.to_device(pts)
    for _ in range(2):
        codec.estimate_normals(t, k)
    torch.cuda.synchronize()
    codec.profile(True)
    for _ in range(reps):
        codec.estimate_normals(t, k)
    prof = {r["tag"]: r for r in codec.profile_report()}
    codec.profile(False)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        codec.estimate_normals(t, k)
    ev1.record()
    ev1.synchronize()
    call_ms = ev0.elapsed_time(ev1) / reps
    n_gpu, knn_gpu = codec.estimate_normals(t, k, return_knn=True)
    n_gpu, knn_gpu = n_gpu.cpu().numpy(), knn_gpu.cpu().numpy()

    t0 = time.perf_counter()
    knn_cpu, n_cpu, w, _ = cpu_oracle(pts, k)
    cpu_s = time.perf_counter() - t0
    dist = np.minimum(np.linalg.norm(n_gpu - n_cpu, axis=1), np.linalg.norm(n_gpu + n_cpu, axis=1))
    angle = 2.0 * np.arcsin(np.minimum(dist / 2.0, 1.0))
    clear = w[:, 1] - w[:, 0] > 1e-6 * w[:, 2]

    src, srcn = os.path.join(tmp, name + ".ply"), os.path.join(tmp, name + "_n.ply")
    iop.write_ply_data(src, pts.astype(np.int32) if np.array_equal(pts, np.rint(pts)) else pts)
    t0 = time.perf_counter()
    subprocess.run([sys.executable, "-m", "pcgcv1_b200.normals", src, srcn, "--knn", str(k)], cwd=ROOT, check=True)
    cli_s = time.perf_counter() - t0
    return {"points": int(len(pts)), "k": k,
            "grid_ms": round(prof["normals_grid"]["ms"] / prof["normals_grid"]["count"], 3),
            "query_ms": round(prof["normals_query"]["ms"] / prof["normals_query"]["count"], 3),
            "call_ms": round(call_ms, 3), "cpu_s": round(cpu_s, 3), "cli_s": round(cli_s, 3),
            "speedup_vs_cpu": round(cpu_s * 1000.0 / call_ms, 1),
            "knn_equal": bool(np.array_equal(knn_gpu[:, :knn_cpu.shape[1]], knn_cpu)),
            "share_within_1e-8_rad": float((angle <= 1e-8).mean()), "share_clear_gap": float(clear.mean()),
            "worst_angle_clear_rad": float(angle[clear].max()) if clear.any() else 0.0}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--knn", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="", help="also write the JSON line to DIR/bench_normals.json")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_normals needs a CUDA device (B200)")
    from pcgcv1_b200 import synthetic
    card, limit = _card()
    res = {"card": card, "power_limit": limit, "cpu_threads": os.cpu_count()}
    with tempfile.TemporaryDirectory() as tmp:
        res["vox10"] = bench_cloud("vox10", synthetic.cloud_vox10(0), args.knn, args.reps, tmp)
        res["vox12"] = bench_cloud("vox12", synthetic.cloud_vox12(0), args.knn, args.reps, tmp)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_normals.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
