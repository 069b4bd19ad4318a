"""Factorized-prior training step (training.FactorizedTrainer, python -m pcgcv1_b200.train_factorized), one JSON line (DESIGN.md
section 7, "factorized training" row; section 4.5).

    python tools/bench_train_factorized.py [--batch 8] [--steps 10] [--reps 10] [--out DIR]

  - step[model]: one train_step (forward, backward, Adam) of model_simple and of the Voxception transforms with the factorized
    prior at --batch synthetic surface cubes: step_ms from CUDA events over --steps synchronised steps after 3 warm-up steps, the
    algorithmic GFLOP of a step (3x the forward A+S convolutions, less the first layer's data gradient, which is never computed)
    and the rate they imply; kernels = the library's per-tag profile of one further step, run on its own.
  - wgrad[layer]: the two weight-gradient forms (tile = wgrad_tile_kernel, slice = wgrad_slice_kernel, forced through
    pcgc_debug_train_wgrad) on conv_1, conv_2, deconv_2 and deconv_3 of model_simple at --batch, alternated in the same run
    (--reps pairs, CUDA events around each call, median), their partial buffers and the largest difference between their dW
    relative to its scale.
The card's name and power limit are read in the same run.  Nothing is written in the repository."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

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


def step_gflop(model: str) -> float:
    """Algorithmic GFLOP of one training step per cube: forward + data gradient + weight gradient of every convolution (3x the
    forward), less the first layer's data gradient."""
    from pcgcv1_b200 import netspec
    a, s = netspec.NETS[(model, "analysis_transform")], netspec.NETS[(model, "synthesis_transform")]
    fwd = 2.0 * (netspec.macs_per_cube(a, 64) + netspec.macs_per_cube(s, 64 // netspec.LATENT_DOWN[model]))
    return (3.0 * fwd - 2.0 * netspec.macs_per_cube(a[:1], 64)) / 1e9


def bench_step(model: str, batch: int, steps: int):
    import torch
    from pcgcv1_b200 import runtime, synthetic, training
    codec = runtime.get_codec(model, "")
    tr = training.FactorizedTrainer(codec, model=model)
    cubes = codec.to_device(synthetic.surface_cubes(batch, seed=6)[0])
    for s in range(3):
        tr.train_step(cubes, seed=s)
    codec.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        tr.train_step(cubes, seed=100 + s)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / steps
    codec.profile(True)
    tr.train_step(cubes, seed=999)
    prof = codec.profile_report()
    codec.profile(False)
    gflop = step_gflop(model) * batch
    kernels = {r["tag"]: {"count": r["count"], "ms": round(r["ms"], 3)} for r in sorted(prof, key=lambda r: -r["ms"])}
    return {"batch": batch, "step_ms": round(ms, 2), "gflop": round(gflop, 1), "tflops": round(gflop / ms, 2), "kernels": kernels}


def bench_wgrad(codec, name: str, batch: int, reps: int):
    import torch
    from pcgcv1_b200 import netspec
    l = {x.name: x for x in netspec.simple_analysis() + netspec.simple_synthesis()}[name]
    n = {"conv_1": 64, "conv_2": 32, "deconv_2": 16, "deconv_3": 32}[name]
    m = n * l.stride if l.transposed else n // l.stride
    gen = torch.Generator(device=codec.dev).manual_seed(5)
    x = torch.randn((batch, n, n, n, l.cin), device=codec.dev, generator=gen)
    g = torch.randn((batch, m, m, m, l.cout), device=codec.dev, generator=gen)
    dws = [torch.empty(netspec.kernel_shape(l), device=codec.dev) for _ in range(2)]
    used = [C.c_int64(0), C.c_int64(0)]

    def run(form):
        codec._check(codec.lib.pcgc_debug_train_wgrad(codec.ctx, form, x.data_ptr(), g.data_ptr(), batch, n, l.cin, l.cout, l.k, l.stride,
                                                      int(l.transposed), dws[form].data_ptr(), None, C.byref(used[form])))
    codec._stream()
    for form in (0, 1, 0, 1):
        run(form)
    codec.synchronize()
    times = {0: [], 1: []}
    for _ in range(reps):
        for form in (0, 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(form)
            e1.record()
            e1.synchronize()
            times[form].append(e0.elapsed_time(e1))
    a, b = dws[0].double(), dws[1].double()
    diff = float((a - b).abs().max() / a.abs().max().clamp_min(1e-30))
    macs = batch * (n if l.transposed else m) ** 3 * l.k ** 3 * l.cin * l.cout
    tile, slc = float(np.median(times[0])), float(np.median(times[1]))
    return {"batch": batch, "k": l.k, "gmac": round(macs / 1e9, 2), "tile_ms": round(tile, 3), "slice_ms": round(slc, 3),
            "speedup": round(tile / slc, 2), "slice_tflops": round(2 * macs / slc / 1e9, 2),
            "tile_partial_mb": round(used[0].value * 4 / 1e6, 1), "slice_partial_mb": round(used[1].value * 4 / 1e6, 1), "max_rel_diff": diff}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="", help="also write the JSON line to DIR/bench_train_factorized.json")
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_factorized needs a CUDA device (B200)")
    from pcgcv1_b200 import runtime
    card, limit = _card()
    res = {"card": card, "power_limit": limit, "step": {}, "wgrad": {}}
    for model in ("simple", "voxception"):
        res["step"][model] = bench_step(model, args.batch, args.steps)
    codec = runtime.get_codec("simple", "")
    for name in ("conv_1", "conv_2", "deconv_2", "deconv_3"):
        res["wgrad"][name] = bench_wgrad(codec, name, args.batch, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_train_factorized.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
