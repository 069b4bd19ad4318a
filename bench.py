#!/usr/bin/env python
"""Benchmark of the per-cube compress+decompress hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = hyper-mode encode + decode of every 64^3 cube of the synthetic vox10 cloud (BASELINE
config 1: ~190 cubes, ~790 k points, model_voxception, rho = 1, seeded synthetic weights) on each GPU
(cubes are independent: weak scaling, no data-path collective).

* ``value``  : cubes/s with the occupancy cubes already resident in HBM -- every GPU kernel of the
               path (analysis, hyper encoder, z quantisation, hyper decoder, Laplace quantise +
               likelihood + bits + min/max, per-element CDF intervals; then on the decode side hyper
               decoder, per-element CDF rows, synthesis, top-k classification).  The host range coder
               (the reference's sequential tail) is not in ``value``; it is in ``e2e``.
* ``e2e``    : the same metric through the public API (transform.compress_hyper ->
               transform.decompress_hyper -> select_voxels) with HOST buffers: pinned uint8 cubes in,
               byte strings + headers between, uint8 occupancy masks out; H2D/D2H copies and the multi-threaded
               host range coder inside the timed region.
* ``roofline``: the dominant kernel group of the timed region, from per-launch CUDA events recorded by
               the library on its stream (pcgc_profile_enable).
* ``cpu_baseline``: the oracle (kind "port": the TF-1.13 reference cannot run offline) on a bounded
               sample of the same cubes, driven one cube per call like the reference's tf.map_fn.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "hyper-mode encode+decode throughput of 64^3 cubes"
UNIT = "cubes/s"
GFLOP_PER_CUBE = 21.5675            # SURVEY.md section 8(d): A+HE+HD (encode) + HD+S (decode)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------ CPU baseline
def cpu_path_one_cube(oracle_mods, w, parts, cube_u8, num_points):
    """The reference's per-cube hyper path restated by the oracle (transform.py:91-259, process.py:54-66)."""
    nets, entropy, topk, W = oracle_mods
    x = cube_u8.astype(np.float32)[None]
    y = nets.run_net("voxception", "analysis", x, parts["analysis_transform"])
    z = nets.run_net("voxception", "hyper_encoder", y, parts["hyper_encoder"])
    z_hat, _ = parts["eb"](z)
    loc, scale = nets.run_net("voxception", "hyper_decoder", z_hat, parts["hyper_decoder"])
    scale = np.maximum(scale, np.float32(1e-9))
    z_str, z_min, z_max = parts["eb"].compress(z)
    sc = parts["sc"]
    y_str, y_min, y_max = sc.compress(y, loc, scale)
    # decode
    z_dec = parts["eb"].decompress(z_str, z_min, z_max, z.shape)
    loc2, scale2 = nets.run_net("voxception", "hyper_decoder", z_dec, parts["hyper_decoder"])
    scale2 = np.maximum(scale2, np.float32(1e-9))
    y_dec = sc.decompress(y_str, loc2, scale2, y_min, y_max, y.shape)
    logits = nets.run_net("voxception", "synthesis", y_dec, parts["synthesis_transform"])
    mask = topk.select_voxels(logits, [num_points], 1.0)
    return len(y_str) + len(z_str), int(mask.sum())


def run_cpu(cubes, nums, n_cubes, threads):
    import torch
    from oracle import build as obuild, entropy, nets, topk
    from pcgcv1_b200 import weights as W
    obuild.build()
    torch.set_num_threads(threads)
    w = W.synthetic_weights("voxception")
    parts = {k: W.net_weights(w, k) for k in ("analysis_transform", "synthesis_transform", "hyper_encoder", "hyper_decoder")}
    parts["eb"] = entropy.EntropyBottleneckOracle(W.net_weights(w, "estimator"))
    parts["sc"] = entropy.SymmetricConditionalOracle()
    mods = (nets, entropy, topk, W)
    t0 = time.perf_counter()
    for i in range(n_cubes):
        cpu_path_one_cube(mods, w, parts, cubes[i % len(cubes)], int(nums[i % len(cubes)]))
    return n_cubes / (time.perf_counter() - t0)


# ------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.1)

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------ GPU arm
def device_step(codec, st):
    """All GPU kernels of encode + decode on device-resident inputs, issued exactly as the product issues them
    (transform.encode_on_device / _decompress_hyper_gpu_coder: conv transforms on the main stream, the GPU range coder on the
    coder stream).  Not in here: the host range coding of the one hyper string z and the PCIe copies -- those are in ``e2e``.
    -> the step's results as device tensors, still being computed (read them after a device synchronise)."""
    from pcgcv1_b200 import transform
    eb, cem = st["eb"], st["cem"]
    codec.deferred_checks(True)
    try:
        _, mm, z_hats, _, packed, offsets, _ = transform.encode_on_device(codec, eb, cem, st["cubes"], want_likelihoods=True)
        # decode side: headers (min/max) and the strings come from the stream, z_hat from the (host) hyper decoder
        z_all = torch_cat(z_hats)
        xs = transform._decompress_hyper_gpu_coder(codec, cem, None, st["mins"], st["maxs"], [1, 16, 16, 16, 16],
                                                   lambda a, b: z_all[a:b], transform._gpu_decode_chunks(st["B"]),
                                                   uploaded=(st["packed"], st["offsets"]), sync=False)
    finally:
        codec.deferred_checks(False)
    mask, _, cnt = codec.topk(xs.raw, st["ks"])                 # same stream as the synthesis: stream order is enough
    return {"y_strings_packed": packed, "y_string_offsets": offsets, "y_minmax": mm, "z_hat": z_all, "occupancy_logits": xs.raw,
            "occupancy": mask, "voxel_counts": cnt}


# --dump-outputs: name -> (dtype written, most elements written); 62 MB in all at most.  The strings of the vox10 cloud (8.0 MB)
# fit whole, so any change of the latents shows; indices, offsets and counts are float64 so that they stay exact.
DUMP_ARRAYS = {"y_strings": (np.float32, 1 << 23), "y_string_offsets": (np.float64, 1 << 16), "y_minmax": (np.float64, 1 << 17),
               "z_hat": (np.float32, 1 << 20), "occupancy_logits": (np.float32, 1 << 21), "occupied_voxels": (np.float64, 1 << 21),
               "voxel_counts": (np.float64, 1 << 16)}
DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(out):
    """device_step's tensors (complete: after a device synchronise) -> the arrays a caller of the path receives: the strings
    (bytes, concatenated; string b = y_strings[off[b]:off[b+1]]), their offsets, the per-cube symbol ranges, the quantised
    hyper-latents, the decoded occupancy logits, the flat indices of the occupied voxels of the [B,64,64,64] masks and the
    voxels set per cube."""
    import torch
    end = int(out["y_string_offsets"][-1])
    return {"y_strings": out["y_strings_packed"][:end], "y_string_offsets": out["y_string_offsets"], "y_minmax": out["y_minmax"],
            "z_hat": out["z_hat"], "occupancy_logits": out["occupancy_logits"],
            "occupied_voxels": torch.nonzero(out["occupancy"].reshape(-1)).reshape(-1), "voxel_counts": out["voxel_counts"]}


def dump_outputs(arrays, directory):
    """Writes every array of DUMP_ARRAYS as ``directory/<name>.npy``, flattened.  An array longer than its cap is replaced by the
    elements at a fixed seeded sample of positions (kept in order; the same positions for the same length), so that two builds
    run with the same arguments can be compared element for element."""
    import torch
    os.makedirs(directory, exist_ok=True)
    total = 0
    for name, (dtype, cap) in DUMP_ARRAYS.items():
        t = arrays[name].reshape(-1)
        if t.numel() > cap:
            pos = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t[torch.from_numpy(pos).to(t.device)]
        a = t.cpu().numpy().astype(dtype)
        np.save(os.path.join(directory, name + ".npy"), a)
        total += a.nbytes
    assert total <= DUMP_LIMIT_BYTES, total


def device_step_transforms(codec, st):
    """The r01 definition of ``value`` for comparison across rounds: every transform / entropy-model / top-k kernel of encode +
    decode, WITHOUT the range coder (r01 ran it on the host, outside ``value``)."""
    B = st["B"]
    y = codec.analysis(st["cubes"])
    z = codec.hyper_encode(y)
    z_hat, _, _, _ = codec.factorized(0, z, want_p=True, want_bits=True)
    loc, scale = codec.hyper_decode(z_hat, 1e-9)
    y2, l2, s2 = y.reshape(B, -1), loc.reshape(B, -1), scale.reshape(B, -1)
    y_hat, _, _, mm = codec.laplace(y2, l2, s2, want_p=True, want_bits=True)
    codec.laplace_intervals(y_hat, l2, s2, mm)
    loc_d, scale_d = codec.hyper_decode(z_hat, 1e-9)
    codec.laplace_cdf(loc_d.reshape(B, -1), scale_d.reshape(B, -1), st["minmax_host"])
    logits = codec.synthesis(y_hat.reshape(y.shape))
    return codec.topk(logits, st["ks"])


def torch_cat(parts):
    import torch
    return torch.cat(parts) if len(parts) > 1 else parts[0]


def e2e_step(st):
    from pcgcv1_b200 import transform
    from pcgcv1_b200.dataprocess import inout_points
    from pcgcv1_b200.models import model_voxception
    out = transform.compress_hyper(st["cubes_host"], model_voxception, "")
    host = [o.numpy() for o in out]
    xs = transform.decompress_hyper(*host, model_voxception, "")
    mask = inout_points.select_voxels(xs, st["nums"], 1.0, codec=st["codec"], dtype="uint8")
    return host, mask


def config1(args, cubes_per_gpu, points_per_gpu):
    """The `config` object of BASELINE config 1, printed identically by the CUDA arm and by --impl reference."""
    return {"workload": "%s synthetic cloud, %d cubes of 64^3 (%d points) per GPU, hyper mode, model_voxception, rho=1.0, "
                        "seeded synthetic weights" % (args.workload, cubes_per_gpu, int(points_per_gpu)),
            "cubes_per_gpu": int(cubes_per_gpu), "points_per_gpu": int(points_per_gpu),
            "l2": "inputs+activations per step >> 126 MB L2 (no flush needed)",
            "range_coder": os.environ.get("PCGC_CODER", "gpu"),
            "e2e_flow": "compress_hyper -> .numpy() of every stream field -> decompress_hyper (returns a pending device result once "
                        "its last kernel is queued) -> select_voxels(codec=, dtype=uint8): top-k on the GPU and the uint8 masks to "
                        "the host part by part behind the synthesis (the reference does .numpy() then NumPy top-k, test.py:115)",
            "decode_schedule": os.environ.get("PCGC_DEC_RAMP", "8,24,64") + " cubes, then the rest",
            "conv_engine": os.environ.get("PCGC_ENGINE", "auto"),
            "far_field_tiles": "off" if os.environ.get("PCGC_FARFIELD", "1") == "0" else "on (analysis K_b16: tiles without an occupied voxel in "
                               "their receptive field are copied from the empty cube's activations, bit-identical)"}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from pcgcv1_b200 import runtime, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    cubes, pos, nums = synthetic.workload(args.workload, seed=0, max_cubes=args.cubes)
    B = len(cubes)
    codec = runtime.get_codec("voxception", "", local)
    pinned = torch.from_numpy(cubes).pin_memory()
    st = {"B": B, "codec": codec, "nums": nums, "cubes_host": pinned, "cubes": pinned.to(codec.dev),
          "ks": torch.from_numpy(nums.astype(np.int32)).to(codec.dev)}
    # the stream (headers + strings) the device-resident decode leg reads: what compress wrote, already uploaded
    from pcgcv1_b200 import transform
    from pcgcv1_b200.models.conditional_entropy_model import SymmetricConditional
    st["eb"] = transform._bottleneck(codec, 8)
    st["cem"] = SymmetricConditional().bind(codec)
    _, mm_all, _, _, packed, offsets, _ = transform.encode_on_device(codec, st["eb"], st["cem"], st["cubes"])
    torch.cuda.synchronize()
    codec.synchronize()
    mm = mm_all.cpu().numpy()
    st["mins"], st["maxs"] = mm[:, 0].copy(), mm[:, 1].copy()
    st["minmax_host"] = mm
    st["packed"], st["offsets"] = packed, offsets

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = a.elapsed_time(b)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=codec.dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    sampler = ClockSampler(local)
    sampler.start()
    # ---- device-resident hot path (value) with per-launch events for the roofline ----
    for _ in range(args.warmup):
        device_step(codec, st)
    codec.profile(True)
    codec.profile_report()
    l0 = codec.launch_count()
    last = {}

    def value_step():
        last["out"] = device_step(codec, st)
    dev_ms, _ = timed(value_step, args.steps, 0)
    launches = codec.launch_count() - l0
    prof = codec.profile_report()
    codec.profile(False)
    clocks = sampler.finish()
    out = last.pop("out")
    if args.dump_outputs and rank == 0:
        codec.synchronize()                                     # raises if a kernel of the timed steps flagged an error
        dump_outputs(step_outputs(out), args.dump_outputs)
    del out
    # the same kernels without the range coder (the r01 definition of value, for comparison across rounds)
    nocoder_steps = max(3, args.steps // 2)
    nocoder_ms, _ = timed(lambda: device_step_transforms(codec, st), nocoder_steps, 1)
    # ---- end to end through the public API with host buffers ----
    runtime.COUNTERS["h2d_bytes"] = runtime.COUNTERS["d2h_bytes"] = 0
    e2e_steps = args.steps
    _, e2e_wall_ms = timed(lambda: e2e_step(st), e2e_steps, 1)
    h2d = runtime.COUNTERS["h2d_bytes"] // (e2e_steps + 1)
    d2h = runtime.COUNTERS["d2h_bytes"] // (e2e_steps + 1)

    if world > 1:
        lt = torch.tensor([launches], dtype=torch.int64, device=codec.dev)
        dist.all_reduce(lt)
        launches = int(lt[0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    value = world * B * args.steps / (dev_ms / 1e3)
    e2e = world * B * e2e_steps / (e2e_wall_ms / 1e3)
    points = float(nums.sum())
    # dominant kernel group.  The GPU range-coder kernels (one warp per cube, latency-bound, on the coder streams BESIDE the conv
    # kernels) have their own entry below: their event times overlap the main stream's and say nothing about a roofline.
    prof.sort(key=lambda r: -r["ms"])
    total_ms = sum(r["ms"] for r in prof)
    main_prof = [r for r in prof if not r["tag"].startswith("range_")]
    top = main_prof[0]
    per_launch_ms = top["ms"] / top["count"]
    per_launch = int(os.environ.get("PCGC_SUB_BATCH", "64"))          # cubes per kernel launch in this run
    tr = None
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                tr = json.load(f).get(top["tag"])
            if tr:
                tr.setdefault("source", "profiles/" + name)
                break
        except (OSError, ValueError):
            pass
    if top["flops"] > 0:
        # SURVEY.md 8(d): the conv transforms are bounded by the TENSOR roofline on algorithmic FLOPs (split-bf16 passes, padded
        # columns and halo recompute do not count).  The HBM picture stays beside it: DRAM bytes from the ncu capture over the same
        # launch time, against the bytes a fused Voxception block would need (read x once, write out once).
        ach = top["flops"] / top["count"] / (per_launch_ms * 1e-3) / 1e12
        roof = {"kernel": top["tag"], "bound": "tensor", "achieved": round(ach, 3), "peak": peaks["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": round(ach / peaks["bf16_tflops_sustained"], 5), "traffic": None,
                "frac_of_burst_peak": round(ach / peaks["bf16_tflops"], 5), "peak_nominal": 2250.0}
        if tr:
            # cubes per launch as this run issued them (the decode ramp launches 8 / 24 / 64-cube batches): from the launch's
            # algorithmic FLOPs; the ncu capture's bytes scale with the cubes
            if tr.get("algorithmic_flops_per_cube"):
                per_launch = top["flops"] / top["count"] / tr["algorithmic_flops_per_cube"]
                roof["cubes_per_launch_avg"] = round(per_launch, 2)
            scale = per_launch / tr.get("cubes_per_launch", per_launch)
            per_capture = tr["dram_bytes_per_launch"]
            if os.environ.get("PCGC_FARFIELD", "1") == "0":          # every tile computed: the capture without far-field copies
                per_capture = tr.get("dram_bytes_per_launch_all_tiles_computed", per_capture)
            traffic = per_capture * scale
            roof["traffic"] = int(traffic)
            roof["traffic_source"] = tr["source"]
            hbm = {"achieved_gbs": round(traffic / (per_launch_ms * 1e-3) / 1e9, 1), "peak_gbs": peaks["hbm_gbs"]}
            hbm["frac"] = round(hbm["achieved_gbs"] / peaks["hbm_gbs"], 4)
            if tr.get("algorithmic_bytes_per_launch"):
                hbm["kernel_algorithmic_bytes"] = int(tr["algorithmic_bytes_per_launch"] * scale)
            if tr.get("fused_block_floor_bytes_per_cube"):
                hbm["fused_block_floor_bytes"] = int(tr["fused_block_floor_bytes_per_cube"] * per_launch)
                hbm["block_traffic_over_fused_floor"] = tr.get("block_traffic_over_fused_floor")
            roof["hbm"] = hbm
            for k in ("sm__pipe_tc_cycles_active_pct", "utchmma_bf16_ops_pct_of_peak", "l1tex_tc_wavefronts_shared_pct_of_peak"):
                if k in tr:
                    roof["ncu_" + k] = tr[k]
    else:
        ach = top["bytes"] / top["count"] / (per_launch_ms * 1e-3) / 1e9
        roof = {"kernel": top["tag"], "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm_gbs"], 5), "traffic": int(tr["dram_bytes_per_launch"]) if tr else None, "peak_nominal": 8000.0}
    roof.update({"peak_source": peaks["source"], "ms_per_launch": round(per_launch_ms, 4), "share_of_step": round(top["ms"] / total_ms, 4)})
    coder = [{"tag": r["tag"], "launches_per_step": r["count"] // max(1, args.steps), "ms_per_launch": round(r["ms"] / r["count"], 3),
              "ns_per_symbol_of_one_cube": round(r["ms"] / r["count"] * 1e6 / 65536, 1),
              "note": "one warp per cube, sequential in the string: latency-bound, runs beside the conv kernels"}
             for r in prof if r["tag"].startswith("range_")]
    conv_ms = sum(r["ms"] for r in prof if r["tag"].startswith("conv"))
    conv_tflops = sum(r["flops"] for r in prof if r["tag"].startswith("conv")) / (conv_ms * 1e-3) / 1e12
    kernels = [{"tag": r["tag"], "share": round(r["ms"] / total_ms, 4),
                "achieved": round((r["flops"] / 1e12 if r["flops"] else r["bytes"] / 1e9) / (r["ms"] * 1e-3), 2),
                "unit": "TFLOP/s" if r["flops"] else "GB/s"} for r in prof[:16]]
    # memory-bound kernels (entropy models, top-k, voxel I/O): achieved algorithmic GB/s against the measured HBM peak, whatever their rank
    hbm_kernels = [{"tag": r["tag"], "share": round(r["ms"] / total_ms, 4), "achieved_gbs": round(r["bytes"] / 1e9 / (r["ms"] * 1e-3), 1),
                    "frac_of_hbm_peak": round(r["bytes"] / 1e9 / (r["ms"] * 1e-3) / peaks["hbm_gbs"], 4)}
                   for r in prof if not r["flops"] and r["bytes"] and r["ms"] > 0 and not r["tag"].startswith("range_")]
    # ---- CPU baseline (rank 0, N=1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        n_cpu = args.cpu_cubes
        v = run_cpu(cubes, nums, n_cpu, cores)
        cpu = {"value": round(v, 4), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d cubes of the same cloud, one cube per call, torch-CPU fp32 convs + NumPy entropy + C range coder" % n_cpu}
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dev_ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config1(args, B, points),
        "points_per_s": round(value * points / B, 1),
        "value_without_range_coder": {"value": round(world * B * nocoder_steps / (nocoder_ms / 1e3), 2), "unit": UNIT, "steps": nocoder_steps,
                                      "note": "r01's definition of value (range coder on the host, outside the timed kernels); `value` above "
                                              "includes the GPU range-coder kernels on the coder streams"},
        "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "points_per_s": round(e2e * points / B, 1), "steps": e2e_steps, "host_threads": runtime.coder_threads()},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
        "conv": {"achieved_tflops": round(conv_tflops, 2), "share_of_step": round(conv_ms / total_ms, 4),
                 "algorithmic_gflop_per_cube": GFLOP_PER_CUBE,
                 "frac_of_bf16_sustained": round(conv_tflops / peaks["bf16_tflops_sustained"], 5)},
        "kernels": kernels, "hbm_kernels": hbm_kernels, "gpu_range_coder": coder, "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------ other BASELINE configs
def _dist_setup(args):
    """(world, rank, local, host_group): NCCL for the timing barriers on N > 1, a gloo group for the host-object exchange."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")
    else:
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1)
        host_group = None
    return world, rank, local, host_group


def run_sharded(args):
    """BASELINE config 3: the sparse vox12 cloud (thousands of 64^3 cubes), hyper mode, STRONG scaling: the cloud's cubes are
    split into contiguous slices over the ranks (pcgcv1_b200.sharding), no data-path collective; the exchange is a host-side
    gather of strings / headers / quantised hyper-latents to rank 0, ONE global range coding of z there (the reference's format
    has a single z string for the whole cloud, entropy_model.py:249-259) and the gather of the decoded points."""
    import torch
    import torch.distributed as dist
    from pcgcv1_b200 import runtime, sharding, synthetic
    world, rank, local, hg = _dist_setup(args)
    cubes, pos, nums = synthetic.workload("vox12", seed=0, max_cubes=args.cubes)
    B = len(cubes)
    a, b = sharding.shard_slices(B, world)[rank]
    lc = sharding.GpuLocalCodec("voxception", "", local)
    mine_host = torch.from_numpy(cubes[a:b]).pin_memory()
    mine_dev = mine_host.to(lc.codec.dev)
    result = {}

    def step(x):
        stream = sharding.compress_sharded(x, lc, group=hg)
        out = sharding.decompress_sharded(stream, nums if rank == 0 else None, 1.0, lc, group=hg, output="points")
        if rank == 0:
            result["stream"], result["points"] = stream, out

    def timed(x, steps, warmup):
        for _ in range(warmup):
            step(x)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step(x)
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=lc.codec.dev if world > 1 else "cpu")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    sampler = ClockSampler(local)
    sampler.start()
    l0 = lc.codec.launch_count()
    dev_ms = timed(mine_dev, args.steps, max(1, min(args.warmup, 2)))
    launches = lc.codec.launch_count() - l0
    clocks = sampler.finish()
    runtime.COUNTERS["h2d_bytes"] = runtime.COUNTERS["d2h_bytes"] = 0
    e2e_ms = timed(mine_host, args.steps, 0)
    h2d, d2h = runtime.COUNTERS["h2d_bytes"] // args.steps, runtime.COUNTERS["d2h_bytes"] // args.steps
    if rank == 0:
        pts, counts = result["points"]
        stream = result["stream"]
        import hashlib
        y_bytes = stream["y_blob"].tobytes() if "y_blob" in stream else b"".join(stream["y_strings"])
        digest = hashlib.sha256(y_bytes + stream["z_string"]).hexdigest()[:16]
        line = {
            "metric": "hyper-mode encode+decode throughput of 64^3 cubes, one cloud sharded over the GPUs", "value": round(B * args.steps / (dev_ms / 1e3), 2),
            "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 2),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "vox12 synthetic sparse cloud, %d cubes of 64^3 (%d points) in total, contiguous slices per GPU, hyper mode, "
                                   "model_voxception, rho=1.0, seeded synthetic weights" % (B, int(nums.sum())),
                       "baseline_config": 3, "cubes_total": B, "points_total": int(nums.sum()), "range_coder": os.environ.get("PCGC_CODER", "gpu"),
                       "exchange": "host-side gather of strings/headers/z_hat to rank 0 (gloo), one global z string coded there, points gathered back; "
                                   "no collective on the data path"},
            "points_per_s": round(float(nums.sum()) * args.steps / (dev_ms / 1e3), 1),
            "e2e": {"value": round(B * args.steps / (e2e_ms / 1e3), 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "note": "h2d/d2h of rank 0 only; value = cube slices resident in HBM, e2e = slices in pinned host memory"},
            "gpu_launches": int(launches) * world, "clocks": clocks,
            "stream_sha256_16": digest, "stream_bytes": int(len(y_bytes) + len(stream["z_string"])),
            "decoded_points": int(len(pts)), "decoded_ge_input_points": bool((counts >= nums).all()),
            "roofline": None, "cpu_baseline": None,
        }
        print(json.dumps(line))
    dist.destroy_process_group()


def run_factorized(args):
    """BASELINE config 2: the vox10 cloud in factorized mode (EntropyBottleneck only) with model_simple on one GPU."""
    import torch
    from pcgcv1_b200 import runtime, synthetic, transform
    from pcgcv1_b200.dataprocess import inout_points
    from pcgcv1_b200.models import model_simple
    torch.cuda.set_device(0)
    cubes, pos, nums = synthetic.workload("vox10", seed=0, max_cubes=args.cubes)
    B = len(cubes)
    codec = runtime.get_codec("simple", "", 0)
    pinned = torch.from_numpy(cubes).pin_memory()
    xd = pinned.to(codec.dev)
    ks = torch.from_numpy(nums.astype(np.int32)).to(codec.dev)
    slot = codec.bottleneck_slot(32)

    def device_step():
        y = codec.analysis(xd)
        y_hat, _, _, _ = codec.factorized(slot, y, want_p=True, want_bits=True)
        logits = codec.synthesis(y_hat)
        return codec.topk(logits, ks)

    def e2e_step():
        s, mn, mx, shp = transform.compress_factorized(pinned, model_simple, "")
        xs = transform.decompress_factorized(s.numpy(), mn.numpy(), mx.numpy(), shp.numpy(), model_simple, "")
        return s, inout_points.select_voxels(xs, nums, 1.0, codec=codec, dtype="uint8")

    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(args.warmup):
        device_step()
    codec.profile(True); codec.profile_report()
    l0 = codec.launch_count()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        device_step()
    b.record(); torch.cuda.synchronize()
    dev_ms = a.elapsed_time(b)
    launches = codec.launch_count() - l0
    prof = codec.profile_report(); codec.profile(False)
    clocks = sampler.finish()
    e2e_step()
    runtime.COUNTERS["h2d_bytes"] = runtime.COUNTERS["d2h_bytes"] = 0
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(args.steps):
        s, mask = e2e_step()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    peaks = load_peaks()
    prof.sort(key=lambda r: -r["ms"])
    total_ms = sum(r["ms"] for r in prof)
    top = prof[0]
    ach = top["flops"] / (top["ms"] * 1e-3) / 1e12 if top["flops"] else 0.0
    GF = 5.4169                      # SURVEY.md 8(d): factorized simple enc+dec GFLOP per cube
    line = {
        "metric": "factorized-mode encode+decode throughput of 64^3 cubes (model_simple)", "value": round(B * args.steps / (dev_ms / 1e3), 2), "unit": UNIT,
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "vox10 synthetic cloud, %d cubes of 64^3 (%d points), factorized mode, model_simple, rho=1.0, seeded synthetic weights"
                               % (B, int(nums.sum())), "baseline_config": 2, "cubes_per_gpu": B},
        "e2e": {"value": round(B * args.steps / (e2e_ms / 1e3), 2), "unit": UNIT, "h2d_bytes_per_step": runtime.COUNTERS["h2d_bytes"] // args.steps,
                "d2h_bytes_per_step": runtime.COUNTERS["d2h_bytes"] // args.steps, "string_bytes": len(s.numpy())},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"kernel": top["tag"], "bound": "tensor", "achieved": round(ach, 3), "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": round(ach / peaks["bf16_tflops_sustained"], 5), "traffic": None, "share_of_step": round(top["ms"] / total_ms, 4),
                     "note": "model_simple: conv_1 / conv_2 / deconv_2 / deconv_3 on the tcgen05 window-GEMM kernel (umma_win.cu); the two 8^3 "
                             "layers (conv_3, deconv_1; 4.8 % of the MACs each way) on the exact-FP32 CUDA-core kernel"},
        "conv": {"achieved_tflops": round(GF * B * args.steps / (dev_ms / 1e3) / 1e3, 2), "algorithmic_gflop_per_cube": GF},
        "kernels": [{"tag": r["tag"], "share": round(r["ms"] / total_ms, 4)} for r in prof[:8]], "cpu_baseline": None,
    }
    print(json.dumps(line))


def run_sweep(args):
    """BASELINE config 4: analysis + synthesis only, batch 8..512 cubes of 64^3, steady state, CUDA events."""
    import torch
    from pcgcv1_b200 import runtime, synthetic
    torch.cuda.set_device(0)
    codec = runtime.get_codec("voxception", "", 0)
    base, _ = synthetic.surface_cubes(8, seed=3)
    peaks = load_peaks()
    GF = 20.7996                     # SURVEY.md 8(d): analysis + synthesis GFLOP per cube
    sweep = {}
    sampler = ClockSampler(0)
    sampler.start()
    l0 = codec.launch_count()
    for B in (8, 16, 32, 64, 128, 256, 512):
        x = codec.to_device(np.tile(base, (B // 8, 1, 1, 1, 1)))
        y = torch.round(codec.analysis(x))
        for _ in range(5):
            codec.analysis(x); codec.synthesis(y)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        it = max(args.steps, 20) if B <= 128 else max(args.steps // 2, 8)
        torch.cuda.synchronize()
        a.record()
        for _ in range(it):
            codec.analysis(x); codec.synthesis(y)
        b.record(); torch.cuda.synchronize()
        ms = a.elapsed_time(b) / it
        sweep[str(B)] = {"ms": round(ms, 3), "cubes_per_s": round(B / ms * 1e3, 1), "tflops": round(B * GF / ms, 2),
                         "frac_of_bf16_sustained": round(B * GF / ms / peaks["bf16_tflops_sustained"], 5)}
        del x, y
    clocks = sampler.finish()
    best = sweep["64"]
    line = {
        "metric": "analysis+synthesis transform throughput of 64^3 cubes (batch sweep)", "value": best["cubes_per_s"], "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": 5, "ms_per_step": best["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "random smooth-surface cubes of 64^3, analysis + synthesis of model_voxception only, batches 8..512 (value: batch 64)",
                   "baseline_config": 4, "l2": "activations per batch >> 126 MB L2 for B >= 8"},
        "sweep": sweep, "gpu_launches": int(codec.launch_count() - l0), "clocks": clocks,
        "roofline": {"kernel": "analysis+synthesis (all conv kernels)", "bound": "tensor", "achieved": best["tflops"], "peak": peaks["bf16_tflops_sustained"],
                     "unit": "TFLOP/s", "frac": best["frac_of_bf16_sustained"], "traffic": None},
        "e2e": None, "cpu_baseline": None,
    }
    print(json.dumps(line))


def run_train(args):
    """BASELINE config 5: train_hyper.py step (alpha = 0.75, beta = 3, gamma = delta = 1, lr = 1e-5, batch 8 cubes of 64^3, BCE
    occupancy loss, noise quantisation), forward + backward + Adam.  N > 1: data parallel, one batch of 8 per GPU, gradients
    averaged with one NCCL all-reduce (weak scaling)."""
    import torch
    import torch.distributed as dist
    from pcgcv1_b200 import runtime, synthetic, training
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    codec = runtime.get_codec("voxception", "", local)
    B = 8
    cubes, _ = synthetic.surface_cubes(B, seed=100 + rank)
    tr = training.HyperTrainer(codec, alpha=0.75, beta=3.0, gamma=1.0, delta=1.0, lr=1e-5, distortion=args.distortion)
    pinned = torch.from_numpy(cubes).pin_memory()
    xd = pinned.to(codec.dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        tr.train_step(xd, seed=i)
    codec.profile(True); codec.profile_report()
    l0 = codec.launch_count()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(args.steps):
        out = tr.train_step(xd, seed=1000 + i)
    b.record()
    barrier()
    dev_ms = a.elapsed_time(b)
    launches = codec.launch_count() - l0
    prof = codec.profile_report(); codec.profile(False)
    clocks = sampler.finish()
    terms = tr.loss_terms(out)
    # end to end: the batch comes from pinned host memory every step and the loss terms go back to the host
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = tr.train_step(pinned, seed=2000 + i)
        terms = tr.loss_terms(out)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=codec.dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    if rank == 0:
        peaks = load_peaks()
        GF = 3 * 21.217                                   # SURVEY.md 8(d): fwd 21.217 GFLOP per cube, bwd ~ 2x fwd
        prof.sort(key=lambda r: -r["ms"])
        total_ms = sum(r["ms"] for r in prof) or 1.0
        steps_s = world * args.steps / (dev_ms / 1e3)
        tfl = GF * B * steps_s / 1e3
        line = {
            "metric": "train_hyper.py step throughput (forward + backward + Adam)", "value": round(steps_s * B, 2), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(dev_ms / args.steps, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "train_hyper.py step: batch 8 cubes of 64^3 per GPU, alpha=0.75 beta=3 gamma=delta=1, lr=1e-5, %s, "
                                   "noise quantisation (seeded Philox), random smooth-surface cubes, seeded synthetic weights"
                                   % ("focal occupancy loss (loss.py:83-93, gamma 2, alpha 0.9, sum) on sigmoid(x_tilde)" if args.distortion == "focal"
                                      else "BCE occupancy loss (loss.py:8-33, what train_hyper.py calls)"),
                       "baseline_config": 5, "batch_per_gpu": B, "engine": "exact FP32 CUDA cores (conv_ffma.cu + train.cu), deterministic"},
            "steps_per_s": round(steps_s, 3),
            "e2e": {"value": round(world * args.steps * B / (e2e_ms / 1e3), 2), "unit": UNIT, "h2d_bytes_per_step": int(pinned.numel()),
                    "d2h_bytes_per_step": 48, "note": "batch from pinned host memory, loss terms read back every step"},
            "gpu_launches": int(launches) * world, "clocks": clocks, "loss_terms_last_step": terms,
            "roofline": {"kernel": prof[0]["tag"], "bound": "tensor", "achieved": round(tfl, 2), "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": round(tfl / peaks["bf16_tflops_sustained"], 5), "traffic": None,
                         "note": "whole step on algorithmic FLOPs (3 x forward); the training path runs on FP32 CUDA cores, not on tcgen05"},
            "kernels": [{"tag": r["tag"], "share": round(r["ms"] / total_ms, 4), "ms_per_step": round(r["ms"] / args.steps, 2)} for r in prof[:6]],
            "cpu_baseline": None,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """Reference arm: the reference's own CPU path.  TF 1.13 cannot be installed offline, so this is the
    oracle port driven exactly as transform.py drives TF (one cube per call), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pcgcv1_b200 import synthetic
    cubes, pos, nums = synthetic.workload(args.workload, seed=0, max_cubes=args.cubes)
    cores = os.cpu_count() or 1
    per_step = args.cpu_cubes
    for _ in range(min(args.warmup, 1)):
        run_cpu(cubes, nums, 1, cores)
    t0 = time.perf_counter()
    for s in range(args.steps):
        run_cpu(cubes[s * per_step:], nums[s * per_step:], per_step, cores)
    dt = time.perf_counter() - t0
    v = args.steps * per_step / dt
    sample = "%d cubes of the %s cloud per step, one cube per call" % (per_step, args.workload)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # exactly the CUDA arm's config object (the step here is a bounded sample of that workload: see cpu_baseline.sample)
        "config": config1(args, len(cubes), int(nums.sum())),
        "note": "TF 1.13 reference not installable offline: CPU oracle port of the same path, one cube per call",
        "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vox10", choices=["vox10", "vox12"])
    ap.add_argument("--cubes", type=int, default=None, help="limit the number of cubes (debug)")
    ap.add_argument("--cpu-cubes", type=int, default=6, help="cubes in the CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json config: 1 vox10 hyper (default, the headline), 2 vox10 factorized + model_simple, "
                         "3 vox12 cloud sharded over --gpus (strong scaling), 4 analysis+synthesis batch sweep, 5 training step (batch 8)")
    ap.add_argument("--distortion", default="bce", choices=["bce", "focal"],
                    help="config 5: occupancy loss of the training step (bce = what train_hyper.py calls; focal = loss.py:83-93)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="config 1: write what the last timed step computed (strings, symbol ranges, hyper-latents, occupancy "
                         "logits and masks) as DIR/<name>.npy, float32 / float64, a seeded sample of the larger ones, <= 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 1 or args.impl != "ours"):
        ap.error("--dump-outputs applies to --config 1 with --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        import __graft_entry__
        __graft_entry__.build()
        {1: run_gpu, 2: run_factorized, 3: run_sharded, 4: run_sweep, 5: run_train}[args.config](args)


if __name__ == "__main__":
    main()
