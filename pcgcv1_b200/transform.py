"""Drop-in for the reference's ``transform.py``: ``compress_factorized`` / ``decompress_factorized`` /
``compress_hyper`` / ``decompress_hyper`` with the reference's signatures and return tuples
(transform.py:24-56,58-87,91-197,200-259).  Every returned value has ``.numpy()`` because the
callers (test.py:81,89,101-103,115; eval.py:56-57,87-89) call it.

What changes underneath: the per-cube ``tf.map_fn(..., parallel_iterations=1)`` loops
(transform.py:48,84,122,131,143,166,183,193,230,247,256) become one batched call per net into
libpcgc_b200.so; quantisation / likelihood / per-element CDF rows are fused GPU kernels; only the
range coder runs on the host (thread pool over cubes).  The hyper decoder is bit-reproducible, so a
stream written by ``compress_hyper`` decodes with ``decompress_hyper`` (the reference's GPU path
does not guarantee that: README.md:111-114).
"""
from __future__ import annotations

import os
import time

import numpy as np
import torch

from . import runtime
from .models.conditional_entropy_model import SymmetricConditional
from .models.entropy_model import EntropyBottleneck

_VERBOSE = bool(int(os.environ.get("PCGC_VERBOSE", "0")))


def _log(msg, start=None):
    if _VERBOSE:
        if start is not None:
            torch.cuda.synchronize()
            print("{}: {}s".format(msg, round(time.time() - start, 4)))
        else:
            print(msg)


TRACE = None        # dev hook (tools/host_trace.py): a list that collects (perf_counter, label) marks of the pipelines below


def _tr(label):
    if TRACE is not None:
        TRACE.append((time.perf_counter(), label))


def _strings_array(strings):
    a = np.empty(len(strings), dtype=object)
    for i, s in enumerate(strings):
        a[i] = s
    return a


def _as_list_of_bytes(strings):
    strings = runtime.unwrap(strings)
    if isinstance(strings, (bytes, bytearray)):
        return [bytes(strings)]
    return [bytes(s) for s in list(strings)]


def _bottleneck(codec, channels):
    return EntropyBottleneck().bind(codec, codec.bottleneck_slot(channels))


# ---------------------------------------------------------------- factorized entropy model
def compress_factorized(cubes, model, ckpt_dir):
    """cubes [B,64,64,64,1] -> (strings, min_v, max_v, shape)  (transform.py:24-56)."""
    _log("===== Compress =====")
    codec = runtime.get_codec(model, ckpt_dir)
    x = codec.to_device(cubes)
    start = time.time()
    ys = codec.analysis(x)
    _log("Analysis Transform", start)
    start = time.time()
    strings, min_v, max_v = _bottleneck(codec, ys.shape[-1]).compress(ys)
    shape = runtime.HostResult(np.array(ys.shape, dtype=np.int32))
    _log("Entropy Encode", start)
    return strings, min_v, max_v, shape


def decompress_factorized(strings, min_v, max_v, shape, model, ckpt_dir):
    """-> xs [B,64,64,64,1] occupancy logits  (transform.py:58-87)."""
    _log("===== Decompress =====")
    codec = runtime.get_codec(model, ckpt_dir)
    shape = np.asarray(runtime.unwrap(shape)).reshape(-1)
    start = time.time()
    B = int(shape[0])
    if B <= _FACT_PART or _VERBOSE:
        ys = _bottleneck(codec, int(shape[-1])).decompress(strings, min_v, max_v, shape, shape[-1])
        _log("Entropy Decode", start)
        start = time.time()
        xs = codec.synthesis(ys.tensor)
        _log("Synthesis Transform", start)
        return runtime.DeviceResult(xs)
    # The ONE string (global range, entropy_model.py:249-259) is sequential and decodes on a host thread (~12 ns per symbol);
    # the cubes come out of it in order, so the synthesis of cubes [a, b) runs while the string's tail is still being read,
    # and the caller gets a pending result whose parts select_voxels can consume as they finish.
    get = _bottleneck(codec, int(shape[-1])).decompress_progressive(strings, min_v, max_v, shape, shape[-1])
    main = torch.cuda.current_stream(codec.dev)
    xs = torch.empty([B, 64, 64, 64, 1], dtype=torch.float32, device=codec.dev)
    parts = []
    codec.deferred_checks(True)
    try:
        for a in range(0, B, _FACT_PART):
            b = min(B, a + _FACT_PART)
            codec.synthesis(get(a, b), out=xs[a:b])
            ev = torch.cuda.Event()
            ev.record(main)
            parts.append((a, b, ev))
    finally:
        codec.deferred_checks(False)
    return runtime.PendingDeviceResult(xs, parts, codec, parts[-1][2])


# ---------------------------------------------------------------- hyperprior (conditional) model
# The batch is processed in chunks as a two-stage software pipeline: while the host range coder (worker thread; the C
# entry points release the GIL and fan out over their own thread pool) works on chunk k, the GPU already runs the
# transforms of chunk k+1 and a copy stream moves the coder's inputs through rotating pinned buffers.
_CHUNK = 64
_CHUNK_EDGE = 16
_FACT_PART = int(os.environ.get("PCGC_FACT_PART", "48"))      # cubes per synthesis call of the progressive factorized decoder


def _chunks(B, small_first=False, small_last=False):
    """[a, b) chunk bounds.  The pipeline's exposed latency is one chunk's host-coder round trip at the start of a decode
    (nothing can be synthesised before the first chunk is decoded) and at the end of an encode (the last chunk's strings):
    those chunks are small (_CHUNK_EDGE cubes), the ones in between large (_CHUNK)."""
    e = _CHUNK_EDGE
    lo, hi = 0, B
    head, tail = [], []
    if small_first and B > 2 * e:
        head.append((0, e)); lo = e
        if hi - lo > 2 * e + _CHUNK:                                    # e, 2e, then full chunks: the GPU gets work early
            head.append((lo, lo + 2 * e)); lo += 2 * e
    if small_last and hi - lo > 2 * e:
        tail.append((hi - e, hi)); hi -= e
    mid = [(a, min(hi, a + _CHUNK)) for a in range(lo, hi, _CHUNK)]
    return head + mid + tail
def _gpu_decode_chunks(B):
    """Chunks of the GPU-coder decode pipeline.  Nothing can be synthesised before the first chunk's hyper latents have come
    out of the (sequential, host-side) hyper string, its CDF rows are built and its strings decoded -- a latency of one cube's
    string (a few ms) whatever the number of cubes -- so the schedule starts small and grows: 8, 24, 64 cubes, then the rest
    (decoded behind the synthesis of the chunk before; a chunk's CDF rows take ~2.5 MB per cube of device memory).  Measured on
    the vox10 cloud (tools/sweep_dec.py, decompress + select): 34.2 ms with one 64-cube head, 31.3 ms with this ramp."""
    ramp = [int(v) for v in os.environ.get("PCGC_DEC_RAMP", "8,24,64").split(",") if v]
    rest = int(os.environ.get("PCGC_DEC_CHUNK", "512"))
    if B <= max(ramp[0], 64):
        return [(0, B)]
    out, a = [], 0
    for r in ramp:
        if B - a <= r:
            break
        out.append((a, a + r)); a += r
    out += [(s, min(B, s + rest)) for s in range(a, B, rest)]
    return out


_POOL = None
_POOL_Z = None


def _pool():
    global _POOL
    if _POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _POOL = ThreadPoolExecutor(max_workers=1)
    return _POOL


def _pool_z():
    """Second worker: the single hyper-latent string (one sequential range coder) is coded beside the per-cube jobs."""
    global _POOL_Z
    if _POOL_Z is None:
        from concurrent.futures import ThreadPoolExecutor
        _POOL_Z = ThreadPoolExecutor(max_workers=1)
    return _POOL_Z


def encode_on_device(codec, entropy_bottleneck, cem, cubes, keep_side_info=False, want_likelihoods=False, z_to_host=None):
    """Every GPU kernel of the hyper encoder for ``cubes`` (host or device resident), enqueued without a host
    synchronisation: transforms chunk by chunk on the current stream, then ONE range-encoder launch for all B cubes on the
    coder stream.  -> (intervals [B,E], minmax [B,2], [z_hat per chunk], [(loc, scale) per chunk], packed bytes, offsets [B+1],
    []); tensors on the device.  The last element is always an empty list: the 7-tuple is kept for the callers that unpack it.
    The caller owns the synchronisation.
    ``z_to_host`` (a dict to fill): every chunk's quantised hyper latents and their (min, max) are also copied to pinned memory
    on the copy stream as soon as they exist -- ["z"] float32 [B,8,8,8,8], ["mm"] int32 [chunks,2], ["done"] an event that fires
    when the LAST chunk's copy has landed, i.e. before that chunk's hyper decoder, intervals and the range encoder have run:
    the host codes the one hyper string beside them."""
    B = cubes.shape[0]
    E = 16 * 16 * 16 * 16
    dev = codec.dev
    main, side = torch.cuda.current_stream(dev), codec.coder_stream()
    iv_all = torch.empty((B, E), dtype=torch.int32, device=dev)
    mm_all = torch.empty((B, 2), dtype=torch.int32, device=dev)
    z_hats, keep = [], []
    chunks = _chunks(B)
    # host-resident input: every chunk's H2D copy is issued up front on the copy stream, so only the first one is exposed
    uploads = None
    if not (isinstance(cubes, torch.Tensor) and cubes.is_cuda):
        cs = runtime.copy_stream(dev)
        uploads = []
        with torch.cuda.stream(cs):
            for a, b in chunks:
                xc = codec.to_device(cubes[a:b])
                ev = torch.cuda.Event()
                ev.record(cs)
                uploads.append((xc, ev))
    if z_to_host is not None:
        zcs = runtime.copy_stream(dev)
        nz = B * 8 * 8 * 8 * 8
        z_to_host["z"] = runtime.pinned_buffer("z_hat_enc", 4 * nz)[:4 * nz].view(torch.float32).view(B, 8, 8, 8, 8)
        z_to_host["mm"] = runtime.pinned_buffer("z_mm_enc", 8 * len(chunks))[:8 * len(chunks)].view(torch.int32).view(len(chunks), 2)
        runtime.COUNTERS["d2h_bytes"] += 4 * nz + 8 * len(chunks)

    for k, (a, b) in enumerate(chunks):
        if uploads is not None:
            x, ev = uploads[k]
            main.wait_event(ev)
            x.record_stream(main)
        else:
            x = cubes[a:b]
        ys = codec.analysis(x)
        zs = codec.hyper_encode(ys)
        z_hat, _, _, z_mm = codec.factorized(entropy_bottleneck._slot, zs, want_p=want_likelihoods, want_bits=want_likelihoods)
        z_hats.append(z_hat)
        if z_to_host is not None:
            zr = torch.cuda.Event()
            zr.record(main)
            z_hat.record_stream(zcs); z_mm.record_stream(zcs)
            with torch.cuda.stream(zcs):
                zcs.wait_event(zr)
                z_to_host["z"][a:b].copy_(z_hat, non_blocking=True)
                z_to_host["mm"][k].copy_(z_mm, non_blocking=True)
                if k == len(chunks) - 1:
                    z_to_host["done"] = torch.cuda.Event()
                    z_to_host["done"].record(zcs)
        locs, scales = codec.hyper_decode(z_hat, 1e-9)                  # lower_bound = 1e-9, transform.py:145-146
        _, mm = cem.intervals_dev(ys, locs, scales, iv_out=iv_all[a:b], want_likelihoods=want_likelihoods)
        mm_all[a:b].copy_(mm)
        if keep_side_info:
            keep.append((locs, scales))
    packed = offsets = None
    if B > 0:
        ready = torch.cuda.Event()
        ready.record(main)
        iv_all.record_stream(side)
        with torch.cuda.stream(side):
            side.wait_event(ready)
            packed, offsets = cem.encode_dev(iv_all)
    mm_all.record_stream(side)
    return iv_all, mm_all, z_hats, keep, packed, offsets, []


def _compress_hyper_gpu_coder(codec, entropy_bottleneck, cem, cubes, decompress, code_z=True, strings_on_device=False):
    """compress_hyper with the per-cube strings written ON THE GPU (csrc/gpu_coder.cu).  The chunks only enqueue kernels (no
    host synchronisation in the loop); the intervals land in one device buffer, ONE encoder launch codes the strings of all
    cubes on the coder stream, and this thread range-codes the single hyper string z on the host meanwhile (``code_z=False``:
    no hyper string)."""
    B = cubes.shape[0]
    side = codec.coder_stream()
    codec.deferred_checks(True)
    try:
        z_host = {} if code_z else None
        _, mm_all, z_hats, keep, packed, offsets, _ = encode_on_device(codec, entropy_bottleneck, cem, cubes, decompress, z_to_host=z_host)
        hdr = runtime.pinned_buffer("enc_hdr", 8 * (B + 1))
        off_h = hdr[:8 * (B + 1)].view(torch.int64)
        with torch.cuda.stream(side):
            off_h.copy_(offsets, non_blocking=True)
            hdr_done = torch.cuda.Event()
            hdr_done.record(side)
        # the ONE hyper string (global range, entropy_model.py:249-259) is coded here on the host, from the pinned copy of the
        # quantised latents that landed before the last chunk's hyper decoder / intervals and the GPU range encoder started
        z_all = torch.cat(z_hats) if len(z_hats) > 1 else z_hats[0]
        z_string = z_min = z_max = None
        _tr("enqueued")
        if code_z:
            z_host["done"].synchronize()
            _tr("z on host")
            z_string, z_min, z_max = entropy_bottleneck.compress_quantized_host(z_host["z"].numpy(), z_host["mm"].numpy())
            _tr("z coded")
        mm = runtime.to_host(mm_all).copy()
        _tr("minmax on host")
        hdr_done.synchronize()
        _tr("encoder done")
        off = off_h.numpy().copy()
        total = int(off[B])
        if strings_on_device:
            # sharded form: the strings stay packed in HBM (string i = packed[off[i]:off[i+1]]) and travel GPU -> GPU
            side.synchronize()
            codec.deferred_checks(False)
            codec.synchronize()
            return (packed[:total], off), mm, z_all, z_string, z_min, z_max, keep
        stage = runtime.pinned_buffer("enc_bytes", max(total, 1))[:total]
        with torch.cuda.stream(side):
            stage.copy_(packed[:total], non_blocking=True)
        side.synchronize()
        _tr("strings on host")
        runtime.COUNTERS["d2h_bytes"] += total + hdr.numel()
        blob = stage.numpy()
        strings = [blob[off[i]:off[i + 1]].tobytes() for i in range(B)]
        _tr("strings sliced")
    finally:
        codec.deferred_checks(False)
    codec.synchronize()                                                   # raises if any kernel of the section flagged an error
    return strings, mm, z_all, z_string, z_min, z_max, keep


def compress_hyper(cubes, model, ckpt_dir, decompress=False):
    """cubes [B,64,64,64,1] -> (y_strings[B], y_min_vs[B], y_max_vs[B], y_shape, z_strings, z_min_v,
    z_max_v, z_shape[, x_decodeds])  (transform.py:91-197)."""
    _log("===== Compress =====")
    codec = runtime.get_codec(model, ckpt_dir)
    entropy_bottleneck = _bottleneck(codec, 8)
    cem = SymmetricConditional().bind(codec)
    cubes = runtime.unwrap(cubes)
    B = cubes.shape[0]
    start = time.time()
    if B == 0:
        # an empty cloud: nothing to code.  (The reference's tf.map_fn / reduce_min raise on an empty batch; an empty stream that
        # decompress_hyper turns back into an empty [0,64,64,64,1] tensor is the useful behaviour for a partitioner that found no cube.)
        out = (runtime.HostResult(_strings_array([])), runtime.HostResult(np.zeros(0, np.int32)), runtime.HostResult(np.zeros(0, np.int32)),
               runtime.HostResult(np.array((1, 16, 16, 16, 16), dtype=np.int64)), runtime.HostResult(b""), runtime.HostResult(np.int32(0)),
               runtime.HostResult(np.int32(0)), runtime.HostResult(np.array((0, 8, 8, 8, 8), dtype=np.int32)))
        if decompress:
            return out + (runtime.DeviceResult(torch.zeros((0, 64, 64, 64, 1), dtype=torch.float32, device=codec.dev)),)
        return out
    if runtime.coder_mode() == "gpu" and B > 0:
        strings, mm, z_all, z_string, z_min, z_max, keep = _compress_hyper_gpu_coder(codec, entropy_bottleneck, cem, cubes, decompress)
        _log("Analysis + hyper transforms + entropy encode (GPU coder)", start)
        y_min_vs, y_max_vs = mm[:, 0].astype(np.int32), mm[:, 1].astype(np.int32)
        out = (runtime.HostResult(_strings_array(strings)), runtime.HostResult(y_min_vs), runtime.HostResult(y_max_vs),
               runtime.HostResult(np.array((1, 16, 16, 16, 16), dtype=np.int64)), runtime.HostResult(z_string),
               runtime.HostResult(np.int32(z_min)), runtime.HostResult(np.int32(z_max)),
               runtime.HostResult(np.array(z_all.shape, dtype=np.int32)))
        if decompress:
            locs = torch.cat([kk[0] for kk in keep])
            scales = torch.cat([kk[1] for kk in keep])
            y_dec = cem.decompress_cubes(strings, locs, scales, y_min_vs, y_max_vs)
            x_dec = codec.synthesis(y_dec.reshape(B, 16, 16, 16, 16))
            return out + (runtime.DeviceResult(x_dec),)
        return out
    jobs, mms, z_hats, keep = [], [], [], []
    chunks = _chunks(B, small_last=True)
    z_job = None
    for k, (a, b) in enumerate(chunks):
        x = codec.to_device(cubes[a:b])
        ys = codec.analysis(x)
        zs = codec.hyper_encode(ys)
        z_hat, _, _, _ = codec.factorized(entropy_bottleneck._slot, zs, want_p=False, want_bits=False)
        z_hats.append(z_hat)
        if k == len(chunks) - 1:
            # every z_hat exists now: start the ONE hyper string (global range, entropy_model.py:249-259) on its own worker so
            # that it is coded while the GPU finishes this chunk and the per-cube coder runs.
            z_all = torch.cat(z_hats) if len(z_hats) > 1 else z_hats[0]
            sym, cdf, z_min, z_max = entropy_bottleneck.compress_begin(z_all)
            z_job = _pool_z().submit(entropy_bottleneck.compress_finish, sym, cdf)
        locs, scales = codec.hyper_decode(z_hat, 1e-9)                  # lower_bound = 1e-9, transform.py:145-146
        if k >= 2:
            jobs[k - 2] = jobs[k - 2].result()                          # slot k%2 is free once its previous user finished
        stage, done, mm = cem.encode_begin(ys, locs, scales, k % 2)
        jobs.append(_pool().submit(cem.encode_finish, stage, done))
        mms.append(mm)
        if decompress:
            keep.append((ys.shape, locs, scales))
    strings = []
    for j in jobs:
        strings += j if isinstance(j, list) else j.result()
    if z_job is None:                                                   # B == 0
        z_all = torch.zeros((0, 8, 8, 8, 8), device=codec.dev)
        z_strings, z_min_v, z_max_v = entropy_bottleneck.compress(z_all)
    else:
        z_strings = runtime.HostResult(z_job.result())
        z_min_v, z_max_v = runtime.HostResult(np.int32(z_min)), runtime.HostResult(np.int32(z_max))
    z_shape = runtime.HostResult(np.array(z_all.shape, dtype=np.int32))
    _log("Analysis + hyper transforms + entropy encode (pipelined)", start)
    mm = np.concatenate(mms) if mms else np.zeros((0, 2), np.int32)
    y_min_vs, y_max_vs = mm[:, 0].astype(np.int32), mm[:, 1].astype(np.int32)
    y_shape = runtime.HostResult(np.array((1, 16, 16, 16, 16), dtype=np.int64))
    out = (runtime.HostResult(_strings_array(strings)), runtime.HostResult(y_min_vs), runtime.HostResult(y_max_vs), y_shape,
           z_strings, z_min_v, z_max_v, z_shape)
    if decompress:
        start = time.time()
        locs = torch.cat([kk[1] for kk in keep])
        scales = torch.cat([kk[2] for kk in keep])
        y_dec = cem.decompress_cubes(strings, locs, scales, y_min_vs, y_max_vs)
        _log("Entropy Decode", start)
        start = time.time()
        x_dec = codec.synthesis(y_dec.reshape(B, 16, 16, 16, 16))
        _log("Synthesis Transform", start)
        return out + (runtime.DeviceResult(x_dec),)
    return out


def _decompress_hyper_gpu_coder(codec, cem, strings, mins, maxs, y_shape, z_get, chunks, uploaded=None, sync=True):
    """decompress_hyper with the per-cube strings read ON THE GPU: the strings go up chunk by chunk (a few KB per cube), CDF
    rows are built and consumed on the device.  Chunk k+1 is decoded on the coder stream while chunk k is synthesised.
    ``sync=False`` -> a PendingDeviceResult (the caller, or its first consumer, waits and checks for device-side errors)."""
    dev = codec.dev
    main = torch.cuda.current_stream(dev)
    B = int(chunks[-1][1])
    xs = torch.empty([B, 64, 64, 64, 1], dtype=torch.float32, device=dev)
    parts, pending = [], None
    sub = int(os.environ.get("PCGC_SYNTH_PART", "64"))             # cubes per synthesis call = granularity of `parts`
    codec.deferred_checks(True)
    try:
        def finish(p):
            (a, b), y_hat, done = p
            main.wait_event(done)
            y5 = y_hat.reshape([b - a] + y_shape[1:])
            for s0 in range(a, b, sub):
                s1 = min(b, s0 + sub)
                codec.synthesis(y5[s0 - a:s1 - a], out=xs[s0:s1])
                ev = torch.cuda.Event()
                ev.record(main)
                parts.append((s0, s1, ev))

        for k, (a, b) in enumerate(chunks):
            # every chunk decodes on its own stream (round robin over 3): the decoder of chunk k+1 must not queue behind the
            # decoder of chunk k -- both are latency-bound single-warp-per-cube kernels that run side by side
            side = codec.coder_stream(1 + k % 3)
            if uploaded is not None:
                packed, offs = uploaded[0], uploaded[1][a:b + 1]
            else:
                packed, offs = codec.upload_strings(strings[a:b], slot=k % 4)     # this chunk's strings only: nothing waits for the rest
            locs, scales = codec.hyper_decode(z_get(a, b), 1e-9)
            ready = torch.cuda.Event()
            ready.record(main)
            for t in (locs, scales, packed, offs):
                t.record_stream(side)
            with torch.cuda.stream(side):
                side.wait_event(ready)
                # the CDF rows are built here beside the synthesis of the chunk before (r02: on the main stream they delayed
                # that synthesis, 32.1 against 31.6 ms)
                rows_pack = cem.decode_rows_dev(locs, scales, mins[a:b], maxs[a:b])
                y_hat = cem.decode_strings_dev(packed, offs, rows_pack)
                done = torch.cuda.Event()
                done.record(side)
            y_hat.record_stream(main)
            if pending is not None:
                finish(pending)                                            # synthesis of chunk k-1 overlaps the GPU decode of chunk k
            pending = ((a, b), y_hat, done)
        finish(pending)
    finally:
        codec.deferred_checks(False)
    if sync:
        codec.synchronize()                                                # raises if any kernel of the section flagged an error
        return xs
    return runtime.PendingDeviceResult(xs, parts, codec, parts[-1][2])


def decompress_hyper(y_strings, y_min_vs, y_max_vs, y_shape, z_strings, z_min_v, z_max_v, z_shape, model, ckpt_dir):
    """-> xs [B,64,64,64,1] occupancy logits  (transform.py:200-259)."""
    _log("===== Decompress =====")
    codec = runtime.get_codec(model, ckpt_dir)
    entropy_bottleneck = _bottleneck(codec, 8)
    cem = SymmetricConditional().bind(codec)
    z_shape = np.asarray(runtime.unwrap(z_shape)).reshape(-1)
    y_shape = [int(v) for v in np.asarray(runtime.unwrap(y_shape)).reshape(-1)]
    start = time.time()
    if int(z_shape[0]) == 0:                                             # the empty cloud (see compress_hyper)
        return runtime.DeviceResult(torch.zeros((0, 64, 64, 64, 1), dtype=torch.float32, device=codec.dev))
    # the hyper string decodes on a worker thread; each chunk below waits only for ITS cubes' symbols (they come first)
    z_get = entropy_bottleneck.decompress_progressive(z_strings, z_min_v, z_max_v, z_shape, z_shape[-1])
    _log("Entropy Decoder (Hyper) started", start)
    strings = _as_list_of_bytes(y_strings)
    B = int(z_shape[0])
    if len(strings) != B:
        raise ValueError("got %d y strings for %d cubes" % (len(strings), B))
    mins = np.asarray(runtime.unwrap(y_min_vs)).reshape(-1)
    maxs = np.asarray(runtime.unwrap(y_max_vs)).reshape(-1)
    start = time.time()
    if B == 0:
        return runtime.DeviceResult(torch.zeros((0, 64, 64, 64, 1), dtype=torch.float32, device=codec.dev))
    if runtime.coder_mode() == "gpu":
        # returned as soon as the last launch is queued: .numpy() / .tensor wait (and raise on a device-side error), and
        # select_voxels(codec=...) consumes the cubes part by part while the rest is still being synthesised
        xs = _decompress_hyper_gpu_coder(codec, cem, strings, mins, maxs, y_shape, z_get, _gpu_decode_chunks(B), sync=False)
        _log("Hyper decoder + entropy decode (GPU coder) + synthesis", start)
        return xs
    chunks = _chunks(B, small_first=True)
    xs_parts, pending = [], None

    def finish(p):
        (a, b), job = p
        y_hat = job.result()                                              # pinned float32 [b-a, E]
        ys = codec.to_device(y_hat).reshape([b - a] + y_shape[1:])
        xs_parts.append(codec.synthesis(ys))

    for k, (a, b) in enumerate(chunks):
        locs, scales = codec.hyper_decode(z_get(a, b), 1e-9)
        stage, done, off, mm, E = cem.decode_begin(locs, scales, mins[a:b], maxs[a:b], k % 2)
        job = _pool().submit(cem.decode_finish, strings[a:b], stage, done, off, mm, E, k % 2)
        if pending is not None:
            finish(pending)                                               # synthesis of chunk k-1 overlaps the host decode of chunk k
        pending = ((a, b), job)
    if pending is not None:
        finish(pending)
    xs = torch.cat(xs_parts) if len(xs_parts) > 1 else xs_parts[0]
    _log("Hyper decoder + entropy decode + synthesis (pipelined)", start)
    return runtime.DeviceResult(xs)
