"""Host-side runtime: one ``Codec`` = one pcgc_ctx on one GPU with one set of weights.

PyTorch is used ONLY for device/pinned buffers and the current CUDA stream; every computation
goes through the C ABI (``_lib``).  No CPU fallback: without CUDA + libpcgc_b200.so the
constructor raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib, netspec, weights as W

_NET_IDS = {
    ("voxception", "analysis_transform"): _lib.NET_VOX_ANALYSIS,
    ("voxception", "synthesis_transform"): _lib.NET_VOX_SYNTHESIS,
    ("voxception", "hyper_encoder"): _lib.NET_HYPER_ENCODER,
    ("voxception", "hyper_decoder"): _lib.NET_HYPER_DECODER,
    ("simple", "analysis_transform"): _lib.NET_SIMPLE_ANALYSIS,
    ("simple", "synthesis_transform"): _lib.NET_SIMPLE_SYNTHESIS,
}
_DTYPES = {np.dtype(np.uint8): _lib.DTYPE_U8, np.dtype(np.bool_): _lib.DTYPE_U8,
           np.dtype(np.float32): _lib.DTYPE_F32, np.dtype(np.float64): _lib.DTYPE_F64}
_TORCH_DTYPES = {torch.uint8: _lib.DTYPE_U8, torch.bool: _lib.DTYPE_U8, torch.float32: _lib.DTYPE_F32,
                 torch.float64: _lib.DTYPE_F64}


# bytes moved across PCIe by the host layer (bench.py e2e accounting)
COUNTERS = {"h2d_bytes": 0, "d2h_bytes": 0}


_PINNED: Dict[tuple, torch.Tensor] = {}


def pinned_buffer(tag: str, nbytes: int) -> torch.Tensor:
    """Reusable page-locked staging buffer (uint8), grown on demand.  One per (current device, calling thread's call-site
    tag): the returned view is valid until the same tag is requested again on that device.  (Two codecs on two devices used to
    share -- and overwrite -- one buffer per tag.)"""
    key = (torch.cuda.current_device() if torch.cuda.is_available() else -1, tag)
    buf = _PINNED.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes * 1.25), 1 << 16), dtype=torch.uint8).pin_memory()
        _PINNED[key] = buf
    return buf


_COPY_STREAMS: Dict[int, "torch.cuda.Stream"] = {}


def copy_stream(dev: torch.device) -> "torch.cuda.Stream":
    """Side stream for D2H copies that overlap the kernels of the next chunk."""
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    s = _COPY_STREAMS.get(idx)
    if s is None:
        s = torch.cuda.Stream(device=dev)
        _COPY_STREAMS[idx] = s
    return s


def to_host_async(t: torch.Tensor, tag: str):
    """Start a device->pinned copy of ``t`` on the copy stream (ordered after the work already queued on the current
    stream).  Returns (pinned view as torch tensor, event to synchronise before reading)."""
    nbytes = t.numel() * t.element_size()
    COUNTERS["d2h_bytes"] += nbytes
    t = t.detach().contiguous()
    stage = pinned_buffer(tag, nbytes)[:nbytes].view(t.dtype).view(t.shape)
    cs = copy_stream(t.device)
    ready = torch.cuda.Event()
    ready.record(torch.cuda.current_stream(t.device))
    cs.wait_event(ready)
    t.record_stream(cs)
    done = torch.cuda.Event()
    with torch.cuda.stream(cs):
        stage.copy_(t, non_blocking=True)
        done.record(cs)
    return stage, done


def to_host(t: torch.Tensor, tag: str = None) -> np.ndarray:
    """Device tensor -> NumPy (counted).  With a ``tag`` the copy lands in a reusable pinned buffer and the
    returned array is a VIEW of it (valid until the next call with the same tag)."""
    if not t.is_cuda:
        return t.detach().numpy()
    nbytes = t.numel() * t.element_size()
    COUNTERS["d2h_bytes"] += nbytes
    if tag is None or nbytes < (1 << 16):
        return t.detach().cpu().numpy()
    t = t.detach().contiguous()
    stage = pinned_buffer(tag, nbytes)[:nbytes].view(t.dtype).view(t.shape)
    stage.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return stage.numpy()


def host_copy(src: np.ndarray) -> np.ndarray:
    """Fresh NumPy copy of a (pinned staging) array through the library's multithreaded memcpy."""
    src = np.ascontiguousarray(src)
    out = np.empty(src.shape, src.dtype)
    if src.nbytes < (8 << 20):
        out[...] = src
        return out
    _lib.check(_lib.lib().pcgc_host_copy(out.ctypes.data, src.ctypes.data, src.nbytes, coder_threads()))
    return out


def host_copy_into(dst: np.ndarray, src: np.ndarray):
    """dst[...] = src for two contiguous arrays of equal size, through the library's multithreaded memcpy when large."""
    if dst.nbytes != src.nbytes or not dst.flags.c_contiguous or not src.flags.c_contiguous:
        raise ValueError("host_copy_into needs contiguous arrays of equal size")
    if src.nbytes < (8 << 20):
        dst.reshape(-1).view(np.uint8)[...] = src.reshape(-1).view(np.uint8)
        return
    _lib.check(_lib.lib().pcgc_host_copy(dst.ctypes.data, src.ctypes.data, src.nbytes, coder_threads()))


def model_name(model) -> str:
    """'voxception' | 'simple' from a model module (test.py:72 importlib seam), a name, or a class."""
    name = model if isinstance(model, str) else getattr(model, "MODEL_NAME", None) or getattr(model, "__name__", "")
    name = name.rsplit(".", 1)[-1]
    if "simple" in name:
        return "simple"
    if "voxception" in name:
        return "voxception"
    raise ValueError("unknown model %r (expected models.model_voxception or models.model_simple)" % (model,))


class DeviceResult:
    """What the drop-in API returns where the reference returns a TF eager tensor: callers do
    ``.numpy()`` on it (test.py:81,89,101-103,115).  ``.tensor`` is the torch CUDA buffer."""

    def __init__(self, tensor: torch.Tensor):
        self.tensor = tensor

    def numpy(self) -> np.ndarray:
        return to_host(self.tensor)

    @property
    def shape(self):
        return tuple(self.tensor.shape)

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a.astype(dtype) if dtype is not None else a

    def __len__(self):
        return self.tensor.shape[0]

    def __getitem__(self, i):
        return DeviceResult(self.tensor[i])


class PendingDeviceResult(DeviceResult):
    """A DeviceResult whose kernels may still be running: ``decompress_hyper`` returns it right after the last launch is queued.
    ``parts`` = [(a, b, event)]: cubes [a, b) of the tensor are final once ``event`` has fired, in this order -- a consumer that
    understands parts (``select_voxels(codec=...)``) starts on the first cubes while the last ones are still being synthesised.
    Every other access (``.tensor``, ``.numpy()``, ``unwrap``) first waits for the whole result and raises if a kernel of the
    section flagged an error, i.e. it behaves like the plain DeviceResult."""

    def __init__(self, tensor: torch.Tensor, parts, codec, done_event):
        self._full = tensor
        self.parts = list(parts)
        self._codec = codec
        self._done = done_event
        self.finalized = False

    @property
    def raw(self) -> torch.Tensor:
        """The tensor WITHOUT waiting: for consumers that queue their work on the producing stream (stream order is enough)."""
        return self._full

    def finalize(self):
        if not self.finalized:
            self.finalized = True
            self._done.synchronize()
            self._codec.synchronize()                  # raises if any kernel of the section flagged an error
        return self._full

    @property
    def tensor(self):
        return self.finalize()

    @property
    def shape(self):
        return tuple(self._full.shape)

    def __len__(self):
        return self._full.shape[0]


class HostResult:
    """Host-resident result (strings, min/max scalars, shapes) with the same ``.numpy()`` face."""

    def __init__(self, value):
        self.value = value

    def numpy(self):
        return self.value

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self.value, dtype=dtype)

    def __len__(self):
        return len(self.value)

    def __getitem__(self, i):
        return self.value[i]

    def __int__(self):
        return int(self.value)

    def __repr__(self):
        return "HostResult(%r)" % (self.value,)


def unwrap(x):
    if isinstance(x, (DeviceResult,)):
        return x.tensor
    if isinstance(x, HostResult):
        return x.value
    return x


class Codec:
    """One GPU context + weights.  Methods take/return torch CUDA tensors (buffers only)."""

    def __init__(self, model: str = "voxception", ckpt_dir: str = "", device: Optional[int] = None,
                 weights: Optional[Dict[str, np.ndarray]] = None, engine: int = _lib.ENGINE_AUTO):
        if not torch.cuda.is_available():
            raise RuntimeError("pcgcv1_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.lib()
        self.model = model
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.dev = torch.device("cuda", self.device)
        h = C.c_void_p()
        rc = self.lib.pcgc_create(C.byref(h), self.device)
        if rc != 0:
            raise _lib.PcgcError(rc, "pcgc_create failed on device %d (needs compute capability 10.x)" % self.device)
        self.ctx = h
        self.set_engine(engine)
        self.weights = weights if weights is not None else W.load(ckpt_dir, model)
        self._load_weights()
        self.latent_c = netspec.LATENT_CHANNELS[model]
        self.latent_n = 64 // netspec.LATENT_DOWN[model]
        self._enc_scratch = {}

    # -- plumbing ---------------------------------------------------------------------------
    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.pcgc_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    def _check(self, rc: int):
        _lib.check(rc, self.ctx)

    def _stream(self):
        self._check(self.lib.pcgc_set_stream(self.ctx, C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)))

    def set_engine(self, engine: int):
        self._check(self.lib.pcgc_set_engine(self.ctx, int(engine)))

    def synchronize(self):
        self._stream()
        self._check(self.lib.pcgc_synchronize(self.ctx))

    def launch_count(self) -> int:
        return int(self.lib.pcgc_launch_count(self.ctx))

    def profile(self, on: bool):
        self._check(self.lib.pcgc_profile_enable(self.ctx, int(on)))

    def profile_report(self):
        import json
        buf = C.create_string_buffer(1 << 16)
        self._stream()
        self._check(self.lib.pcgc_profile_report(self.ctx, buf, len(buf)))
        return json.loads(buf.value.decode())

    def _load_weights(self):
        w = self.weights
        for (m, net), layers in netspec.NETS.items():
            if m != self.model:
                continue
            nid = _NET_IDS[(m, net)]
            if "%s/%s/kernel" % (net, layers[0].name) not in w:
                continue            # e.g. a factorized-mode checkpoint has no hyper nets; using one then fails with NOT_READY
            for l in layers:
                k = np.ascontiguousarray(w["%s/%s/kernel" % (net, l.name)], dtype=np.float32)
                shape = (C.c_int64 * 5)(*k.shape)
                b = w.get("%s/%s/bias" % (net, l.name))
                bptr = None
                if b is not None:
                    b = np.ascontiguousarray(b, dtype=np.float32)
                    bptr = b.ctypes.data
                self._check(self.lib.pcgc_load_conv(self.ctx, nid, l.name.encode(), k.ctypes.data, shape, bptr))
        for slot, prefix in ((0, "estimator/"), (1, "estimator_y/")):
            if prefix + "matrix_0" in w:
                self.load_bottleneck(slot, {k[len(prefix):]: v for k, v in w.items() if k.startswith(prefix)})

    def load_bottleneck(self, slot: int, p: Dict[str, np.ndarray]):
        c = p["matrix_0"].shape[0]
        cat = lambda name: np.ascontiguousarray(
            np.concatenate([np.asarray(p["%s_%d" % (name, i)], np.float32).reshape(-1) for i in range(4)]))
        m, b, f = cat("matrix"), cat("bais"), cat("factor")
        self._check(self.lib.pcgc_load_bottleneck(self.ctx, slot, c, m.ctypes.data, b.ctypes.data, f.ctypes.data))
        if not hasattr(self, "bn_channels"):
            self.bn_channels = {}
        self.bn_channels[slot] = c

    def to_device(self, a, dtype=None) -> torch.Tensor:
        """numpy / torch / Result -> contiguous torch tensor on this codec's device."""
        a = unwrap(a)
        if isinstance(a, torch.Tensor):
            if not a.is_cuda:
                COUNTERS["h2d_bytes"] += a.numel() * a.element_size()
            t = a.to(self.dev, non_blocking=True)
        else:
            a = np.ascontiguousarray(a)
            if a.dtype == np.bool_:
                a = a.view(np.uint8)
            COUNTERS["h2d_bytes"] += a.nbytes
            t = torch.from_numpy(a).to(self.dev, non_blocking=True)
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.contiguous()

    def bottleneck_slot(self, channels: int) -> int:
        for slot, c in getattr(self, "bn_channels", {}).items():
            if c == channels:
                return slot
        raise RuntimeError("no EntropyBottleneck with %d channels is loaded" % channels)

    # -- transforms ---------------------------------------------------------------------------
    def analysis(self, cubes: torch.Tensor) -> torch.Tensor:
        """[B,64,64,64,1] uint8/float32/float64 -> y [B,n,n,n,C] float32."""
        if cubes.dtype not in _TORCH_DTYPES:
            cubes = cubes.to(torch.float32)
        if tuple(cubes.shape[1:]) != (64, 64, 64, 1):
            raise ValueError("cubes must be [B,64,64,64,1], got %s" % (tuple(cubes.shape),))
        B = cubes.shape[0]
        n, c = self.latent_n, self.latent_c
        y = torch.empty((B, n, n, n, c), dtype=torch.float32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_analysis(self.ctx, _NET_IDS[(self.model, "analysis_transform")], cubes.data_ptr(),
                                           _TORCH_DTYPES[cubes.dtype], B, y.data_ptr()))
        return y

    def synthesis(self, y: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        n, c = self.latent_n, self.latent_c
        if tuple(y.shape[1:]) != (n, n, n, c) or y.dtype != torch.float32:
            raise ValueError("y must be float32 [B,%d,%d,%d,%d], got %s %s" % (n, n, n, c, tuple(y.shape), y.dtype))
        B = y.shape[0]
        if out is not None:
            if tuple(out.shape) != (B, 64, 64, 64, 1) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.dev:
                raise ValueError("out must be a contiguous float32 [B,64,64,64,1] tensor on the codec's device")
            x = out
        else:
            x = torch.empty((B, 64, 64, 64, 1), dtype=torch.float32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_synthesis(self.ctx, _NET_IDS[(self.model, "synthesis_transform")], y.data_ptr(), B,
                                            x.data_ptr()))
        return x

    def hyper_encode(self, y: torch.Tensor) -> torch.Tensor:
        if tuple(y.shape[1:]) != (16, 16, 16, 16) or y.dtype != torch.float32:
            raise ValueError("y must be float32 [B,16,16,16,16]")
        B = y.shape[0]
        z = torch.empty((B, 8, 8, 8, 8), dtype=torch.float32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_hyper_encode(self.ctx, y.data_ptr(), B, z.data_ptr()))
        return z

    def hyper_decode(self, z_hat: torch.Tensor, scale_floor: float = 1e-9) -> Tuple[torch.Tensor, torch.Tensor]:
        if tuple(z_hat.shape[1:]) != (8, 8, 8, 8) or z_hat.dtype != torch.float32:
            raise ValueError("z_hat must be float32 [B,8,8,8,8]")
        B = z_hat.shape[0]
        loc = torch.empty((B, 16, 16, 16, 16), dtype=torch.float32, device=self.dev)
        scale = torch.empty_like(loc)
        self._stream()
        self._check(self.lib.pcgc_hyper_decode(self.ctx, z_hat.data_ptr(), B, scale_floor, loc.data_ptr(), scale.data_ptr()))
        return loc, scale

    # -- entropy models -------------------------------------------------------------------------
    def factorized(self, slot: int, x: torch.Tensor, bound: float = 1e-9, want_p: bool = True, want_bits: bool = True):
        """-> (x_hat, p|None, bits (double[1] tensor)|None, minmax int32[2] tensor)."""
        Cc = x.shape[-1]
        n_vox = x.numel() // Cc
        x_hat = torch.empty_like(x)
        p = torch.empty_like(x) if want_p else None
        bits = torch.zeros(1, dtype=torch.float64, device=self.dev) if want_bits else None
        mm = torch.empty(2, dtype=torch.int32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_factorized_quantize_likelihood(
            self.ctx, slot, x.data_ptr(), n_vox, Cc, bound, x_hat.data_ptr(), p.data_ptr() if want_p else None,
            bits.data_ptr() if want_bits else None, mm.data_ptr()))
        return x_hat, p, bits, mm

    def factorized_cdf(self, slot: int, min_v: int, max_v: int, bound: float = 1e-9, precision: int = 16) -> np.ndarray:
        Cc = self.bn_channels[slot]
        N = int(max_v) - int(min_v) + 1
        cdf = np.empty((Cc, max(N, 1) + 1), np.int32)
        self._stream()
        self._check(self.lib.pcgc_factorized_cdf(self.ctx, slot, int(min_v), int(max_v), bound, precision, cdf.ctypes.data))
        return cdf

    def laplace(self, y: torch.Tensor, loc: torch.Tensor, scale: torch.Tensor, bound: float = 1e-9,
                want_p: bool = True, want_bits: bool = True):
        """per cube -> (y_hat, p|None, bits double[B]|None, minmax int32[B,2])."""
        B = y.shape[0]
        E = y.numel() // max(B, 1)
        y_hat = torch.empty_like(y)
        p = torch.empty_like(y) if want_p else None
        bits = torch.zeros(B, dtype=torch.float64, device=self.dev) if want_bits else None
        mm = torch.empty((B, 2), dtype=torch.int32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_laplace_quantize_likelihood(
            self.ctx, y.data_ptr(), loc.data_ptr(), scale.data_ptr(), B, E, bound, y_hat.data_ptr(),
            p.data_ptr() if want_p else None, bits.data_ptr() if want_bits else None, mm.data_ptr()))
        return y_hat, p, bits, mm

    def widen_symbol_ranges(self, mm: torch.Tensor):
        """In place: every per-cube (min_v, max_v) gets 0 inside it and at least two symbols (codable by pmf_to_quantized_cdf,
        storable in the .strings_head byte)."""
        self._stream()
        self._check(self.lib.pcgc_widen_symbol_ranges(self.ctx, mm.data_ptr(), mm.numel() // 2))
        return mm

    def laplace_intervals(self, y_hat, loc, scale, mm: torch.Tensor, bound: float = 1e-9, out: torch.Tensor = None) -> torch.Tensor:
        B = y_hat.shape[0]
        E = y_hat.numel() // max(B, 1)
        iv = out if out is not None else torch.empty((B, E), dtype=torch.int32, device=self.dev)     # uint32 payload
        self._stream()
        self._check(self.lib.pcgc_laplace_intervals(self.ctx, y_hat.data_ptr(), loc.data_ptr(), scale.data_ptr(), B, E,
                                                    mm.data_ptr(), bound, 16, iv.data_ptr()))
        return iv

    def laplace_cdf(self, loc, scale, minmax_host: np.ndarray, bound: float = 1e-9):
        """-> (rows uint16 device tensor, row_offset int64 host array [B+1])."""
        B = loc.shape[0]
        E = loc.numel() // max(B, 1)
        mm = np.ascontiguousarray(minmax_host, dtype=np.int32).reshape(B, 2)
        N = (mm[:, 1] - mm[:, 0] + 1).astype(np.int64)
        off = np.zeros(B + 1, np.int64)
        np.cumsum(N * E, out=off[1:])
        rows = torch.empty(int(off[-1]), dtype=torch.int16, device=self.dev)    # uint16 payload
        self._stream()
        self._check(self.lib.pcgc_laplace_cdf(self.ctx, loc.data_ptr(), scale.data_ptr(), B, E, mm.ctypes.data, bound, 16,
                                              off.ctypes.data, rows.data_ptr()))
        return rows, off

    # -- GPU-side range coder (csrc/gpu_coder.cu) ------------------------------------------------------
    def coder_stream(self, which: int = 0) -> "torch.cuda.Stream":
        """Side streams of this codec for the (latency-bound, one warp per cube) coder kernels: they run beside the conv kernels
        of the main stream instead of between them.  0: encoder, 1: decoder (CDF rows + range decoder)."""
        ss = getattr(self, "_coder_streams", None)
        if ss is None:
            ss = self._coder_streams = {}
        if which not in ss:
            ss[which] = torch.cuda.Stream(device=self.dev)
        return ss[which]

    def deferred_checks(self, on: bool):
        """Pipelined sections: entry points stop synchronising just to read the device error flag; ``synchronize()`` at the
        end of the section reports it (and raises)."""
        self._check(self.lib.pcgc_set_deferred_checks(self.ctx, int(bool(on))))

    def set_quantize_mode(self, noise: bool, seed: int = 0):
        """"symbols" (round, default) or "noise" (x + U(-1/2, 1/2), seeded Philox) for factorized() / laplace()."""
        self._check(self.lib.pcgc_set_quantize_mode(self.ctx, int(bool(noise)), int(seed) & 0xFFFFFFFFFFFFFFFF))

    @staticmethod
    def row_offsets(minmax_host: np.ndarray, E: int) -> np.ndarray:
        mm = np.ascontiguousarray(minmax_host, dtype=np.int32).reshape(-1, 2)
        N = (mm[:, 1] - mm[:, 0] + 1).astype(np.int64)
        off = np.zeros(len(mm) + 1, np.int64)
        np.cumsum(N * E, out=off[1:])
        return off

    def laplace_cdf_dev(self, loc, scale, mm_dev: torch.Tensor, off_dev: torch.Tensor, total: int, bound: float = 1e-9):
        """Per-element CDF rows with device-resident headers; no host synchronisation.  -> rows (uint16 payload) on the device."""
        B = loc.shape[0]
        E = loc.numel() // max(B, 1)
        rows = torch.empty(max(int(total), 1), dtype=torch.int16, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_laplace_cdf_dev(self.ctx, loc.data_ptr(), scale.data_ptr(), B, E, mm_dev.data_ptr(), off_dev.data_ptr(),
                                                  float(total), bound, 16, rows.data_ptr()))
        return rows

    def gpu_range_encode(self, iv: torch.Tensor):
        """iv int32 [B,E] (pcgc_laplace_intervals payload) on the device -> (packed uint8 [cap], offsets int64 [B+1]), both on the
        device; string b = packed[offsets[b]:offsets[b+1]].  Asynchronous on the current stream."""
        B, E = iv.shape
        stride = 6 * E + 64                    # per cube: the string (<= 2E + 2 bytes) + the encoder's 32-bit digit sums
        # the 400 KB-per-cube scratch is kept per (stream, capacity): allocating ~100 MB per call made the caching allocator fall
        # back to cudaMalloc every few calls (a 5 ms stall inside the coder's launch, seen as 1.7 vs 7.1 ms per launch)
        key = (torch.cuda.current_stream(self.dev).cuda_stream, stride)
        held = self._enc_scratch.get(key)
        if held is None or held[0].shape[0] < max(B, 1):
            held = (torch.empty((max(B, 1), stride), dtype=torch.uint8, device=self.dev),
                    torch.empty(max(B, 1), dtype=torch.int64, device=self.dev))
            self._enc_scratch[key] = held
        scratch, lens = held
        packed = torch.empty(max(B, 1) * (2 * E + 8), dtype=torch.uint8, device=self.dev)
        offsets = torch.empty(B + 1, dtype=torch.int64, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_range_encode_intervals_dev(self.ctx, iv.data_ptr(), B, E, 16, scratch.data_ptr(), stride, lens.data_ptr(),
                                                             packed.data_ptr(), packed.numel(), offsets.data_ptr()))
        return packed, offsets

    def gpu_range_decode(self, packed: torch.Tensor, offsets: torch.Tensor, rows: torch.Tensor, off_dev: torch.Tensor, total: int,
                         mm_dev: torch.Tensor, max_n: int, B: int, E: int) -> torch.Tensor:
        """-> y_hat float32 [B,E] on the device (symbol + min_v).  Asynchronous on the current stream."""
        y_hat = torch.empty((B, E), dtype=torch.float32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_range_decode_rows_dev(self.ctx, packed.data_ptr(), offsets.data_ptr(), B, E, rows.data_ptr(), off_dev.data_ptr(),
                                                        float(total), mm_dev.data_ptr(), int(max_n), 16, y_hat.data_ptr()))
        return y_hat

    def upload_strings(self, strings, slot: int = 0):
        """list of byte strings -> (packed uint8 device tensor, offsets int64 [B+1] device tensor) in ONE H2D copy.  ``slot``
        picks one of the rotating pinned staging buffers; a slot is only rewritten after its previous copy has completed."""
        B = len(strings)
        prev = getattr(self, "_upload_events", None)
        if prev is None:
            prev = self._upload_events = {}
        if slot in prev:
            prev[slot].synchronize()
        lens = np.fromiter((len(s) for s in strings), np.int64, B)
        off = np.zeros(B + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        total = int(off[B])
        pad = (-total) % 8                                                   # keep the offsets 8-byte aligned inside the buffer
        n = total + pad + 8 * (B + 1)
        stage = pinned_buffer("dec_bytes%d" % slot, n)[:n]
        h = stage.numpy()
        if total:
            h[:total] = np.frombuffer(b"".join(bytes(s) for s in strings), np.uint8)
        h[total + pad:] = off.view(np.uint8)
        COUNTERS["h2d_bytes"] += n
        up = stage.to(self.dev, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        prev[slot] = ev
        return up, up[total + pad:].view(torch.int64)

    def factorized_cdf_host(self, slot: int, min_v: int, max_v: int, bound: float = 1e-9, precision: int = 16) -> np.ndarray:
        """Host twin of factorized_cdf (same det_math.h density, same normaliser): must be bit-identical to it."""
        Cc = self.bn_channels[slot]
        N = int(max_v) - int(min_v) + 1
        cdf = np.empty((Cc, max(N, 1) + 1), np.int32)
        self._check(self.lib.pcgc_factorized_cdf_host(self.ctx, slot, int(min_v), int(max_v), bound, precision, cdf.ctypes.data))
        return cdf

    # -- top-k ---------------------------------------------------------------------------------
    def topk(self, logits: torch.Tensor, ks: torch.Tensor):
        """logits float32 [B,...]; ks int32 [B] -> (mask uint8 same shape, thres float[B], count int32[B])."""
        B = logits.shape[0]
        V = logits.numel() // max(B, 1)
        mask = torch.empty(logits.shape, dtype=torch.uint8, device=self.dev)
        thres = torch.empty(B, dtype=torch.float32, device=self.dev)
        cnt = torch.empty(B, dtype=torch.int32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_topk_select(self.ctx, logits.data_ptr(), B, V, ks.data_ptr(), mask.data_ptr(),
                                              thres.data_ptr(), cnt.data_ptr()))
        return mask, thres, cnt

    def threshold(self, logits: torch.Tensor, thres: float):
        B = logits.shape[0]
        V = logits.numel() // max(B, 1)
        mask = torch.empty(logits.shape, dtype=torch.uint8, device=self.dev)
        cnt = torch.empty(B, dtype=torch.int32, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_threshold_select(self.ctx, logits.data_ptr(), B, V, float(thres), mask.data_ptr(), cnt.data_ptr()))
        return mask, cnt


    def voxelize(self, local: np.ndarray, offsets: np.ndarray, S: int = 64) -> torch.Tensor:
        """points grouped per cube (int16 [n,3], offsets int64 [B+1]) -> uint8 occupancy [B,S,S,S,1] on the device
        (points2voxels, inout_points.py:116-132)."""
        local = np.ascontiguousarray(local, dtype=np.int16).reshape(-1, 3)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        B = len(offsets) - 1
        cubes = torch.empty((B, S, S, S, 1), dtype=torch.uint8, device=self.dev)
        ld = self.to_device(local) if len(local) else torch.zeros((1, 3), dtype=torch.int16, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_voxelize(self.ctx, ld.data_ptr(), offsets.ctypes.data, B, S, cubes.data_ptr()))
        return cubes

    def extract_points(self, mask: torch.Tensor, cap: Optional[int] = None):
        """uint8 mask [B,S,S,S(,1)] on the device -> (points int16 [total,3] NumPy, counts int32 [B] NumPy): the non-zero
        voxels of every cube in np.where order (voxels2points, inout_points.py:134-143).  ``cap`` = an upper bound of the
        total when the caller knows one (saves a second pass)."""
        pts, counts = self.extract_points_device(mask, cap)
        return to_host(pts, "extract_points").copy(), to_host(counts, "extract_counts").copy()

    def extract_points_device(self, mask: torch.Tensor, cap: Optional[int] = None):
        """extract_points with the results left on the device: (points int16 [total,3], counts int32 [B]) torch tensors.
        Synchronises once to read the total."""
        B, S = mask.shape[0], mask.shape[1]
        counts = torch.empty(max(B, 1), dtype=torch.int32, device=self.dev)
        total = torch.empty(1, dtype=torch.int64, device=self.dev)
        self._stream()
        for attempt in range(2):
            n = int(cap) if cap is not None else 0
            pts = torch.empty((max(n, 1), 3), dtype=torch.int16, device=self.dev)
            self._check(self.lib.pcgc_extract_points(self.ctx, mask.data_ptr(), B, S, counts.data_ptr(), pts.data_ptr(), n, total.data_ptr()))
            t = int(to_host(total, "extract_total")[0])
            if t <= n:
                break
            cap = t
        return pts[:t], counts[:B]

    def geometry_sums(self, a: torch.Tensor, b: torch.Tensor, normals_a: Optional[torch.Tensor] = None) -> torch.Tensor:
        """D1 / D2 sums of two point sets on the device (pcgc_geometry_sums): a, b float64 [n,3] (normals_a float64 [n_a,3] or
        None) on this codec's device -> float64 [2,2,2] device tensor [direction 1 (a -> b), 2 (b -> a)][p2point, p2plane][sum,
        max] (p2plane zero without normals).  Asynchronous on the current stream."""
        for name, t in (("a", a), ("b", b), ("normals_a", normals_a)):
            if t is None:
                continue
            if t.dtype != torch.float64 or t.dim() != 2 or t.shape[1] != 3 or t.device != self.dev or not t.is_contiguous():
                raise ValueError("%s must be a contiguous float64 [n,3] tensor on %s" % (name, self.dev))
        if len(a) == 0 or len(b) == 0:
            raise ValueError("geometry_sums: empty point cloud")
        if normals_a is not None and len(normals_a) != len(a):
            raise ValueError("normals_a must have one row per point of a")
        out = torch.empty((2, 2, 2), dtype=torch.float64, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_geometry_sums(self.ctx, a.data_ptr(), len(a), b.data_ptr(), len(b),
                                                normals_a.data_ptr() if normals_a is not None else None, out.data_ptr()))
        return out

    def estimate_normals(self, points: torch.Tensor, k: int = 30, return_knn: bool = False):
        """k-nearest-neighbour PCA normals of one point set on the device (pcgc_estimate_normals; contract, tie rule and sign rule
        in include/pcgc_b200.h): points float64 [n,3] on this codec's device -> normals float64 [n,3] device tensor, and with
        ``return_knn`` also the int32 [n,k] neighbour indices in (distance, index) order (-1 beyond n).  1 <= k <= 64.
        Asynchronous on the current stream."""
        if points.dtype != torch.float64 or points.dim() != 2 or points.shape[1] != 3 or points.device != self.dev \
                or not points.is_contiguous():
            raise ValueError("points must be a contiguous float64 [n,3] tensor on %s" % self.dev)
        if len(points) == 0:
            raise ValueError("estimate_normals: empty point cloud")
        if not 1 <= int(k) <= 64:
            raise ValueError("estimate_normals: k must be in 1 .. 64, got %s" % k)
        k = int(k)
        normals = torch.empty((len(points), 3), dtype=torch.float64, device=self.dev)
        knn = torch.empty((len(points), k), dtype=torch.int32, device=self.dev) if return_knn else None
        self._stream()
        self._check(self.lib.pcgc_estimate_normals(self.ctx, points.data_ptr(), len(points), k, normals.data_ptr(),
                                                   knn.data_ptr() if knn is not None else None))
        return (normals, knn) if return_knn else normals

    def sample_mesh(self, verts: torch.Tensor, tris: torch.Tensor, n: int, seed: int, resolution: int, rotation=None,
                    return_samples: bool = False):
        """Uniform surface samples of a triangle mesh on a grid, deduplicated (pcgc_mesh_sample; the exact rule is in
        include/pcgc_b200.h): verts float64 [V,3] and tris int32 [F,3] on this codec's device, ``n`` samples drawn with ``seed``,
        rotated by ``rotation`` (float64 [3,3]; None = identity), on a ``resolution``^3 grid -> the distinct grid points as an int32
        [m,3] device tensor in lexicographic order, and with ``return_samples`` also the rotated samples float64 [n,3] and their
        faces int32 [n] in sample order.  Synchronises once."""
        if verts.dtype != torch.float64 or verts.dim() != 2 or verts.shape[1] != 3 or verts.device != self.dev \
                or not verts.is_contiguous():
            raise ValueError("verts must be a contiguous float64 [V,3] tensor on %s" % self.dev)
        if tris.dtype != torch.int32 or tris.dim() != 2 or tris.shape[1] != 3 or tris.device != self.dev or not tris.is_contiguous():
            raise ValueError("tris must be a contiguous int32 [F,3] tensor on %s" % self.dev)
        if len(verts) == 0 or len(tris) == 0:
            raise ValueError("sample_mesh: the mesh has no vertices or no faces")
        if not 1 <= int(n) <= 2 ** 28:
            raise ValueError("sample_mesh: n must be in 1 .. 2^28, got %s" % n)
        if not 2 <= int(resolution) <= 4096:
            raise ValueError("sample_mesh: resolution must be in 2 .. 4096, got %s" % resolution)
        if not 0 <= int(seed) < 2 ** 64:
            raise ValueError("sample_mesh: seed must be in 0 .. 2^64 - 1, got %s" % seed)
        rot = np.eye(3) if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64)
        if rot.shape != (3, 3) or not np.all(np.isfinite(rot)):
            raise ValueError("sample_mesh: rotation must be a finite [3,3] matrix")
        n = int(n)
        points = torch.empty((n, 3), dtype=torch.int32, device=self.dev)
        samples = torch.empty((n, 3), dtype=torch.float64, device=self.dev) if return_samples else None
        faces = torch.empty(n, dtype=torch.int32, device=self.dev) if return_samples else None
        m = C.c_int64()
        self._stream()
        self._check(self.lib.pcgc_mesh_sample(self.ctx, verts.data_ptr(), len(verts), tris.data_ptr(), len(tris), rot.ctypes.data, n,
                                              int(seed), int(resolution), points.data_ptr(), C.byref(m),
                                              samples.data_ptr() if return_samples else None,
                                              faces.data_ptr() if return_samples else None))
        points = points[:m.value]
        return (points, samples, faces) if return_samples else points

    def count_voxels(self, cubes: torch.Tensor) -> np.ndarray:
        """number of non-zero voxels per cube (np.sum(cubes, axis=(1,2,3,4)), process.py:44)."""
        B, S = cubes.shape[0], cubes.shape[1]
        counts = torch.empty(max(B, 1), dtype=torch.int32, device=self.dev)
        total = torch.empty(1, dtype=torch.int64, device=self.dev)
        self._stream()
        self._check(self.lib.pcgc_extract_points(self.ctx, cubes.data_ptr(), B, S, counts.data_ptr(), None, 0, total.data_ptr()))
        return to_host(counts[:B], "extract_counts").copy()


_CODECS: Dict[tuple, Codec] = {}


def get_codec(model="voxception", ckpt_dir: str = "", device: Optional[int] = None) -> Codec:
    """Cached codec per (model, checkpoint, device): the reference rebuilds and restores its Keras
    models on every call (transform.py:33-38); weights here are uploaded once."""
    name = model_name(model)
    dev = torch.cuda.current_device() if (device is None and torch.cuda.is_available()) else device
    key = (name, os.path.abspath(ckpt_dir) if ckpt_dir else "", dev)
    c = _CODECS.get(key)
    if c is None:
        c = Codec(name, ckpt_dir, dev)
        _CODECS[key] = c
    return c


# ---- host coder helpers (no ctx) ---------------------------------------------------------------
def range_encode(sym: np.ndarray, cdf: np.ndarray, precision: int = 16) -> bytes:
    """sym int16 [n] coded with cdf row (i % rows); cdf int32 [rows, N+1]."""
    L = _lib.lib()
    sym = np.ascontiguousarray(sym, dtype=np.int16).reshape(-1)
    cdf = np.ascontiguousarray(cdf, dtype=np.int32)
    rows, N = cdf.shape[0], cdf.shape[1] - 1
    cap = 2 * sym.size + 64
    out = np.empty(cap, np.uint8)
    ln = C.c_int64()
    _lib.check(L.pcgc_range_encode(sym.ctypes.data, sym.size, cdf.ctypes.data, rows, N, precision, out.ctypes.data, cap, C.byref(ln)))
    return out[:ln.value].tobytes()


class ProgressiveDecode:
    """One long string decoded on a worker thread with its position published (pcgc_range_decode_progress): ``wait(n)``
    returns once the first ``n`` symbols are in ``sym``."""

    def __init__(self, data: bytes, n: int, cdf: np.ndarray, precision: int = 16, step: int = 1 << 15):
        self._data = bytes(data)
        self._buf = np.frombuffer(self._data, np.uint8) if len(self._data) else np.zeros(1, np.uint8)
        self._cdf = np.ascontiguousarray(cdf, dtype=np.int32)
        self.n = int(n)
        self.sym = np.empty(self.n, np.int16)
        self._progress = C.c_int64(0)
        self._rc = None
        rows, N = self._cdf.shape[0], self._cdf.shape[1] - 1
        L = _lib.lib()

        def run():
            self._rc = L.pcgc_range_decode_progress(self._buf.ctypes.data, len(self._data), self.n, self._cdf.ctypes.data, rows, N, precision,
                                                    self.sym.ctypes.data, C.byref(self._progress), int(step))
        import threading
        self._thread = threading.Thread(target=run, daemon=True)
        self._thread.start()

    def wait(self, n: int) -> np.ndarray:
        n = min(int(n), self.n)
        import time
        while self._progress.value < n and self._progress.value >= 0 and self._rc is None:
            time.sleep(0)                                        # yield; the decoder thread holds no GIL inside the C call
        if self._progress.value < n:                             # finished (or failed) before reaching n
            self._thread.join()
            _lib.check(self._rc if self._rc is not None else 0)
        return self.sym[:n]

    def finish(self) -> np.ndarray:
        self._thread.join()
        _lib.check(self._rc)
        return self.sym


def range_decode(data: bytes, n: int, cdf: np.ndarray, precision: int = 16) -> np.ndarray:
    L = _lib.lib()
    cdf = np.ascontiguousarray(cdf, dtype=np.int32)
    rows, N = cdf.shape[0], cdf.shape[1] - 1
    buf = np.frombuffer(bytes(data), np.uint8) if len(data) else np.zeros(1, np.uint8)
    sym = np.empty(n, np.int16)
    _lib.check(L.pcgc_range_decode(buf.ctypes.data, len(data), n, cdf.ctypes.data, rows, N, precision, sym.ctypes.data))
    return sym


def host_laplace_cdf(loc: np.ndarray, scale: np.ndarray, minmax: np.ndarray, bound: float = 1e-9, threads: int = 0):
    """Host twin of Codec.laplace_cdf (bit-identical rows): loc/scale float32 [B,E] -> (rows uint16 flat, row_offset int64 [B+1])."""
    L = _lib.lib()
    loc = np.ascontiguousarray(loc, dtype=np.float32)
    scale = np.ascontiguousarray(scale, dtype=np.float32)
    B = loc.shape[0]
    E = loc.size // max(B, 1)
    mm = np.ascontiguousarray(minmax, dtype=np.int32).reshape(B, 2)
    off = Codec.row_offsets(mm, E)
    rows = np.empty(int(off[-1]), np.uint16)
    _lib.check(L.pcgc_host_laplace_cdf(loc.ctypes.data, scale.ctypes.data, B, E, mm.ctypes.data, bound, 16, off.ctypes.data, rows.ctypes.data,
                                       threads or coder_threads()))
    return rows, off


def coder_mode() -> str:
    """Where the per-cube range coder runs: "gpu" (default; csrc/gpu_coder.cu) or "host" (the thread-pool coder of coder.cpp,
    PCGC_CODER=host).  Both write the same bytes."""
    m = os.environ.get("PCGC_CODER", "gpu").lower()
    if m not in ("gpu", "host"):
        raise ValueError("PCGC_CODER must be 'gpu' or 'host'")
    return m


def coder_threads() -> int:
    """Host threads one process gives the per-cube range coder: ``PCGC_CODER_THREADS`` if set, else the cores divided by
    the processes of this node (torchrun's LOCAL_WORLD_SIZE) so that N ranks do not oversubscribe the host."""
    env = os.environ.get("PCGC_CODER_THREADS")
    if env:
        return max(1, int(env))
    cores = os.cpu_count() or 1
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, cores // max(1, local_world))


def range_encode_intervals_batch(iv: np.ndarray, threads: int = 0):
    """iv uint32/int32 [B,E] (host) -> list of B byte strings."""
    L = _lib.lib()
    iv = np.ascontiguousarray(iv)
    B, E = iv.shape
    stride = 2 * E + 64
    out = np.empty((B, stride), np.uint8)
    lens = np.empty(B, np.int64)
    _lib.check(L.pcgc_range_encode_intervals_batch(iv.ctypes.data, B, E, 16, out.ctypes.data, stride, lens.ctypes.data, threads or coder_threads()))
    return [out[b, :lens[b]].tobytes() for b in range(B)]


def range_decode_rows_batch_f32(strings, E: int, rows: np.ndarray, row_offset: np.ndarray, minmax: np.ndarray,
                                threads: int = 0, out_tag: str = "y_hat_dec") -> torch.Tensor:
    """-> pinned float32 torch tensor [B,E] holding y_hat = symbol + min_v (valid until the next call)."""
    L = _lib.lib()
    B = len(strings)
    bufs = [np.frombuffer(bytes(s), np.uint8) if len(s) else np.zeros(1, np.uint8) for s in strings]
    ptrs = (C.c_void_p * B)(*[b.ctypes.data for b in bufs])
    nbytes = np.array([len(s) for s in strings], np.int64)
    rows = np.ascontiguousarray(rows)
    row_offset = np.ascontiguousarray(row_offset, dtype=np.int64)
    minmax = np.ascontiguousarray(minmax, dtype=np.int32)
    out = pinned_buffer(out_tag, B * E * 4)[:B * E * 4].view(torch.float32).view(B, E)
    _lib.check(L.pcgc_range_decode_rows_batch_f32(ptrs, nbytes.ctypes.data, B, E, rows.ctypes.data, row_offset.ctypes.data,
                                                  minmax.ctypes.data, 16, out.data_ptr(), threads or coder_threads()))
    return out


def range_decode_rows_batch(strings, E: int, rows: np.ndarray, row_offset: np.ndarray, minmax: np.ndarray,
                            threads: int = 0) -> np.ndarray:
    """-> int16 [B,E] symbols (0-based; add min_v)."""
    L = _lib.lib()
    B = len(strings)
    bufs = [np.frombuffer(bytes(s), np.uint8) if len(s) else np.zeros(1, np.uint8) for s in strings]
    ptrs = (C.c_void_p * B)(*[b.ctypes.data for b in bufs])
    nbytes = np.array([len(s) for s in strings], np.int64)
    rows = np.ascontiguousarray(rows)
    row_offset = np.ascontiguousarray(row_offset, dtype=np.int64)
    minmax = np.ascontiguousarray(minmax, dtype=np.int32)
    sym = np.empty((B, E), np.int16)
    _lib.check(L.pcgc_range_decode_rows_batch(ptrs, nbytes.ctypes.data, B, E, rows.ctypes.data, row_offset.ctypes.data,
                                              minmax.ctypes.data, 16, sym.ctypes.data, threads or coder_threads()))
    return sym
