"""Host part of libpcgc_b200.so (range coder, 16-bit CDF normaliser) against the oracle.  CPU only:
these entry points take no ctx and need no GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import coder
from oracle.entropy import SymmetricConditionalOracle
from pcgcv1_b200 import _lib, runtime


def _lib_cdf(pmf, precision=16):
    L = _lib.lib()
    pmf = np.ascontiguousarray(pmf, np.float32)
    out = np.empty((pmf.shape[0], pmf.shape[1] + 1), np.int32)
    rc = L.pcgc_pmf_to_quantized_cdf(pmf.ctypes.data, pmf.shape[0], pmf.shape[1], precision, out.ctypes.data)
    assert rc == 0
    return out


def test_oracle_c_equals_python_definition():
    rng = np.random.default_rng(3)
    for _ in range(60):
        n, rows = int(rng.integers(2, 20)), int(rng.integers(1, 4))
        pmf = rng.random((rows, n)).astype(np.float32) ** int(rng.integers(1, 6))
        pmf = np.maximum(pmf / pmf.sum(-1, keepdims=True) * rng.choice([1.0, 0.99, 1.01]), 1e-9).astype(np.float32)
        a = coder.pmf_to_quantized_cdf(pmf, 16, force_python=True)
        assert np.array_equal(a, coder.pmf_to_quantized_cdf(pmf, 16))
        cnt = int(rng.integers(0, 300))
        sym = rng.integers(0, n, cnt).astype(np.int16)
        idx = rng.integers(0, rows, cnt).astype(np.int32)
        s = coder.range_encode(sym, a, idx, force_python=True)
        assert s == coder.range_encode(sym, a, idx)
        assert np.array_equal(coder.range_decode(s, cnt, a, idx, force_python=True), sym)
        assert np.array_equal(coder.range_decode(s, cnt, a, idx), sym)


def test_normaliser_equals_greedy_definition():
    """Water-filling normaliser == step-by-step greedy of the oracle, incl. large deficits."""
    rng = np.random.default_rng(0)
    for _ in range(150):
        n, rows = int(rng.integers(2, 64)), int(rng.integers(1, 6))
        pmf = rng.random((rows, n)).astype(np.float32) ** int(rng.integers(1, 10))
        pmf /= pmf.sum(-1, keepdims=True)
        pmf = np.maximum(pmf * rng.choice([1.0, 0.97, 0.9, 0.5, 0.2, 1.02]), 1e-9).astype(np.float32)
        ref = coder.pmf_to_quantized_cdf(pmf, 16)
        out = _lib_cdf(pmf)
        assert np.array_equal(ref, out)
        assert (out[:, 0] == 0).all() and (out[:, -1] == 65536).all() and (np.diff(out, axis=-1) >= 1).all()


@pytest.mark.parametrize("N", [2, 5, 13, 31, 64])
def test_normaliser_on_laplace_rows(N):
    rng = np.random.default_rng(N)
    loc = rng.normal(0, 2, 200).astype(np.float32)
    sc = (np.abs(rng.normal(0, 1, 200)) + 1e-3).astype(np.float32)
    sc[:4] = [1e-9, 1e-4, 30.0, 1000.0]
    mn = -(N // 2)
    pmf = SymmetricConditionalOracle().pmf(loc, sc, mn, mn + N - 1)
    assert np.array_equal(coder.pmf_to_quantized_cdf(pmf, 16), _lib_cdf(pmf))


def test_single_symbol_alphabet_is_rejected():
    L = _lib.lib()
    pmf = np.ones((1, 1), np.float32)
    out = np.empty((1, 2), np.int32)
    assert L.pcgc_pmf_to_quantized_cdf(pmf.ctypes.data, 1, 1, 16, out.ctypes.data) == -2     # BAD_RANGE
    with pytest.raises(ValueError):
        coder.pmf_to_quantized_cdf(pmf, 16)


def test_range_coder_bytes_equal_oracle_and_round_trip():
    rng = np.random.default_rng(1)
    for _ in range(80):
        n, rows = int(rng.integers(2, 33)), int(rng.integers(1, 9))
        pmf = rng.random((rows, n)).astype(np.float32) ** 3
        pmf = np.maximum(pmf / pmf.sum(-1, keepdims=True), 1e-9).astype(np.float32)
        cdf = coder.pmf_to_quantized_cdf(pmf, 16)
        cnt = int(rng.integers(0, 3000))
        sym = rng.integers(0, n, cnt).astype(np.int16)
        idx = (np.arange(cnt) % rows).astype(np.int32)
        s = runtime.range_encode(sym, cdf)
        assert s == coder.range_encode(sym, cdf, idx)
        assert np.array_equal(runtime.range_decode(s, cnt, cdf), sym)


def test_carry_propagation_stress():
    """Skewed tables force long 0xFFFF runs and carries through the delayed word."""
    rng = np.random.default_rng(2)
    for hi_first in (False, True):
        v = np.array([65533, 1, 1, 1] if hi_first else [1, 1, 1, 65533])
        cdf = np.concatenate([[0], np.cumsum(v)]).astype(np.int32)[None]
        top = 0 if hi_first else 3
        for _ in range(40):
            cnt = int(rng.integers(1, 4000))
            sym = np.where(rng.random(cnt) < 0.999, top, rng.integers(0, 4, cnt)).astype(np.int16)
            s = runtime.range_encode(sym, cdf)
            assert s == coder.range_encode(sym, cdf, np.zeros(cnt, np.int32), force_python=True)
            assert np.array_equal(runtime.range_decode(s, cnt, cdf), sym)


def test_interval_and_row_entry_points_batch():
    """The per-element forms used by the conditional model: intervals in, uint16 rows out."""
    rng = np.random.default_rng(5)
    B, E = 5, 777
    mm = np.array([[-3, 4], [0, 1], [-15, 15], [-1, 1], [2, 9]], np.int32)
    sc_or = SymmetricConditionalOracle()
    ivs = np.zeros((B, E), np.uint32)
    syms = []
    rows_all, off = [], [0]
    for b in range(B):
        N = mm[b, 1] - mm[b, 0] + 1
        loc = rng.normal((mm[b, 0] + mm[b, 1]) / 2, 1.5, E).astype(np.float32)
        scale = (np.abs(rng.normal(0, 1, E)) + 0.01).astype(np.float32)
        cdf = coder.pmf_to_quantized_cdf(sc_or.pmf(loc, scale, int(mm[b, 0]), int(mm[b, 1])), 16)
        sym = rng.integers(0, N, E)
        lower = cdf[np.arange(E), sym].astype(np.uint32)
        width = (cdf[np.arange(E), sym + 1] - cdf[np.arange(E), sym]).astype(np.uint32)
        ivs[b] = lower | ((width - 1) << 16)
        syms.append(sym)
        rows_all.append(cdf[:, :N].astype(np.uint16).reshape(-1))
        off.append(off[-1] + E * N)
        # bytes equal the oracle's
        ref = coder.range_encode(sym.astype(np.int16), cdf, np.arange(E, dtype=np.int32))
        assert runtime.range_encode_intervals_batch(ivs[b:b + 1], 1)[0] == ref
    strings = runtime.range_encode_intervals_batch(ivs, 3)
    dec = runtime.range_decode_rows_batch(strings, E, np.concatenate(rows_all), np.array(off, np.int64), mm, 3)
    for b in range(B):
        assert np.array_equal(dec[b], syms[b])


def test_coded_size_close_to_entropy():
    rng = np.random.default_rng(7)
    pmf = np.array([[0.5, 0.25, 0.125, 0.125]], np.float32)
    cdf = coder.pmf_to_quantized_cdf(pmf, 16)
    n = 20000
    sym = rng.choice(4, n, p=pmf[0]).astype(np.int16)
    s = runtime.range_encode(sym, cdf)
    ideal_bits = -np.log2(pmf[0][sym]).sum()
    assert len(s) * 8 <= ideal_bits + 64
    assert len(s) * 8 >= ideal_bits - 64


def test_encoder16_equals_generic_encoder():
    """range_coder.h has two encoder state machines: the generic 64-bit one (host batch coder) and RangeEncoder16 (32-bit base +
    carry flag, what the GPU encoder runs; reachable on the host through pcgc_range_encode_intervals at precision 16).  Same
    bytes on random intervals, including long carry chains (tiny intervals at the top of the range) and certain symbols."""
    import ctypes as C
    from pcgcv1_b200 import _lib, runtime
    L = _lib.lib()
    rng = np.random.default_rng(5)
    cases = []
    for n, kind in ((1, "any"), (2, "any"), (5000, "any"), (20000, "top"), (20000, "sure"), (3000, "tiny"), (0, "any")):
        if kind == "any":
            lower = rng.integers(0, 65535, n)
            width = np.minimum(rng.integers(1, 65536, n), 65536 - lower)
        elif kind == "top":                   # intervals hugging the top of the range: carries and 0xFFFF runs
            width = rng.integers(1, 4, n)
            lower = 65536 - width - rng.integers(0, 2, n) * rng.integers(0, 3, n)
            lower = np.clip(lower, 0, 65536 - width)
        elif kind == "sure":                  # p ~ 1 symbols: the interval barely shrinks
            lower = np.zeros(n, np.int64)
            width = np.full(n, 65535)
            lower[::7] = 1
        else:                                 # width 1 everywhere: 16 bits per symbol
            lower = rng.integers(0, 65536, n)
            width = np.ones(n, np.int64)
        cases.append((lower.astype(np.uint32) | ((width - 1).astype(np.uint32) << 16)).astype(np.uint32))
    for iv in cases:
        n = iv.size
        cap = 2 * n + 64
        out = np.zeros(cap, np.uint8)
        ln = C.c_int64()
        src = iv if n else np.zeros(1, np.uint32)
        assert L.pcgc_range_encode_intervals(src.ctypes.data, n, 16, out.ctypes.data, cap, C.byref(ln)) == 0
        fast = out[:ln.value].tobytes()
        if n:
            generic = runtime.range_encode_intervals_batch(iv[None], 1)[0]
            assert fast == generic


def test_shared_edge_likelihoods_equal_the_per_symbol_form(tmp_path):
    """tools/cdf_check.cpp (host build of det_math.h, the header the CUDA kernels compile): the shared-edge likelihood row
    det_laplace_pmf_row gives the same bits as the per-symbol likelihood on 300 000 random Laplace rows (all symbol counts up to 32)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(str(tmp_path), "cdf_check")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-I", os.path.join(root, "pcgcv1_b200", "csrc"), "-o", exe,
                    os.path.join(root, "tools", "cdf_check.cpp")], check=True, capture_output=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "0 mismatches" in r.stdout.strip().splitlines()[-1]


def test_every_encoder_equals_the_literal_upstream_state_machine():
    """oracle.coder.UpstreamRangeEncoder restates tensorflow/contrib/coder's RangeEncoder::Encode / Finalize statement by statement
    (32-bit wrapping base, delay_ word + byte count, Finalize's three cases).  The carry-propagating coders -- the oracle's Python
    definition, the oracle's C, the library's generic host encoder and its RangeEncoder16 (what the GPU encoder runs) -- must
    write the same bytes, including strings that END in the delayed (wrapped) state and strings whose base ends at zero."""
    L = _lib.lib()
    rng = np.random.default_rng(11)
    ended_delayed = ended_zero = total = 0
    for trial in range(1500):
        N = int(rng.integers(2, 33))
        cuts = np.sort(rng.choice(np.arange(1, 65536), N - 1, replace=False))
        cdf = np.concatenate([[0], cuts, [65536]]).astype(np.int32)
        n = int(rng.integers(0, 120))
        kind = trial % 3
        if kind == 0:
            sym = rng.integers(0, N, n)
        elif kind == 1:                                   # mostly the first symbol (lower = 0): bases that end at zero
            sym = np.where(rng.random(n) < 0.7, 0, rng.integers(0, N, n))
        else:                                             # mostly the last symbol (upper = 2^16): intervals at the top, long delays
            sym = np.where(rng.random(n) < 0.7, N - 1, rng.integers(0, N, n))
        sym = sym.astype(np.int16)
        up = coder.UpstreamRangeEncoder(16)
        for s in sym.tolist():
            up.encode(int(cdf[s]), int(cdf[s + 1]))
        ended_delayed += up.delay != 0
        ended_zero += up.delay == 0 and up.base == 0 and n > 0
        want = up.finish()
        idx = np.zeros(n, np.int32)
        assert coder.range_encode(sym, cdf[None], idx, force_python=True) == want, trial
        assert coder.range_encode(sym, cdf[None], idx) == want, trial
        assert runtime.range_encode(sym, cdf[None]) == want, trial
        if n:
            iv = (cdf[sym].astype(np.uint32) | ((cdf[sym + 1] - cdf[sym] - 1).astype(np.uint32) << 16)).astype(np.uint32)
            out = np.zeros(2 * n + 64, np.uint8)
            ln = C.c_int64()
            assert L.pcgc_range_encode_intervals(iv.ctypes.data, n, 16, out.ctypes.data, out.size, C.byref(ln)) == 0
            assert out[:ln.value].tobytes() == want, trial
            assert runtime.range_encode_intervals_batch(iv[None], 1)[0] == want, trial
        assert np.array_equal(coder.range_decode(want, n, cdf[None], idx), sym)
        assert np.array_equal(runtime.range_decode(want, n, cdf[None]), sym)
        total += 1
    print("%d strings: %d ended in the delayed state, %d with base 0" % (total, ended_delayed, ended_zero))
    assert ended_delayed > 30 and ended_zero > 10
