"""GPU-side range coder (csrc/gpu_coder.cu) and the bit-exact CDF builders (csrc/det_math.h).

What is pinned here (the bar for integer / byte work is bit-exact):
  * strings written by the GPU encoder == strings written by the host coder of the same library, byte for byte;
  * symbols read by the GPU decoder == symbols read by the host decoder == the encoder's input;
  * per-element CDF rows built on the GPU == rows built by the library's host twin (pcgc_host_laplace_cdf), 100 % of rows,
    and the same for the factorized (hyper-latent) table;
  * a CPU can decode a GPU-written hyper stream: host-twin rows + the ORACLE's C range decoder give back the GPU's y_hat.
``tf.contrib.coder`` itself stays unpinned (no wheel, no golden stream in the reference): "symbol-compatible", not
"byte-identical to TF".
"""
import os

import numpy as np
import pytest
import torch

from oracle import coder as ocoder, entropy
from pcgcv1_b200 import runtime, synthetic, transform
from pcgcv1_b200.models import conditional_entropy_model, entropy_model, model_voxception

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def latents(codec):
    """y, loc, scale of 6 cubes of the vox10 workload straight from the CUDA transforms."""
    cubes, _, nums = synthetic.workload("vox10", seed=0, max_cubes=6)
    y = codec.analysis(codec.to_device(cubes))
    z_hat = torch.round(codec.hyper_encode(y))
    loc, scale = codec.hyper_decode(z_hat, 1e-9)
    B = y.shape[0]
    return dict(B=B, y=y.reshape(B, -1), loc=loc.reshape(B, -1), scale=scale.reshape(B, -1))


def _host_strings(iv_host):
    return runtime.range_encode_intervals_batch(iv_host, 4)


def test_gpu_encoder_is_byte_identical_to_host_coder(codec, latents):
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    iv, mm = cem.intervals_dev(latents["y"], latents["loc"], latents["scale"])
    packed, offsets = cem.encode_dev(iv)
    codec.synchronize()
    off = offsets.cpu().numpy()
    blob = packed.cpu().numpy()
    gpu = [blob[off[b]:off[b + 1]].tobytes() for b in range(latents["B"])]
    host = _host_strings(iv.cpu().numpy())
    assert [len(s) for s in gpu] == [len(s) for s in host]
    assert gpu == host
    assert all(len(s) > 100 for s in gpu)


def test_gpu_decoder_reads_what_both_encoders_wrote(codec, latents):
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    B = latents["B"]
    iv, mm = cem.intervals_dev(latents["y"], latents["loc"], latents["scale"])
    mm_h = mm.cpu().numpy()
    strings = _host_strings(iv.cpu().numpy())
    packed, offsets = codec.upload_strings(strings)
    y_hat = cem.decode_dev(packed, offsets, latents["loc"], latents["scale"], mm_h[:, 0], mm_h[:, 1])
    codec.synchronize()
    want = torch.round(latents["y"])
    assert torch.equal(y_hat, want)
    # the host decoder on GPU rows gives the same symbols
    rows, off = codec.laplace_cdf(latents["loc"], latents["scale"], mm_h)
    host = runtime.range_decode_rows_batch(strings, latents["y"].shape[1], rows.cpu().numpy(), off, mm_h, 4)
    assert np.array_equal(host.astype(np.int32) + mm_h[:, :1], want.cpu().numpy().astype(np.int32))


def test_cdf_rows_bit_identical_to_host_twin_and_cpu_decodes_gpu_stream(codec, latents):
    """100 % of the GPU's CDF rows equal the host twin's; then a CPU-only decode (host-twin rows + the oracle's C range decoder)
    of the GPU-written strings returns the GPU's quantised latents."""
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    B, E = latents["B"], latents["y"].shape[1]
    iv, mm = cem.intervals_dev(latents["y"], latents["loc"], latents["scale"])
    mm_h = mm.cpu().numpy()
    rows_gpu, off = codec.laplace_cdf(latents["loc"], latents["scale"], mm_h)
    rows_gpu = rows_gpu.cpu().numpy().view(np.uint16)
    loc_h, scale_h = latents["loc"].cpu().numpy(), latents["scale"].cpu().numpy()
    rows_cpu, off2 = runtime.host_laplace_cdf(loc_h, scale_h, mm_h)
    assert np.array_equal(off, off2)
    assert np.array_equal(rows_gpu, rows_cpu), "%d of %d CDF entries differ" % ((rows_gpu != rows_cpu).sum(), rows_cpu.size)
    # GPU-written strings, decoded without the GPU
    packed, offsets = cem.encode_dev(iv)
    codec.synchronize()
    o = offsets.cpu().numpy()
    blob = packed.cpu().numpy()
    want = torch.round(latents["y"]).cpu().numpy().astype(np.int32)
    for b in range(2):
        n = int(mm_h[b, 1] - mm_h[b, 0] + 1)
        table = np.concatenate([rows_cpu[off[b]:off[b + 1]].reshape(E, n).astype(np.int32), np.full((E, 1), 65536, np.int32)], 1)
        sym = ocoder.range_decode(blob[o[b]:o[b + 1]].tobytes(), E, table, np.arange(E, dtype=np.int32), 16)
        assert np.array_equal(sym.astype(np.int32) + mm_h[b, 0], want[b])


def test_factorized_table_bit_identical_to_host_twin(codec):
    for mn, mx in ((-3, 4), (-20, 17), (0, 1), (-31, 31)):
        a = codec.factorized_cdf(0, mn, mx)
        b = codec.factorized_cdf_host(0, mn, mx)
        assert np.array_equal(a, b)
        assert (np.diff(a, axis=1) >= 1).all() and (a[:, -1] == 65536).all()


@pytest.mark.parametrize("span", [2, 33, 40, 64])
def test_gpu_coder_wide_and_narrow_alphabets(codec, span):
    """Symbol counts on both sides of the decoder's 32-lane boundary (N = 2 .. 64)."""
    rng = np.random.default_rng(span)
    B, E = 3, 4096
    lo = -(span // 2)
    y = rng.integers(lo, lo + span, size=(B, E)).astype(np.float32)
    y[:, 0], y[:, 1] = lo, lo + span - 1                                  # every cube spans the full range
    loc = (y + rng.normal(0, 2.0, size=y.shape)).astype(np.float32)
    scale = rng.uniform(0.3, 6.0, size=y.shape).astype(np.float32)
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    yd, ld, sd = codec.to_device(y), codec.to_device(loc), codec.to_device(scale)
    iv, mm = cem.intervals_dev(yd, ld, sd)
    mm_h = mm.cpu().numpy()
    assert (mm_h[:, 1] - mm_h[:, 0] + 1 == span).all()
    packed, offsets = cem.encode_dev(iv)
    codec.synchronize()
    o, blob = offsets.cpu().numpy(), packed.cpu().numpy()
    gpu = [blob[o[b]:o[b + 1]].tobytes() for b in range(B)]
    assert gpu == _host_strings(iv.cpu().numpy())
    y_hat = cem.decode_dev(packed, offsets, ld, sd, mm_h[:, 0], mm_h[:, 1])
    codec.synchronize()
    assert torch.equal(y_hat, yd)


def test_gpu_coder_empty_and_ragged_strings(codec):
    """Cubes whose symbols are all (almost) certain code to short strings of zero words -- the upstream coder writes every word it
    renormalises out, only the LAST word is trimmed (Finalize), so such a string is not empty; the packed buffer then holds ragged
    pieces."""
    B, E = 4, 2048
    y = np.zeros((B, E), np.float32)
    y[:, 0] = 1.0                                                           # two symbols (N >= 2 is a format requirement)
    rng = np.random.default_rng(0)
    y[2] = rng.integers(0, 2, E)
    loc = y.copy()
    scale = np.full((B, E), 1e-3, np.float32)                               # p(symbol) ~ 1
    scale[2] = 3.0
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    yd, ld, sd = codec.to_device(y), codec.to_device(loc), codec.to_device(scale)
    iv, mm = cem.intervals_dev(yd, ld, sd)
    packed, offsets = cem.encode_dev(iv)
    codec.synchronize()
    o, blob = offsets.cpu().numpy(), packed.cpu().numpy()
    lens = np.diff(o)
    assert lens[2] > 1500 and lens[0] < lens[2] // 4 and lens[1] == lens[0]
    iv_h = iv.cpu().numpy().view(np.uint32)
    up = ocoder.UpstreamRangeEncoder(16)
    for w in iv_h[0].tolist():
        up.encode(w & 0xFFFF, (w & 0xFFFF) + (w >> 16) + 1)
    assert blob[o[0]:o[1]].tobytes() == up.finish()
    assert [blob[o[b]:o[b + 1]].tobytes() for b in range(B)] == _host_strings(iv.cpu().numpy())
    mm_h = mm.cpu().numpy()
    y_hat = cem.decode_dev(packed, offsets, ld, sd, mm_h[:, 0], mm_h[:, 1])
    codec.synchronize()
    assert torch.equal(y_hat, yd)


def test_hyper_streams_do_not_depend_on_where_the_coder_runs(codec, monkeypatch):
    """transform.compress_hyper with PCGC_CODER=gpu and =host writes the same bytes (y strings and their min / max, the z string
    and its min / max); each side decodes the other's."""
    cubes, _, nums = synthetic.workload("vox10", seed=0, max_cubes=20)
    outs = {}
    for mode in ("gpu", "host"):
        monkeypatch.setenv("PCGC_CODER", mode)
        outs[mode] = [o.numpy() for o in transform.compress_hyper(cubes, model_voxception, "")]
    g, h = outs["gpu"], outs["host"]
    assert list(g[0]) == list(h[0]) and g[4] == h[4] and int(g[5]) == int(h[5]) and int(g[6]) == int(h[6])
    assert np.array_equal(g[1], h[1]) and np.array_equal(g[2], h[2])
    monkeypatch.setenv("PCGC_CODER", "gpu")
    x_gpu = transform.decompress_hyper(*h, model_voxception, "").numpy()
    monkeypatch.setenv("PCGC_CODER", "host")
    x_host = transform.decompress_hyper(*g, model_voxception, "").numpy()
    assert np.array_equal(x_gpu, x_host)


def test_noise_quantisation_matches_oracle_philox(codec, latents):
    """training=True ("noise", entropy_model.py:105-107, conditional_entropy_model.py:62-64): the draws are the oracle's
    Philox4x32-10 stream bit for bit; likelihoods at the noisy values within 1e-3."""
    seed = 20260117
    B = 2
    y = latents["y"][:B].reshape(B, 16, 16, 16, 16)
    loc, scale = latents["loc"][:B].reshape(y.shape), latents["scale"][:B].reshape(y.shape)
    cem = conditional_entropy_model.SymmetricConditional().bind(codec)
    y_t, p = cem(y, loc, scale, training=True, seed=seed)
    y_h = y.cpu().numpy()
    ref_y, ref_p = entropy.SymmetricConditionalOracle()(y_h, loc.cpu().numpy(), scale.cpu().numpy(), training=True, seed=seed)
    assert np.array_equal(y_t.numpy(), ref_y)
    assert np.abs(y_t.numpy() - y_h).max() <= 0.5
    np.testing.assert_allclose(p.numpy(), ref_p, rtol=1e-3, atol=3e-7)
    # a second call without training is back to rounding
    y_r, _ = cem(y, loc, scale)
    assert np.array_equal(y_r.numpy(), np.rint(y_h))
    # factorized model on z
    from pcgcv1_b200 import weights as W
    z = codec.hyper_encode(y)
    eb = entropy_model.EntropyBottleneck().bind(codec, 0)
    z_t, pz = eb(z, training=True, seed=seed)
    eb_or = entropy.EntropyBottleneckOracle(W.net_weights(W.synthetic_weights("voxception"), "estimator"))
    ref_z, ref_pz = eb_or(z.cpu().numpy(), training=True, seed=seed)
    assert np.array_equal(z_t.numpy(), ref_z)
    np.testing.assert_allclose(pz.numpy(), ref_pz, rtol=1e-3, atol=3e-7)


def test_gpu_encoder_equals_the_literal_upstream_state_machine(codec):
    """Raw interval words through the GPU encoder against oracle.coder.UpstreamRangeEncoder (tensorflow/contrib/coder's
    RangeEncoder::Encode / Finalize restated statement by statement): random intervals, intervals with lower = 0 (bases that end at
    zero: nothing is written for the last word, earlier zero words stay) and intervals hugging the top of the range (strings that END
    in the delayed, wrapped state: the value 2^32 is written)."""
    rng = np.random.default_rng(21)
    B, E = 384, 64
    lower = rng.integers(0, 65535, (B, E))
    width = np.minimum(rng.integers(1, 65536, (B, E)), 65536 - lower)
    k = B // 3
    zero = rng.random((k, E)) < 0.7                                            # cubes [k, 2k): mostly [0, w)
    lower[k:2 * k][zero] = 0
    top = rng.random((B - 2 * k, E)) < 0.7                                      # cubes [2k, B): mostly [2^16 - w, 2^16)
    lower[2 * k:][top] = (65536 - width[2 * k:])[top]
    iv = (lower.astype(np.uint32) | ((width - 1).astype(np.uint32) << 16)).astype(np.uint32)
    packed, offsets = codec.gpu_range_encode(codec.to_device(iv.view(np.int32)))
    codec.synchronize()
    o, blob = offsets.cpu().numpy(), packed.cpu().numpy()
    delayed = zero_base = 0
    for b in range(B):
        up = ocoder.UpstreamRangeEncoder(16)
        for lo, w in zip(lower[b].tolist(), width[b].tolist()):
            up.encode(lo, lo + w)
        delayed += up.delay != 0
        zero_base += up.delay == 0 and up.base == 0
        assert blob[o[b]:o[b + 1]].tobytes() == up.finish(), b
    print("%d strings: %d ended in the delayed state, %d with base 0" % (B, delayed, zero_base))
    assert delayed >= 10 and zero_base >= 3
    assert [blob[o[b]:o[b + 1]].tobytes() for b in range(B)] == _host_strings(iv)
