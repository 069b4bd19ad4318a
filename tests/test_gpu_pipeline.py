"""The chunked encode / decode pipelines of pcgcv1_b200/transform.py: whatever the schedule (decode ramp, how many cubes an encoder
launch codes, whether the caller consumes the result part by part) the streams and the reconstructions are the same bits."""
import numpy as np
import pytest
import torch

from pcgcv1_b200 import runtime, synthetic, transform
from pcgcv1_b200.dataprocess import inout_points
from pcgcv1_b200.models import model_voxception

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cloud():
    cubes, _, nums = synthetic.workload("vox10", seed=0, max_cubes=140)      # > 64 cubes: several chunks on both sides
    return cubes, nums


@pytest.fixture(scope="module")
def stream(codec, cloud):
    out = transform.compress_hyper(cloud[0], model_voxception, "")
    return [o.numpy() for o in out]


def test_pending_result_behaves_like_a_device_result_and_select_consumes_it_in_parts(codec, cloud, stream):
    cubes, nums = cloud
    xs = transform.decompress_hyper(*stream, model_voxception, "")
    assert isinstance(xs, runtime.PendingDeviceResult) and not xs.finalized
    assert len(xs) == len(cubes) and xs.shape == (len(cubes), 64, 64, 64, 1)
    assert [a for a, _, _ in xs.parts] == sorted(a for a, _, _ in xs.parts) and xs.parts[0][0] == 0 and xs.parts[-1][1] == len(cubes)
    mask_parts = inout_points.select_voxels(xs, nums, 1.0, codec=codec, dtype="uint8")          # pipelined path
    assert xs.finalized
    mask_plain = inout_points.select_voxels(xs.tensor, nums, 1.0, codec=codec, dtype="uint8")   # plain path on the same logits
    assert mask_parts.dtype == np.uint8 and np.array_equal(mask_parts, mask_plain)
    assert (mask_parts.reshape(len(cubes), -1).sum(1) >= nums).all()
    # float32 form (the reference's dtype) through the pipelined path
    xs2 = transform.decompress_hyper(*stream, model_voxception, "")
    m32 = inout_points.select_voxels(xs2, nums, 1.0, codec=codec)
    assert m32.dtype == np.float32 and np.array_equal(m32, mask_plain.astype(np.float32))
    # .numpy() on a pending result waits for all of it
    xs3 = transform.decompress_hyper(*stream, model_voxception, "")
    assert np.array_equal(xs3.numpy(), xs.tensor.cpu().numpy())
    # a k larger than the cube raises like get_adaptive_thres (inout_points.py:170-179), before any work is queued
    xs4 = transform.decompress_hyper(*stream, model_voxception, "")
    with pytest.raises(IndexError):
        inout_points.select_voxels(xs4, np.full(len(cubes), 300000), 1.0, codec=codec)
    xs4.finalize()


@pytest.mark.parametrize("ramp,rest", [("64", "512"), ("8,24,64", "512"), ("16", "32"), ("200", "512")])
def test_reconstruction_does_not_depend_on_the_decode_schedule(codec, cloud, stream, monkeypatch, ramp, rest):
    ref = transform.decompress_hyper(*stream, model_voxception, "").tensor.clone()
    monkeypatch.setenv("PCGC_DEC_RAMP", ramp)
    monkeypatch.setenv("PCGC_DEC_CHUNK", rest)
    got = transform.decompress_hyper(*stream, model_voxception, "").tensor
    assert torch.equal(ref, got)


def test_streams_of_several_chunks_equal_the_host_coders(codec, cloud, stream, monkeypatch):
    """140 cubes (several encoder chunks): the GPU path's y strings, their min / max, the z string and its min / max are the bytes
    the host coder writes (PCGC_CODER=host codes every chunk's strings and the hyper string on the host after the GPU)."""
    monkeypatch.setenv("PCGC_CODER", "host")
    host = [o.numpy() for o in transform.compress_hyper(cloud[0], model_voxception, "")]
    assert bytes(host[4]) == bytes(stream[4]) and int(host[5]) == int(stream[5]) and int(host[6]) == int(stream[6])
    assert [bytes(s) for s in host[0]] == [bytes(s) for s in stream[0]]
    assert np.array_equal(host[1], stream[1]) and np.array_equal(host[2], stream[2])


@pytest.mark.parametrize("reps,per_launch", [(1, 1), (1, 9), (1, 64), (2, 280), (32, 4480)])
def test_strings_do_not_depend_on_how_the_encoder_launch_is_spread(codec, cloud, stream, reps, per_launch):
    """The encoder pads its one-warp CTAs with unused shared memory by the number of cubes in the launch (98 KB per CTA up to 148
    cubes, 64 KB at 280, none from 4441 on): the 140 cubes' strings are the same bytes whatever the launch size.  (The decoder's
    side is covered by the round trips.)"""
    from pcgcv1_b200.models.conditional_entropy_model import SymmetricConditional
    cem = SymmetricConditional().bind(codec)
    iv = transform.encode_on_device(codec, transform._bottleneck(codec, 8), cem, cloud[0])[0].repeat(reps, 1)
    got = []
    for a in range(0, iv.shape[0], per_launch):
        packed, offsets = cem.encode_dev(iv[a:a + per_launch])
        codec.synchronize()
        o, blob = offsets.cpu().numpy(), packed.cpu().numpy()
        got += [blob[o[i]:o[i + 1]].tobytes() for i in range(len(o) - 1)]
    assert got == [bytes(s) for s in stream[0]] * reps


def test_factorized_decode_is_progressive_and_equal_to_the_plain_form(codec_simple, cloud, monkeypatch):
    from pcgcv1_b200.models import model_simple
    cubes, nums = cloud
    s, mn, mx, shp = transform.compress_factorized(cubes, model_simple, "")
    args = (s.numpy(), mn.numpy(), mx.numpy(), shp.numpy(), model_simple, "")
    xs = transform.decompress_factorized(*args)
    assert isinstance(xs, runtime.PendingDeviceResult) and len(xs.parts) == 3            # 140 cubes in parts of 48
    mask = inout_points.select_voxels(xs, nums, 1.0, codec=codec_simple, dtype="uint8")
    monkeypatch.setattr(transform, "_FACT_PART", 1 << 20)                                 # one piece: the plain form
    plain = transform.decompress_factorized(*args)
    assert not isinstance(plain, runtime.PendingDeviceResult)
    assert torch.equal(xs.tensor, plain.tensor)
    assert np.array_equal(mask, inout_points.select_voxels(plain, nums, 1.0, codec=codec_simple, dtype="uint8"))


@pytest.mark.parametrize("B", [0, 1, 9, 33, 65, 97])
def test_round_trip_at_chunk_boundaries(codec, cloud, B):
    """Cube counts on both sides of every chunk boundary of the two pipelines (decode ramp 8 / 24 / 64, encode chunks of 64),
    the empty cloud included: the decoder's reconstruction equals the encoder-side one bit for bit and the masks hold >= k voxels."""
    cubes, nums = cloud[0][:B], cloud[1][:B]
    out = transform.compress_hyper(cubes, model_voxception, "", decompress=True)
    host = [o.numpy() for o in out[:8]]
    assert len(host[0]) == B and list(host[7]) == [B, 8, 8, 8, 8]
    xs = transform.decompress_hyper(*host, model_voxception, "")
    mask = inout_points.select_voxels(xs, nums, 1.0, codec=codec, dtype="uint8")
    assert mask.shape == (B, 64, 64, 64, 1)
    assert np.array_equal(xs.numpy(), out[8].numpy())
    if B:
        assert (mask.reshape(B, -1).sum(1) >= nums).all()


def test_factorized_round_trip_just_over_one_part(codec_simple, cloud):
    from pcgcv1_b200.models import model_simple
    cubes = cloud[0][:49]
    s, mn, mx, shp = transform.compress_factorized(cubes, model_simple, "")
    xs = transform.decompress_factorized(s.numpy(), mn.numpy(), mx.numpy(), shp.numpy(), model_simple, "")
    ref = codec_simple.synthesis(torch.round(codec_simple.analysis(codec_simple.to_device(cubes))))
    assert torch.equal(xs.tensor, ref)
