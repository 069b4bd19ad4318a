"""Far-field tiles across calls (DESIGN 4.1): the analysis 64^3 stage keeps each layer in a buffer of its own per sub-batch slot and
skips the far tiles a slot already holds the empty cube's values for.  Whatever ran in a slot before -- another cloud, a synthesis call,
a shorter sub-batch, a float32 batch computed without masks, other weights -- the latents must be the same BITS as with every tile
computed (PCGC_FARFIELD=0).  Each case computes its references first: a call with every tile computed leaves the slots unknown, so the
far-field calls after it restore them and then track them from cube to cube."""
import numpy as np
import pytest
import torch

from pcgcv1_b200 import runtime, synthetic, weights as W

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ffcodec():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return runtime.Codec("voxception", "", weights=W.synthetic_weights("voxception"))


@pytest.fixture(scope="module")
def clouds():
    a, _, _ = synthetic.workload("vox10", seed=0)
    b, _, _ = synthetic.workload("vox10", seed=1)
    return a, b


def _special():
    x = np.zeros((6, 64, 64, 64, 1), np.uint8)
    x[1][0, 0, 0, 0] = 1                                                       # corner
    x[2][63, 31, 0, 0] = 1                                                     # edge
    x[3][32, 32, 32, 0] = 1                                                    # centre
    x[4][:, 40, :, 0] = 1                                                      # a full plane
    x[5][17, 5, 60, 0] = 1                                                     # x[0] stays empty
    return x


def _run(codec, monkeypatch, x, ff):
    monkeypatch.setenv("PCGC_FARFIELD", "1" if ff else "0")
    t = x if isinstance(x, torch.Tensor) else codec.to_device(x)
    y = codec.analysis(t).clone()
    codec.synchronize()
    return y


def _refs(codec, monkeypatch, *xs):
    return [_run(codec, monkeypatch, x, False) for x in xs]


def test_two_clouds_back_to_back(ffcodec, clouds, monkeypatch):
    a, b = clouds[0][:64], clouds[1][:64]
    ra, rb = _refs(ffcodec, monkeypatch, a, b)
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)
    assert torch.equal(_run(ffcodec, monkeypatch, b, True), rb)          # restores the near tiles of a
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)


def test_synthesis_between_calls(ffcodec, clouds, monkeypatch):
    a = clouds[0][:64]
    (ra,) = _refs(ffcodec, monkeypatch, a)
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)
    ffcodec.synthesis(ra)
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)


def test_sub_batch_sizes_change(ffcodec, clouds, monkeypatch):
    a, b = clouds[0][:64], clouds[1][:17]
    ra, rb = _refs(ffcodec, monkeypatch, a, b)
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)
    assert torch.equal(_run(ffcodec, monkeypatch, b, True), rb)          # slots 17.. keep the masks of a
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)


def test_float32_batch_between_uint8_batches(ffcodec, clouds, monkeypatch):
    a, b = clouds[0][:64], clouds[1][:64]
    ra, rb = _refs(ffcodec, monkeypatch, a, b)
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)
    assert torch.equal(_run(ffcodec, monkeypatch, ffcodec.to_device(b).float(), True), rb)   # float32: every tile computed
    assert torch.equal(_run(ffcodec, monkeypatch, a, True), ra)


def test_special_cubes_and_two_sub_batches(ffcodec, clouds, monkeypatch):
    s = _special()
    x = np.concatenate([clouds[0][:70], s])                                   # 76 cubes: two sub-batches of 64 and 12
    rs, rx, r70 = _refs(ffcodec, monkeypatch, s, x, clouds[1][:70])
    assert torch.equal(_run(ffcodec, monkeypatch, s, True), rs)
    assert torch.equal(_run(ffcodec, monkeypatch, x, True), rx)
    assert torch.equal(_run(ffcodec, monkeypatch, clouds[1][:70], True), r70)
    assert torch.equal(_run(ffcodec, monkeypatch, s, True), rs)


def test_new_weights_between_calls(clouds, monkeypatch):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    a, b = clouds[0][:64], clouds[1][:64]
    c = runtime.Codec("voxception", "", weights=W.synthetic_weights("voxception"))
    other = runtime.Codec("voxception", "", weights=W.synthetic_weights("voxception", seed=77))
    (rb,) = _refs(other, monkeypatch, b)
    del other
    _run(c, monkeypatch, a, True)
    c.weights = W.synthetic_weights("voxception", seed=77)
    c._load_weights()
    assert torch.equal(_run(c, monkeypatch, b, True), rb)


def test_streams_of_two_clouds(clouds, monkeypatch):
    from pcgcv1_b200 import transform
    from pcgcv1_b200.models import model_voxception
    a, b = clouds[0][:40], clouds[1][:40]

    def streams(ff):
        monkeypatch.setenv("PCGC_FARFIELD", "1" if ff else "0")
        return [[np.asarray(o.numpy()) for o in transform.compress_hyper(x, model_voxception, "")] for x in (a, b)]

    ref = streams(False)
    got = streams(True)
    for u, v in zip(ref, got):
        for p, q in zip(u, v):
            assert np.array_equal(p, q)
