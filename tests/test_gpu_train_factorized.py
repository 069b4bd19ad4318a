"""Factorized-prior training on the GPU (pcgcv1_b200/training.py:FactorizedTrainer, pcgcv1_b200/train_factorized.py): the conv
primitives at the six model_simple layer shapes and both weight-gradient forms against float64 autograd, the whole step against
the oracle (tests/oracle_train_factorized.py), the trained checkpoint in the codec and the loop.  Tolerances are those of
tests/test_gpu_train.py: 2e-5 on outputs / input gradients, 5e-5 on weight / bias gradients, loss terms 5e-5 relative, every
gradient tensor within 2e-3 of its own scale."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import nets, train as otrain
from oracle_train_factorized import forward_backward_factorized
from pcgcv1_b200 import netspec, synthetic, train_factorized as TF, train_hyper as TH, training, weights as W

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMPLE = {l.name: l for l in netspec.simple_analysis() + netspec.simple_synthesis()}


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _layer_case(layer, n, B=2):
    rng = np.random.default_rng(layer.cin * 100 + layer.cout + layer.k + n)
    x = rng.normal(size=(B, n, n, n, layer.cin)).astype(np.float32)
    kern = (rng.normal(size=netspec.kernel_shape(layer)) / math.sqrt(layer.k ** 3 * layer.cin)).astype(np.float32)
    bias = rng.normal(size=layer.cout).astype(np.float32) if layer.bias else None
    return rng, x, kern, bias


def _oracle(layer, x, kern, bias, g):
    xo = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    wo = {"c/kernel": torch.tensor(kern, dtype=torch.float64, requires_grad=True)}
    if layer.bias:
        wo["c/bias"] = torch.tensor(bias, dtype=torch.float64, requires_grad=True)
    fn = nets.conv3d_transpose_same if layer.transposed else nets.conv3d_same
    yo = fn(xo, wo, "c", stride=layer.stride, relu=layer.relu)
    yo.backward(torch.tensor(g, dtype=torch.float64))
    return yo.detach().numpy(), xo.grad.numpy(), wo["c/kernel"].grad.numpy(), (wo["c/bias"].grad.numpy() if layer.bias else None)


def _debug_wgrad(codec, form, x, g, layer, B, n):
    """pcgc_debug_train_wgrad: dW, db (bias layers) and the partial floats of the forced form."""
    dw = torch.empty(netspec.kernel_shape(layer), dtype=torch.float32, device=codec.dev)
    db = torch.empty(layer.cout, dtype=torch.float32, device=codec.dev) if layer.bias else None
    used = C.c_int64(-1)
    codec._stream()
    codec._check(codec.lib.pcgc_debug_train_wgrad(codec.ctx, form, x.data_ptr(), g.data_ptr(), B, n, layer.cin, layer.cout, layer.k, layer.stride,
                                                  int(layer.transposed), dw.data_ptr(), None if db is None else db.data_ptr(), C.byref(used)))
    codec.synchronize()
    return dw.cpu().numpy(), (None if db is None else db.cpu().numpy()), used.value


# every model_simple layer at its own grid and, where the output grid allows (a multiple of 8), at a reduced one
@pytest.mark.parametrize("name,n", [("conv_1", 64), ("conv_1", 16), ("conv_2", 32), ("conv_2", 16), ("conv_3", 16), ("deconv_1", 8),
                                    ("deconv_2", 16), ("deconv_2", 8), ("deconv_3", 32), ("deconv_3", 8)])
def test_simple_layer_primitives_and_both_wgrad_forms_vs_autograd(codec, name, n):
    layer = SIMPLE[name]
    B = 2
    rng, x, kern, bias = _layer_case(layer, n, B)
    ops = training._Ops(codec)
    xd = torch.tensor(x, device=codec.dev, requires_grad=True)
    wd = torch.tensor(kern, device=codec.dev, requires_grad=True)
    bd = torch.tensor(bias, device=codec.dev, requires_grad=True) if layer.bias else None
    y = training._Conv.apply(xd, wd, bd, ops, layer)
    g = rng.normal(size=tuple(y.shape)).astype(np.float32)
    y.backward(torch.tensor(g, device=codec.dev))
    codec.synchronize()
    yo, gxo, gwo, gbo = _oracle(layer, x, kern, bias, g)
    assert _rel(y.detach().cpu().numpy(), yo) < 2e-5
    assert _rel(xd.grad.cpu().numpy(), gxo) < 2e-5
    assert _rel(wd.grad.cpu().numpy(), gwo) < 5e-5
    if layer.bias:
        assert _rel(bd.grad.cpu().numpy(), gbo) < 5e-5
    # both dW forms on the gradient the layer's wgrad sees (behind the ReLU)
    g_eff = np.where(y.detach().cpu().numpy() > 0, g, 0).astype(np.float32) if layer.relu else g
    gd = torch.tensor(g_eff, device=codec.dev)
    xc = torch.tensor(x, device=codec.dev)
    for form in (0, 1):
        dw, db, _ = _debug_wgrad(codec, form, xc, gd, layer, B, n)
        assert _rel(dw, gwo) < 5e-5, form
        if layer.bias:
            assert _rel(db, gbo) < 5e-5, form


def test_wgrad_is_deterministic_and_the_slice_workspace_does_not_grow(codec):
    layer = SIMPLE["conv_1"]
    used = {}
    for B in (2, 16):
        rng = np.random.default_rng(B)
        x = torch.tensor(rng.normal(size=(B, 64, 64, 64, 1)).astype(np.float32), device=codec.dev)
        g = torch.tensor(rng.normal(size=(B, 32, 32, 32, 32)).astype(np.float32), device=codec.dev)
        a, da, used[B] = _debug_wgrad(codec, 1, x, g, layer, B, 64)
        b, db, _ = _debug_wgrad(codec, 1, x, g, layer, B, 64)
        assert np.array_equal(a, b) and np.array_equal(da, db)
        # the product path picks the slice form for this shape: the same bits
        dw = torch.empty_like(torch.tensor(a, device=codec.dev))
        codec._stream()
        codec._check(codec.lib.pcgc_train_conv_wgrad(codec.ctx, x.data_ptr(), g.data_ptr(), B, 64, 1, 32, 9, 2, 0, dw.data_ptr(), None))
        codec.synchronize()
        assert np.array_equal(dw.cpu().numpy(), a)
    assert used[2] == used[16] > 0
    # the tile form's partial buffer is one row per anchor tile: it grows with the batch
    x = torch.zeros((2, 16, 16, 16, 1), dtype=torch.float32, device=codec.dev)
    g = torch.zeros((2, 8, 8, 8, 32), dtype=torch.float32, device=codec.dev)
    t2 = _debug_wgrad(codec, 0, x, g, layer, 2, 16)[2]
    x4 = torch.zeros((4, 16, 16, 16, 1), dtype=torch.float32, device=codec.dev)
    g4 = torch.zeros((4, 8, 8, 8, 32), dtype=torch.float32, device=codec.dev)
    assert _debug_wgrad(codec, 0, x4, g4, layer, 4, 16)[2] == 2 * t2
    # the slice form refuses what it does not cover
    with pytest.raises(Exception):
        _debug_wgrad(codec, 1, x, g, netspec.Layer("c", 1, 32, 7, 2), 2, 16)


# ------------------------------------------------------------------------------------------------- the step
def _terms_keys(distortion):
    return (("focal_full", "focal_empty") if distortion == "focal" else ("zeros", "ones")) + ("distortion", "bpp_ae", "loss")


@pytest.mark.parametrize("model,distortion", [("simple", "bce"), ("simple", "focal"), ("voxception", "bce"), ("voxception", "focal")])
def test_factorized_step_vs_oracle(model, distortion):
    from pcgcv1_b200 import runtime
    codec = runtime.get_codec(model, "")
    w = W.synthetic_weights(model)
    cubes, _ = synthetic.surface_cubes(1, seed=4)
    tr = training.FactorizedTrainer(codec, w, model=model, distortion=distortion)
    out = tr.forward_backward(cubes, seed=3)
    terms = tr.loss_terms(out)
    grads = {k: v.grad.detach().cpu().numpy().copy() for k, v in tr.params.items() if v.grad is not None}
    ref_terms, ref_grads, _ = forward_backward_factorized(w, cubes, model=model, seed=3, distortion=distortion)
    for k in _terms_keys(distortion):
        a, b = terms[k], ref_terms[k]
        print("%-12s gpu %.8g oracle %.8g rel %.2e" % (k, a, b, abs(a - b) / abs(b)))
        assert abs(a - b) <= 5e-5 * abs(b), k
    prefix = tr.prefix
    worst, n = ("", 0.0), 0
    for key, ref in ref_grads.items():
        if key.startswith(prefix):
            continue
        e = _rel(grads[key], ref)
        worst = max(worst, (key, e), key=lambda t: t[1])
        n += 1
        assert e < 2e-3, (key, e)
    assert n == sum(2 if l.bias else 1 for net in ("analysis_transform", "synthesis_transform") for l in netspec.NETS[(model, net)])
    for name in ("matrix", "bais", "factor"):
        ref = np.concatenate([ref_grads["%s%s_%d" % (prefix, name, i)].reshape(-1) for i in range(4)])
        assert _rel(grads[prefix + name], ref) < 2e-3, name
    print("%s/%s: worst relative gradient error %.2e (%s)" % (model, distortion, worst[1], worst[0]))
    # the same seed gives the same bits
    tr.forward_backward(cubes, seed=3)
    for k, v in tr.params.items():
        assert np.array_equal(v.grad.detach().cpu().numpy(), grads[k]), k
    # the first Adam step
    p0 = {k: v.detach().cpu().numpy().astype(np.float64) for k, v in tr.params.items()}
    tr.adam_step()
    codec.synchronize()
    for key in ("synthesis_transform/%s/kernel" % netspec.NETS[(model, "synthesis_transform")][-1].name, prefix + "matrix"):
        ref = otrain.adam_update(p0[key], grads[key].astype(np.float64), 0.0, 0.0, 1, lr=tr.lr)[0]
        got = tr.params[key].detach().cpu().numpy()
        assert np.abs(got - ref).max() <= 1e-6 * np.abs(ref).max() + 1e-9, key
        assert np.abs(got - p0[key]).max() > 0


def test_trainer_refuses_a_mismatched_codec_or_model(codec):
    with pytest.raises(ValueError):
        training.FactorizedTrainer(codec, model="simple")
    with pytest.raises(ValueError):
        training.FactorizedTrainer(codec, model="hyper")
    with pytest.raises(ValueError):
        training.FactorizedTrainer(codec, model="voxception", distortion="dice")


# ------------------------------------------------------------------------------------------ checkpoint in the codec
@pytest.mark.parametrize("model", ["simple", "voxception"])
def test_trained_checkpoint_round_trips_in_the_codec(model, tmp_path):
    from pcgcv1_b200 import runtime, transform
    from pcgcv1_b200.models import model_simple, model_voxception
    mod = model_simple if model == "simple" else model_voxception
    cubes, _ = synthetic.surface_cubes(2, seed=8)
    tr = training.FactorizedTrainer(runtime.get_codec(model, ""), model=model, lr=1e-4)
    for s in range(2):
        tr.train_step(cubes, seed=s)
    exported = tr.export_weights()
    prefix = tr.prefix
    assert not any(k.startswith(("hyper_encoder/", "hyper_decoder/")) for k in exported)
    assert sorted(k for k in exported if "/" in k and k.split("/")[0] + "/" == prefix) == \
        sorted("%s%s_%d" % (prefix, n, i) for n in ("matrix", "bais", "factor") for i in range(4))
    ckpt = str(tmp_path / ("ckpt_" + model))
    W.save(ckpt, exported)
    strings, min_v, max_v, shape = transform.compress_factorized(cubes, mod, ckpt)
    xs = transform.decompress_factorized(strings.numpy(), min_v.numpy(), max_v.numpy(), shape.numpy(), mod, ckpt).numpy()
    codec = runtime.get_codec(mod, ckpt)
    y = codec.analysis(codec.to_device(cubes))
    y_hat = codec.factorized(codec.bottleneck_slot(y.shape[-1]), y, want_p=False, want_bits=False)[0]
    assert np.array_equal(xs, codec.synthesis(y_hat).cpu().numpy())
    # the trained weights are the ones in use
    for k, v in exported.items():
        assert np.array_equal(codec.weights[k], v), k


def test_cli_compress_decompress_with_a_trained_checkpoint(tmp_path):
    from pcgcv1_b200 import runtime
    from pcgcv1_b200.dataprocess import inout_points
    cubes, _ = synthetic.surface_cubes(2, seed=9)
    tr = training.FactorizedTrainer(runtime.get_codec("simple", ""), model="simple", lr=1e-4)
    tr.train_step(cubes, seed=0)
    ckpt = str(tmp_path / "ckpt")
    W.save(ckpt, tr.export_weights())
    pts = np.concatenate([np.argwhere(cubes[i, ..., 0] > 0) + [64 * i, 0, 0] for i in range(2)]).astype(np.int32)
    inout_points.write_ply_data(str(tmp_path / "cloud.ply"), pts)
    env = dict(os.environ, PYTHONPATH=ROOT)
    common = ["--mode", "factorized", "--modelname", "models.model_simple", "--ckpt_dir", ckpt]
    for argv in (["compress", "cloud.ply"], ["decompress", "compressed/cloud"]):
        r = subprocess.run([sys.executable, "-m", "pcgcv1_b200.test"] + argv + common, cwd=str(tmp_path), env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    rec = inout_points.load_ply_data(str(tmp_path / "cloud_rec.ply"))
    assert len(rec) == len(pts)                                     # rho = 1: as many points out as in


# ------------------------------------------------------------------------------------------------------ the loop
def _write_cubes(tmp_path, n, seed=0):
    cubes, _ = synthetic.surface_cubes(n, seed=seed)
    files = []
    for i in range(n):
        f = os.path.join(str(tmp_path), "cube_%03d.npy" % i)
        np.save(f, np.array(np.where(cubes[i, ..., 0] > 0)).T.astype(np.int16))
        files.append(f)
    return files


@pytest.mark.parametrize("model", ["simple", "voxception"])
def test_loop_resumes_bit_for_bit_seeds_from_init_and_logs(model, tmp_path):
    files = _write_cubes(tmp_path, 27, seed=12)
    kw = dict(model=model, alpha=0.75, beta=3.0, lr=1e-4, batch_size=2, display_step=2, eval_cubes=2, log=lambda *a: None)
    a_dir = os.path.join(str(tmp_path), "run_a")
    wa = TF.train(files, a_dir, num_iteration=4, save_step=2, reset_optimizer=1, **kw).export_weights()
    assert int(TH.load_train_state(a_dir)["global_step"]) == 4
    log = [json.loads(l) for l in open(os.path.join(a_dir, "log.jsonl"))]
    assert [r["event"] for r in log] == ["train", "eval", "train", "eval"]
    assert set(log[0]) == {"event", "iteration", "bpp_ae", "IoU", "loss", "minutes"}
    assert set(log[1]) == {"event", "iteration", "bpp_ae", "IoU"}
    assert all(np.isfinite(r["bpp_ae"]) and r["bpp_ae"] > 0 and 0.0 <= r["IoU"] <= 1.0 for r in log)
    b_dir = os.path.join(str(tmp_path), "run_b")
    TF.train(files, b_dir, num_iteration=2, save_step=2, reset_optimizer=1, **kw)
    wb = TF.train(files, b_dir, num_iteration=4, save_step=2, reset_optimizer=1, **kw).export_weights()
    assert sorted(wa) == sorted(wb)
    for k in wa:
        assert np.array_equal(wa[k], wb[k]), k
    c_dir = os.path.join(str(tmp_path), "run_c")
    wc = TF.train(files, c_dir, num_iteration=0, init_ckpt_dir=a_dir, save_step=2, **kw).export_weights()
    for k in wa:
        assert np.array_equal(wa[k], wc[k]), k


def test_loop_runs_on_dataset_files_and_training_lowers_the_loss(tmp_path):
    from oracle import meshsample as om
    from pcgcv1_b200 import dataset as ds, runtime
    src = tmp_path / "meshes"
    src.mkdir()
    v, f = om.icosphere(3)
    with open(str(src / "ball.obj"), "w") as fh:
        fh.write("".join("v %r %r %r\n" % tuple(p) for p in v.tolist()))
        fh.write("".join("f %d %d %d\n" % tuple(t) for t in (f + 1).tolist()))
    out = tmp_path / "cubes"
    assert ds.main([str(src / "*.obj"), str(out), "--points", "300000", "--resolution", "160", "--min_num", "32", "--seed", "4"]) == 0
    files = sorted(str(out / p) for p in os.listdir(out) if p.endswith(".npy"))
    assert len(files) >= 2
    ckpt = str(tmp_path / "ckpt")
    TF.train(files, ckpt, model="simple", num_iteration=2, batch_size=2, display_step=1, save_step=10 ** 6, log=lambda *a: None)
    recs = [json.loads(x) for x in open(os.path.join(ckpt, "log.jsonl"))]
    assert [r["event"] for r in recs] == ["train", "train"] and all(math.isfinite(r["loss"]) for r in recs)
    # a run shorter than the save interval still ends with a checkpoint the codec loads
    assert int(TH.load_train_state(ckpt)["global_step"]) == 2
    assert runtime.Codec("simple", ckpt).bottleneck_slot(32) == 0
    # 30 seeded steps on one fixed batch lower the loss of that batch
    cubes = TF.CubeFiles.voxels(files[:2])
    tr = training.FactorizedTrainer(runtime.get_codec("simple", ""), model="simple", lr=1e-3)
    before = tr.loss_terms(tr.forward_backward(cubes, seed=0))["loss"]
    for s in range(30):
        tr.train_step(cubes, seed=s)
    after = tr.loss_terms(tr.forward_backward(cubes, seed=0))["loss"]
    print("loss %.6f -> %.6f" % (before, after))
    assert after < before
