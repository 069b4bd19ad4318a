"""The factorized training step's oracle (tests/oracle_train_factorized.py) against central finite differences of its own
loss, and the command line of pcgcv1_b200/train_factorized.py (CPU only)."""
import os

import numpy as np
import pytest
import torch

from oracle_train_factorized import forward_backward_factorized
from pcgcv1_b200 import synthetic, train_factorized as TF, weights as W


@pytest.mark.parametrize("model,distortion,key", [
    ("simple", "bce", "synthesis_transform/deconv_3/bias"),
    ("simple", "focal", "synthesis_transform/deconv_3/kernel"),
    ("simple", "bce", "estimator/bais_3"),
    ("voxception", "bce", "estimator_y/bais_0"),
])
def test_factorized_oracle_gradient_matches_finite_differences(model, distortion, key):
    w = W.synthetic_weights(model)
    cubes, _ = synthetic.surface_cubes(1, seed=4)
    kw = dict(model=model, seed=3, entropy_dtype=torch.float64, distortion=distortion)     # smooth loss for the finite differences
    terms, grads, _ = forward_backward_factorized(w, cubes, **kw)
    assert np.isfinite(terms["loss"]) and terms["bpp_ae"] > 0
    assert abs(terms["loss"] - (0.75 * terms["distortion"] + terms["bpp_ae"])) <= 1e-12 * abs(terms["loss"])
    assert not any(k.startswith(("hyper_", "estimator/" if model == "voxception" else "estimator_y/")) for k in grads)
    eps = 1e-4                              # parameters past the last ReLU: the loss is smooth in them
    idx = (0,) * np.asarray(w[key]).ndim
    wp, wm = dict(w), dict(w)
    wp[key] = np.asarray(w[key], np.float64).copy()
    wm[key] = np.asarray(w[key], np.float64).copy()
    wp[key][idx] += eps
    wm[key][idx] -= eps
    fd = (forward_backward_factorized(wp, cubes, **kw)[0]["loss"] - forward_backward_factorized(wm, cubes, **kw)[0]["loss"]) / (2 * eps)
    assert abs(fd - grads[key][idx]) <= 1e-5 * max(1.0, abs(fd)), (fd, grads[key][idx])


def test_cli_arguments_and_checkpoint_naming():
    a = TF.parse_args(["--data", "p/*.npy"])
    assert (a.modelname, a.alpha, a.beta, a.delta, a.lr, a.num_iteration, a.batch_size) == ("models.model_simple", 2.0, 3.0, 1.0, 1e-5, 300000, 8)
    assert (a.prefix, a.init_ckpt_dir, a.reset_optimizer, a.lower_bound, a.checkpoint_dir, a.distortion) == ("", "", 0, 1e-9, "./checkpoints", "bce")
    a = TF.parse_args(["--data", "x", "--modelname", "models.model_voxception", "--alpha", "0.5", "--beta", "2", "--delta", "0.25", "--lr", "1e-4",
                       "--num_iteration", "7", "--batch_size", "4", "--prefix", "run1_", "--init_ckpt_dir", "init", "--reset_optimizer", "1",
                       "--lower_bound", "1e-6", "--checkpoint_dir", "ck", "--distortion", "focal"])
    assert (a.modelname, a.alpha, a.beta, a.delta, a.lr, a.num_iteration, a.batch_size) == ("models.model_voxception", 0.5, 2.0, 0.25, 1e-4, 7, 4)
    assert (a.prefix, a.init_ckpt_dir, a.reset_optimizer, a.lower_bound, a.checkpoint_dir, a.distortion) == ("run1_", "init", 1, 1e-6, "ck", "focal")
    assert TF.checkpoint_dir("ck", "run1_", "voxception", 0.5, 2.0) == os.path.join("ck", "run1_factorized_voxception|a0.50b2.00")
    assert TF.checkpoint_dir("./checkpoints", "", "simple", 2.0, 3.0) == os.path.join("./checkpoints", "factorized_simple|a2.00b3.00")
    for bad in (["--data", "x", "--modelname", "models.model_other"], ["--data", "x", "--distortion", "dice"], []):
        with pytest.raises(SystemExit):
            TF.parse_args(bad)
