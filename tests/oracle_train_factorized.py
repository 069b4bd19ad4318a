"""Oracle of one factorized-prior training step (test infrastructure only), for tests/test_train_factorized.py and
tests/test_gpu_train_factorized.py: the graph of ``pcgcv1_b200.training.FactorizedTrainer`` restated with torch-CPU autograd in
float64 from the pieces of oracle/train.py (the bottleneck likelihood, the BCE and focal losses) and oracle/nets.py (the
transforms), the gradients coming from ``loss.backward()``.  Noise = the Philox stream of oracle/entropy.py."""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

from oracle import entropy, nets
from oracle.train import LN2, _net, bce_loss, bottleneck_likelihood, focal_loss


def forward_backward_factorized(weights: Dict[str, np.ndarray], cubes: np.ndarray, model: str = "simple", seed: int = 0, alpha=0.75, beta=3.0,
                                delta=1.0, likelihood_bound=1e-9, dtype=torch.float64, noise_dtype=np.float32, entropy_dtype=torch.float32,
                                distortion="bce", focal_gamma=2.0, focal_alpha=0.9):
    """The factorized-prior step of ``pcgcv1_b200.training.FactorizedTrainer``: analysis -> EntropyBottleneck(y, training=True)
    -> synthesis with ``loss = alpha * D + delta * bpp_y`` (D as in ``forward_backward``), the hyperprior step with its hyperprior
    terms removed.  ``model`` "simple" trains ``estimator/*`` (32 channels), "voxception" ``estimator_y/*`` (16 channels).  The
    noise on y is the Philox stream the hyperprior step draws for z (seed = ``seed``).  The bottleneck likelihood is evaluated in
    ``entropy_dtype`` (float32 like TF; see ``oracle.train.forward_backward``), the transforms and reductions in ``dtype``.
    -> (terms, grads keyed like the weight file, {"y", "x_tilde"})."""
    prefix = {"simple": "estimator/", "voxception": "estimator_y/"}[model]
    P = {k: torch.tensor(np.asarray(v), dtype=dtype, requires_grad=True) for k, v in weights.items()
         if k.split("/")[0] in ("analysis_transform", "synthesis_transform") or k.startswith(prefix)}
    x = torch.tensor(cubes.astype(np.float64), dtype=dtype)
    y = nets.NETS[(model, "analysis")](x, _net(P, "analysis_transform"))
    ny = entropy.philox_uniform(seed, y.numel()).astype(noise_dtype).reshape(y.shape)
    y_t = y + torch.tensor(ny, dtype=dtype)
    ed = entropy_dtype
    Pe = {"estimator/" + k[len(prefix):]: v.to(ed) for k, v in P.items() if k.startswith(prefix)}
    p_y = torch.clamp(bottleneck_likelihood(y_t.to(ed), Pe), min=likelihood_bound).to(dtype)
    x_t = nets.NETS[(model, "synthesis")](y_t, _net(P, "synthesis_transform"))
    num_points = float((x.sum(-1) > 0).sum())
    bpp_ae = torch.log(p_y).sum() / (-LN2 * num_points)
    if distortion == "focal":
        f_full, f_empty = focal_loss(torch.sigmoid(x_t), x, focal_gamma, focal_alpha)
        dist = f_full + f_empty
        parts = (("focal_full", f_full), ("focal_empty", f_empty))
    else:
        zeros, ones = bce_loss(x_t, x)
        dist = beta * zeros + 1.0 * ones
        parts = (("zeros", zeros), ("ones", ones))
    loss = alpha * dist + delta * bpp_ae
    loss.backward()
    terms = {k: float(v.detach()) for k, v in parts + (("distortion", dist), ("bpp_ae", bpp_ae), ("loss", loss))}
    grads = {k: (v.grad.numpy().copy() if v.grad is not None else np.zeros(v.shape)) for k, v in P.items()}
    return terms, grads, {"y": y.detach().numpy(), "x_tilde": x_t.detach().numpy()}
