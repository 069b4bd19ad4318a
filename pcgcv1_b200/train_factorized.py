"""The training loop of the factorized-prior models (the reference's second training script, ``train_factorized.py``) around
the GPU step of ``training.FactorizedTrainer``: analysis -> EntropyBottleneck(y, training=True) -> synthesis.

* ``--modelname models.model_simple`` (the default) trains ``model_simple`` with its 32-channel bottleneck (``estimator/*``);
  ``models.model_voxception`` trains the Voxception transforms with the 16-channel bottleneck the codec's factorized path loads
  (``estimator_y/*``) and no hyper nets.
* The loss is ``alpha * (beta * empty + full) + delta * bpp_y`` (``--distortion focal``: ``alpha * focal + delta * bpp_y``).  The
  reference script is not available; this is the hyperprior loss of ``train_hyper`` with its hyperprior terms removed, this
  project's definition rather than a parity claim.
* ``--lower_bound`` is the likelihood bound of the bottleneck (the factorized model has no scale to floor).
* Data, sampling, resume / ``--init_ckpt_dir``, ``--reset_optimizer``, torchrun with one NCCL all-reduce per step, checkpoints
  (``weights.npz`` + ``train_state.npz``) and ``log.jsonl`` are those of ``train_hyper`` (``train_hyper.run_loop``).  A run whose
  ``--num_iteration`` is not a multiple of the save interval (5000 steps) also writes a checkpoint of its last step, so that a
  short run leaves a directory the codec can load.
* Evaluation runs the inference kernels: analysis (``umma_win`` for ``model_simple``), ``Codec.factorized`` on the bottleneck
  slot of y's channels (bits), synthesis and ``select_voxels``; it logs ``bpp_ae`` and ``IoU``.
* The default checkpoint directory is ``<checkpoint_dir>/<prefix>factorized_<model>|a{alpha:.2f}b{beta:.2f}`` (this project's
  naming, after ``train_hyper``'s ``<prefix>hyper|a..b..``).  The written directory is a codec ``ckpt_dir``:
  ``python -m pcgcv1_b200.test compress cloud.ply --mode factorized --modelname models.model_simple --ckpt_dir <it>``.

``python -m pcgcv1_b200.train_factorized --data 'points64/*.npy' --modelname models.model_simple --num_iteration 300000``
"""
from __future__ import annotations

import argparse
import glob
import os
from typing import Dict, Optional, Sequence

import numpy as np

from .train_hyper import DISPLAY_STEP, SAVE_STEP, CubeFiles, add_loop_arguments, init_distributed, iou, run_loop, save_checkpoint


def evaluate(weights, files: Sequence[str], model: str = "simple", batch_size: int = 8, device: Optional[int] = None) -> Dict[str, float]:
    """Forward with "symbols" quantisation through the inference kernels: bpp of y from the bottleneck's likelihoods, IoU of the
    top-k reconstruction with each cube's true point count; the mean over batches of ``batch_size`` cubes, the last one possibly
    smaller, so that every given cube is scored.  No files: ``{}``."""
    import torch
    from . import runtime
    from .dataprocess import inout_points
    if not files:
        return {}
    codec = runtime.Codec(model, "", device, weights=weights)
    slot = codec.bottleneck_slot(codec.latent_c)
    acc = {"bpp_ae": 0.0, "IoU": 0.0}
    starts = range(0, len(files), batch_size)
    n_batches = len(starts)
    for i in starts:
        vox = CubeFiles.voxels(files[i:i + batch_size])
        y = codec.analysis(codec.to_device(vox))
        y_hat, _, bits, _ = codec.factorized(slot, y, want_p=False, want_bits=True)
        logits = codec.synthesis(y_hat)
        B = y.shape[0]
        nums = vox.reshape(B, -1).sum(1).astype(np.int32)
        mask = inout_points.select_voxels(runtime.DeviceResult(logits), nums, 1.0, codec=codec, dtype="uint8")
        acc["bpp_ae"] += float(bits.sum().item()) / float(max(int(nums.sum()), 1))
        acc["IoU"] += iou(mask, vox)
    del codec
    torch.cuda.empty_cache()
    return {k: v / n_batches for k, v in acc.items()}


def train(files: Sequence[str], ckpt_dir: str, model: str = "simple", alpha=2.0, beta=3.0, delta=1.0, lr=1e-5, num_iteration=int(3e5),
          batch_size=8, init_ckpt_dir: str = "", reset_optimizer: int = 0, lower_bound: float = 1e-9, display_step: int = DISPLAY_STEP,
          save_step: int = SAVE_STEP, eval_cubes: int = 256, log=print, distortion: str = "bce"):
    """Train ``model`` ("simple" | "voxception") with the factorized prior.  Returns the trainer (rank-local)."""
    from . import training

    def make_trainer(codec, w0):
        return training.FactorizedTrainer(codec, weights=w0, model=model, alpha=alpha, beta=beta, delta=delta, lr=lr, likelihood_bound=lower_bound,
                                          distortion=distortion)
    tr = run_loop(files, ckpt_dir, model, make_trainer, lambda w, f, device: evaluate(w, f, model, batch_size=8, device=device), ("bpp_ae",),
                  num_iteration, batch_size, init_ckpt_dir, reset_optimizer, display_step, save_step, eval_cubes, log)
    # a run whose length is not a multiple of save_step ends with a checkpoint of its last step, so that it leaves a ckpt_dir
    import torch.distributed as dist
    if int(num_iteration) > 0 and int(num_iteration) % save_step and (not dist.is_initialized() or dist.get_rank() == 0):
        save_checkpoint(ckpt_dir, tr, int(num_iteration), bool(reset_optimizer))
    return tr


def checkpoint_dir(checkpoint_root: str, prefix: str, model: str, alpha: float, beta: float) -> str:
    """``<checkpoint_root>/<prefix>factorized_<model>|a{alpha:.2f}b{beta:.2f}``."""
    return os.path.join(checkpoint_root, prefix + "factorized_{0}|a{1:.2f}b{2:.2f}".format(model, alpha, beta))


def parse_args(argv=None) -> argparse.Namespace:
    p = argparse.ArgumentParser(prog="pcgcv1_b200.train_factorized", formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    add_loop_arguments(p)
    p.add_argument("--modelname", type=str, default="models.model_simple", choices=["models.model_simple", "models.model_voxception"],
                   help="transforms to train")
    p.add_argument("--lower_bound", type=float, default=1e-9, help="likelihood bound of the EntropyBottleneck")
    return p.parse_args(argv)


def main(argv=None):
    from . import runtime
    a = parse_args(argv)
    model = runtime.model_name(a.modelname)
    init_distributed()
    files = sorted(glob.glob(a.data))
    train(files, checkpoint_dir(a.checkpoint_dir, a.prefix, model, a.alpha, a.beta), model, a.alpha, a.beta, a.delta, a.lr, a.num_iteration,
          a.batch_size, a.init_ckpt_dir, a.reset_optimizer, a.lower_bound, distortion=a.distortion)


if __name__ == "__main__":
    main()
