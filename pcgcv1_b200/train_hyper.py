"""The training LOOP of the hyperprior model (SURVEY.md 8f rank 4; the reference's ``train_hyper.py:100-268``) around the
GPU training step of ``pcgcv1_b200/training.py`` (``train_hyper.py:184-214``, row a22).

What the reference's loop does, and where it is here:

* data (``:121-122,171-177``): a directory of per-cube point files (``h5py.File(f)['data']``: integer [n,3] points of one 64^3
  cube), ``random.sample(train_list, BATCH_SIZE)`` per step with ``random.seed(3)`` (``:17``), the first ``1/RATIO_EVAL`` of the
  file list held out for evaluation -> ``CubeFiles`` (h5 when h5py is importable, .npy / .npz otherwise; same sampling).
  ``python -m pcgcv1_b200.dataset`` writes such files from meshes (OBJ / OFF / PLY; the reference's ``generate_dataset.py`` and
  ``dataprocess/mesh2pc.py``).
* the step (``:179-214``) -> ``HyperTrainer.train_step`` (seeded Philox noise: step number = seed).
* running means of bpp / IoU every DISPLAY_STEP (``:216-248``): ``select_voxels`` of the reconstruction with the TRUE point count
  of every cube, then ``get_classify_metrics`` (``loss.py:60-78``) -> ``iou`` below.
* every SAVE_STEP (``:254-266``): evaluation with "symbols" quantisation on 256 held-out cubes in batches of 8 (``eval``,
  ``:123-163``) and a checkpoint -> ``evaluate`` / ``save_checkpoint``.  A checkpoint directory holds ``weights.npz`` (the file
  the codec's ``ckpt_dir`` argument loads: the trained model compresses right away) and ``train_state.npz`` (global step, Adam
  moments).  A checkpoint found in the run's own directory is resumed with its global step; otherwise ``init_ckpt_dir`` seeds the
  variables and the step restarts at 0 (``:272-282``).  ``reset_optimizer`` follows the reference's (inverted-looking) rule at ``:100-114``: 0 -> the optimizer state is
  neither saved nor restored, otherwise it is.
* N > 1 (the reference is single-GPU): one process per GPU under torchrun, every rank samples its own batch, gradients are
  averaged by ONE NCCL all-reduce per step (``HyperTrainer.allreduce_gradients``); rank 0 evaluates and writes checkpoints.

TensorBoard summaries (``tf.contrib.summary``) become one JSON line per display / evaluation event in ``<ckpt>/log.jsonl``.
The rho search of ``eval_ablation_studies.py:152-205`` needs the external ``pc_error`` binary and is not built.

``python -m pcgcv1_b200.train_hyper --data 'points64/*.h5' --alpha 0.75 --beta 3 --num_iteration 300000``

The factorized-prior models (``model_simple`` and the Voxception transforms without the hyperprior) train with the same loop
(``run_loop``): ``python -m pcgcv1_b200.train_factorized`` (pcgcv1_b200/train_factorized.py).
"""
from __future__ import annotations

import argparse
import glob
import json
import math
import os
import random
import time
from typing import Dict, List, Optional, Sequence

import numpy as np

RATIO_EVAL = 9          # train_hyper.py:85
DISPLAY_STEP = 100      # :83
SAVE_STEP = 5000        # :84


# --------------------------------------------------------------------------------------------- data
def load_cube_points(path: str) -> np.ndarray:
    """One training sample: integer points [n,3] inside a 64^3 cube (``h5py.File(f, 'r')['data'][:].astype('int')``, :175)."""
    if path.endswith((".h5", ".hdf5")):
        try:
            import h5py
        except ImportError as e:                                     # pragma: no cover - h5py is absent in this image
            raise RuntimeError("reading %s needs h5py; convert the dataset to .npy (one [n,3] array per cube)" % path) from e
        with h5py.File(path, "r") as f:
            return f["data"][:].astype("int")
    if path.endswith(".npz"):
        with np.load(path) as z:
            return z["data"].astype("int")
    return np.load(path).astype("int")


class CubeFiles:
    """The reference's file list with its evaluation split (:121,167,257) and its sampling (``random.sample``, seeded)."""

    def __init__(self, files: Sequence[str], ratio_eval: int = RATIO_EVAL, seed: int = 3, rank: int = 0):
        self.files = list(files)
        if not self.files:
            raise ValueError("no training files")
        n_eval = len(self.files) // ratio_eval
        self.eval_list = self.files[:n_eval]
        self.train_list = self.files[n_eval:]
        self.rng = random.Random(seed + 7919 * rank)                 # rank 0 draws the reference's sequence
        self.eval_rng = random.Random(seed + 1)                      # own stream: a resumed run replays the training draws only

    def sample_train(self, batch_size: int) -> List[str]:
        return self.rng.sample(self.train_list, batch_size)

    def sample_eval(self, n: int) -> List[str]:
        n = min(n, len(self.eval_list))
        return self.eval_rng.sample(self.eval_list, n) if n else []

    @staticmethod
    def voxels(paths: Sequence[str], cube_size: int = 64) -> np.ndarray:
        """-> uint8 occupancy [B,S,S,S,1] (``points2voxels``, inout_points.py:116-132)."""
        from .dataprocess import inout_points
        return inout_points.points2voxels([load_cube_points(p) for p in paths], cube_size)


# ------------------------------------------------------------------------------------------ metrics
def iou(mask: np.ndarray, label: np.ndarray) -> float:
    """``get_classify_metrics(pred, label)[2]`` (loss.py:36-78, th = 0): TP / (TP + FP + FN) over the whole batch."""
    p = np.asarray(mask).reshape(-1) > 0
    t = np.asarray(label).reshape(-1) > 0
    tp = np.count_nonzero(p & t)
    fp = np.count_nonzero(p & ~t)
    fn = np.count_nonzero(~p & t)
    return float(tp) / float(max(tp + fp + fn, 1))


# -------------------------------------------------------------------------------------- checkpoints
def save_checkpoint(ckpt_dir: str, trainer, global_step: int, with_optimizer: bool) -> str:
    """weights.npz (loadable as the codec's ``ckpt_dir``) + train_state.npz; written to temporary names and renamed, so an
    interrupted save leaves the previous checkpoint intact."""
    from . import weights as W
    os.makedirs(ckpt_dir, exist_ok=True)
    tmp = os.path.join(ckpt_dir, ".tmp_save")
    os.makedirs(tmp, exist_ok=True)
    W.save(tmp, trainer.export_weights())
    os.replace(os.path.join(tmp, "weights.npz"), os.path.join(ckpt_dir, "weights.npz"))
    state: Dict[str, np.ndarray] = {"global_step": np.int64(global_step), "adam_t": np.int64(trainer.step_count if with_optimizer else 0),
                                    "with_optimizer": np.int64(int(with_optimizer))}
    if with_optimizer:
        for k, v in trainer.adam_m.items():
            state["m/" + k] = v.detach().cpu().numpy()
        for k, v in trainer.adam_v.items():
            state["v/" + k] = v.detach().cpu().numpy()
    path = os.path.join(ckpt_dir, "train_state.npz")
    np.savez(os.path.join(tmp, "train_state.npz"), **state)
    os.replace(os.path.join(tmp, "train_state.npz"), path)
    os.rmdir(tmp)
    return path


def load_train_state(ckpt_dir: str) -> Optional[Dict[str, np.ndarray]]:
    path = os.path.join(ckpt_dir, "train_state.npz")
    if not os.path.exists(path):
        return None
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def restore(trainer, state: Optional[Dict[str, np.ndarray]], with_optimizer: bool) -> int:
    """Adam moments / step counter into ``trainer`` (when both the checkpoint and the caller keep them) -> global step."""
    import torch
    if state is None:
        return 0
    if with_optimizer and int(state.get("with_optimizer", 0)):
        trainer.step_count = int(state["adam_t"])
        for k in trainer.adam_m:
            trainer.adam_m[k].copy_(torch.from_numpy(state["m/" + k]))
            trainer.adam_v[k].copy_(torch.from_numpy(state["v/" + k]))
    return int(state["global_step"])


# ------------------------------------------------------------------------------------- evaluation
def evaluate(weights, files: Sequence[str], batch_size: int = 8, device: Optional[int] = None) -> Dict[str, float]:
    """``eval(data, batch_size)`` (train_hyper.py:123-163): forward with "symbols" quantisation through the INFERENCE kernels
    (tcgen05 transforms, fused entropy models), bpp of y and z from the likelihoods, IoU of the top-k reconstruction."""
    import torch
    from . import runtime
    from .dataprocess import inout_points
    codec = runtime.Codec("voxception", "", device, weights=weights)
    acc = {"bpp_ae": 0.0, "bpp_hyper": 0.0, "IoU": 0.0}
    n_batches = len(files) // batch_size
    for i in range(n_batches):
        vox = CubeFiles.voxels(files[i * batch_size:(i + 1) * batch_size])
        x = codec.to_device(vox)
        y = codec.analysis(x)
        z = codec.hyper_encode(y)
        z_hat, _, bits_z, _ = codec.factorized(codec.bottleneck_slot(8), z, want_p=False, want_bits=True)
        loc, scale = codec.hyper_decode(z_hat, 1e-9)
        B = y.shape[0]
        y_hat, _, bits_y, _ = codec.laplace(y.reshape(B, -1), loc.reshape(B, -1), scale.reshape(B, -1), want_p=False, want_bits=True)
        logits = codec.synthesis(y_hat.reshape(y.shape))
        nums = vox.reshape(B, -1).sum(1).astype(np.int32)
        mask = inout_points.select_voxels(runtime.DeviceResult(logits), nums, 1.0, codec=codec, dtype="uint8")
        n_pts = float(max(int(nums.sum()), 1))
        acc["bpp_ae"] += float(bits_y.sum().item()) / n_pts
        acc["bpp_hyper"] += float(bits_z.sum().item()) / n_pts
        acc["IoU"] += iou(mask, vox)
    del codec
    torch.cuda.empty_cache()
    return {k: v / max(n_batches, 1) for k, v in acc.items()}


# ------------------------------------------------------------------------------------------- loop
def run_loop(files: Sequence[str], ckpt_dir: str, model: str, make_trainer, evaluate_fn, rate_keys: Sequence[str], num_iteration: int,
             batch_size: int, init_ckpt_dir: str, reset_optimizer: int, display_step: int, save_step: int, eval_cubes: int, log):
    """The loop both training commands share (train_hyper.py:165-266): resume / seeding, seeded sampling, one ``train_step`` per
    step (seed = step * world + rank), running bpp / IoU every ``display_step``, evaluation and checkpoint every ``save_step``,
    ``log.jsonl``.  ``make_trainer(codec, weights)`` builds the rank-local trainer, ``evaluate_fn(weights, files, device)`` scores
    held-out cubes, ``rate_keys`` are the bpp terms it reports.  Returns the trainer."""
    import torch
    import torch.distributed as dist
    from . import runtime, weights as W
    from .dataprocess import inout_points

    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    device = torch.cuda.current_device()
    with_opt = bool(reset_optimizer)                                  # the reference's rule, see the module docstring
    # :272-282: a checkpoint in the run's own directory is resumed (global step kept); otherwise init_ckpt_dir seeds the
    # variables and the global step restarts at 0
    resume = os.path.exists(os.path.join(ckpt_dir, "weights.npz")) and load_train_state(ckpt_dir) is not None
    src = ckpt_dir if resume else init_ckpt_dir
    w0 = W.load(src, model) if src else None
    codec = runtime.get_codec(model, "", device)
    tr = make_trainer(codec, w0)
    step0 = restore(tr, load_train_state(src) if src else None, with_opt)
    if not resume:
        step0 = 0
    data = CubeFiles(files, rank=rank)
    for _ in range(step0):                                            # a resumed run continues the sampling sequence
        data.sample_train(batch_size)
    sums = {k: 0.0 for k in tuple(rate_keys) + ("IoU",)}
    num = 0
    start = time.time()
    logf = None
    if rank == 0:
        os.makedirs(ckpt_dir, exist_ok=True)
        logf = open(os.path.join(ckpt_dir, "log.jsonl"), "a")

    def emit(rec):
        if logf is not None:
            logf.write(json.dumps(rec) + "\n")
            logf.flush()

    def bpps(d):
        return " + ".join("%.4f" % d[k] for k in rate_keys)

    for step in range(step0, int(num_iteration)):
        vox = CubeFiles.voxels(data.sample_train(batch_size))
        out = tr.train_step(vox, seed=step * world + rank, group=None)
        terms = tr.loss_terms(out)
        if not all(math.isfinite(v) for v in terms.values()):
            raise FloatingPointError("non-finite loss at step %d: %s" % (step, terms))
        nums = vox.reshape(len(vox), -1).sum(1).astype(np.int32)
        mask = inout_points.select_voxels(runtime.DeviceResult(out["x_tilde"]), nums, 1.0, codec=codec, dtype="uint8")
        for k in rate_keys:
            sums[k] += terms[k]
        sums["IoU"] += iou(mask, vox)
        num += 1
        if (step + 1) % display_step == 0:
            rec = {"event": "train", "iteration": step}
            rec.update({k: sums[k] / num for k in rate_keys})
            rec.update({"IoU": sums["IoU"] / num, "loss": terms["loss"], "minutes": round((time.time() - start) / 60.0, 2)})
            if rank == 0:
                log("Iteration:%d\nBpps: %s\nIoU: %.4f\nRunning time:(mins): %s\n" % (step, bpps(rec), rec["IoU"], rec["minutes"]))
                emit(rec)
            sums = {k: 0.0 for k in sums}
            num = 0
        if (step + 1) % save_step == 0:
            if rank == 0:
                log("evaluating...")
                ev = evaluate_fn(tr.export_weights(), data.sample_eval(eval_cubes), device) if data.eval_list else {}
                if ev:
                    log("Bpps: %s\nIoU: %.4f" % (bpps(ev), ev["IoU"]))
                    emit(dict(ev, event="eval", iteration=step))
                save_checkpoint(ckpt_dir, tr, step + 1, with_opt)
            if world > 1:
                dist.barrier()
    if logf is not None:
        logf.close()
    return tr


def train(files: Sequence[str], ckpt_dir: str, alpha=2.0, beta=3.0, gamma=1.0, delta=1.0, lr=1e-5, num_iteration=int(3e5), batch_size=8,
          init_ckpt_dir: str = "", reset_optimizer: int = 0, lower_bound: float = 1e-9, display_step: int = DISPLAY_STEP,
          save_step: int = SAVE_STEP, eval_cubes: int = 256, log=print, distortion: str = "bce"):
    """``train()`` of train_hyper.py:165-266.  Returns the trainer (rank-local)."""
    from . import training

    def make_trainer(codec, w0):
        return training.HyperTrainer(codec, weights=w0, alpha=alpha, beta=beta, gamma=gamma, delta=delta, lr=lr, lower_bound=lower_bound,
                                     distortion=distortion)
    return run_loop(files, ckpt_dir, "voxception", make_trainer, lambda w, f, device: evaluate(w, f, batch_size=8, device=device),
                    ("bpp_ae", "bpp_hyper"), num_iteration, batch_size, init_ckpt_dir, reset_optimizer, display_step, save_step, eval_cubes, log)


def add_loop_arguments(p: argparse.ArgumentParser):
    """The command-line options both training commands share."""
    p.add_argument("--data", required=True, help="glob of per-cube point files (.h5 / .npy / .npz with key 'data')")
    p.add_argument("--alpha", type=float, default=2.0, help="weight of the distortion term (BCE) in the loss")
    p.add_argument("--beta", type=float, default=3.0, help="weight of the empty-voxel part of the BCE against the occupied part")
    p.add_argument("--delta", type=float, default=1.0, help="weight of the latent rate (bpp of y)")
    p.add_argument("--lr", type=float, default=1e-5)
    p.add_argument("--num_iteration", type=int, default=int(3e5))
    p.add_argument("--batch_size", type=int, default=8)
    p.add_argument("--prefix", type=str, default="")
    p.add_argument("--init_ckpt_dir", type=str, default="")
    p.add_argument("--reset_optimizer", type=int, default=0)
    p.add_argument("--checkpoint_dir", type=str, default="./checkpoints")
    p.add_argument("--distortion", type=str, default="bce", choices=["bce", "focal"],
                   help="occupancy loss: bce = get_bce_loss as the reference script calls it; focal = get_focal_loss (loss.py:83-93)")


def init_distributed():
    """One process per GPU under torchrun (WORLD_SIZE > 1): bind the local GPU and join the NCCL group."""
    import torch
    import torch.distributed as dist
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")


def main(argv=None):
    p = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    add_loop_arguments(p)
    p.add_argument("--gamma", type=float, default=1.0, help="weight of the hyper-latent rate (bpp of z)")
    p.add_argument("--lower_bound", type=float, default=1e-9)
    a = p.parse_args(argv)
    init_distributed()
    files = sorted(glob.glob(a.data))
    ckpt = os.path.join(a.checkpoint_dir, a.prefix + "hyper|a{0:.2f}b{1:.2f}".format(a.alpha, a.beta))          # train_hyper.py:269-271
    train(files, ckpt, a.alpha, a.beta, a.gamma, a.delta, a.lr, a.num_iteration, a.batch_size, a.init_ckpt_dir, a.reset_optimizer, a.lower_bound,
          distortion=a.distortion)


if __name__ == "__main__":
    main()
