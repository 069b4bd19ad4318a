"""The rho search of the reference's evaluation driver (SURVEY.md section 8(f) rank 4): ``select_optimal_rho`` and
``cfg_post_process`` of ``eval_ablation_studies.py:152-205`` with their argument lists.  The rest of that script (the RD sweep
over checkpoints, its .ini bookkeeping of scales and checkpoint paths, the CSV / plots) is driver code around external files and
is not rebuilt.

What runs per candidate rho: ``process.postprocess`` -- top-k classification ON the GPU over the decoded logits, which stay
resident on the device across the whole search when ``cubes_d`` is the handle ``decompress_hyper`` returned (the reference re-sorts
every cube on the host for each rho), ordered extraction, .ply -- then ``myutils.pc_error_wrapper.pc_error`` (the MPEG binary when
present, the built-in D1 / D2 figures otherwise).

``DeviceRhoSearch`` provides a ``post`` / ``metric`` pair for the same two functions that keeps the whole search on the GPU: the
input cloud and its normals are loaded once, every candidate's reconstruction stays on the device and is scored by
``geometry_metrics_device``; no file is written unless the caller asks for one (``write``).

The search loop keeps the reference's exact control flow, including its quirk: the first candidate's PSNR never enters
``MAX_PSNR`` (it is initialised to 0 at i == 0), so the second candidate is always accepted and the search stops at the first
candidate from the third on whose PSNR drops below the best of candidates 2..i."""
from __future__ import annotations

import os

import numpy as np

from .myutils.pc_error_wrapper import _load_xyz_normals, geometry_metrics_device, pc_error
from .process import postprocess

RHOS_D1 = [0.8, 0.9, 1.0, 1.02, 1.05, 1.10, 1.15, 1.2, 1.25, 1.30, 1.40, 1.50, 1.75, 2.0, 2.5, 3.0]           # :180
RHOS_D2 = [1.0, 0.98, 0.95, 0.92, 0.90, 0.88, 0.85, 0.82, 0.80, 0.75, 0.70, 0.65, 0.50, 0.40, 0.30]           # :192
ITEM_D1, ITEM_D2 = "mseF,PSNR (p2point)", "mseF,PSNR (p2plane)"


def _scalar(results, item):
    v = results[item]
    return float(v.iloc[0]) if hasattr(v, "iloc") else float(v)


def select_optimal_rho(item, rhos, input_file, output_file, input_file_n, cubes_d, points_numbers_d, cube_positions_d, scale, cube_size, res,
                       post=postprocess, metric=pc_error):
    """eval_ablation_studies.py:152-174.  ``post`` / ``metric`` default to this package's ``postprocess`` / ``pc_error``."""
    optimal_rho = None
    for i, rho in enumerate(rhos):
        print("===== select rho =====")
        post(output_file, cubes_d, points_numbers_d, cube_positions_d, scale, cube_size, rho)
        results = metric(input_file, output_file, input_file_n, res, show=False)
        PSNR = _scalar(results, item)
        print("===== results: ", i, rho, item, PSNR)
        if i == 0:
            MAX_PSNR = 0
            optimal_rho = rho
        else:
            MAX_PSNR = max(PSNR, MAX_PSNR)
        if PSNR < MAX_PSNR:
            break
        else:
            optimal_rho = rho
    return optimal_rho


def cfg_post_process(config, config_file, rate, input_file, output_file, input_file_n, cubes_d, points_numbers_d, cube_positions_d, scale,
                     cube_size, res, post=postprocess, metric=pc_error):
    """eval_ablation_studies.py:177-203: rho_d1 / rho_d2 of section ``rate`` from the .ini when present, else searched and written back."""
    found = {}
    for key, item, rhos in (("rho_d1", ITEM_D1, RHOS_D1), ("rho_d2", ITEM_D2, RHOS_D2)):
        if config.has_option(rate, key):
            found[key] = float(config.get(rate, key))
        else:
            found[key] = select_optimal_rho(item, rhos, input_file, output_file, input_file_n, cubes_d, points_numbers_d, cube_positions_d,
                                            scale, cube_size, res, post=post, metric=metric)
            config.set(rate, key, str(found[key]))
            with open(config_file, "w") as f:
                config.write(f)
    return found["rho_d1"], found["rho_d2"]


class DeviceRhoSearch:
    """A ``post`` / ``metric`` pair for ``select_optimal_rho`` / ``cfg_post_process`` with the search resident on the GPU.

    ``post`` does what ``process.postprocess`` does -- top-k of ``rho * points_numbers[i]`` voxels per cube over the decoded logits,
    ordered extraction, cube offsets in sorted cube order, the ``1/scale`` factor in float32 -- but keeps the points on the device
    and writes nothing; ``metric`` scores them against the input cloud loaded once by the constructor (the built-in D1 / D2 figures,
    ``geometry_metrics_device``).  The figures are those of the file-based path except for two things: at ``scale != 1`` the points
    are not rounded through the .ply text, and among equidistant neighbours the lowest index wins.  ``write(path)`` stores the
    current candidate's reconstruction as ``postprocess`` would have."""

    def __init__(self, input_file, input_file_n="", codec=None):
        import torch
        from . import runtime
        self.codec = codec or runtime.get_codec("voxception", "")
        a, _ = _load_xyz_normals(input_file)
        normals = None
        if input_file_n and os.path.isfile(input_file_n):
            an, normals = _load_xyz_normals(input_file_n)
            if normals is not None and (len(an) != len(a) or not np.array_equal(an, a)):
                raise ValueError("%s does not list the points of %s in the same order" % (input_file_n, input_file))
        self.input = self.codec.to_device(a, torch.float64)
        self.normals = None if normals is None else self.codec.to_device(normals, torch.float64)
        self.points = None            # current candidate: float64 [n,3] on the device
        self._int_points, self._scale = None, 1

    def post(self, output_file, cubes_d, points_numbers_d, cube_positions_d, scale, cube_size, rho):
        import torch
        from . import runtime
        from .dataprocess import inout_points as iop
        c = self.codec
        logits = c.to_device(cubes_d, torch.float32)
        counts = np.asarray(runtime.unwrap(points_numbers_d)).reshape(-1)
        ks = np.array([int(rho * np.array(counts[i])) for i in range(logits.shape[0])], np.int32)
        if (ks > logits[0].numel()).any():
            raise IndexError("select_voxels: k exceeds the number of voxels (get_adaptive_thres would raise IndexError)")
        mask, _, _ = c.topk(logits, c.to_device(ks))
        local, per_cube = c.extract_points_device(runtime.unwrap(mask))
        ordered = iop._ordered_positions(cube_positions_d)
        per_cube = per_cube[:len(ordered)].long()                     # zip() truncation of the reference's save_points
        m = int(per_cube.sum())
        base = c.to_device(ordered[:len(per_cube)].astype(np.int64) * cube_size)
        pts = local[:m].long() + torch.repeat_interleave(base, per_cube, dim=0, output_size=m)
        self._int_points, self._scale = pts, scale
        if scale == 1:
            self.points = pts.double()
        else:                                                          # postprocess: float32 points * float(1 / scale)
            factor = torch.tensor(np.float32(1 / scale), device=pts.device)
            self.points = (pts.float() * factor).double()

    def metric(self, input_file, output_file, input_file_n, res, show=False):
        out = geometry_metrics_device(self.input, self.points, self.normals, peak=float(res - 1), codec=self.codec)
        if show:
            for k, v in out.items():
                print("%s: %s" % (k, v))
        return out

    def write(self, path):
        """The current candidate's reconstruction as ``process.postprocess`` writes it."""
        from .dataprocess import inout_points as iop
        pts = self._int_points.cpu().numpy()
        if self._scale == 1:
            iop.write_ply_data(path, pts.astype("int"))
        else:
            iop.write_ply_data(path, pts.astype("float32") * float(1 / self._scale))
