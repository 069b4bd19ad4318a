"""Point normals for D2 (point-to-plane): k-nearest-neighbour PCA on the GPU, and the ``_n.ply`` file that D2 reads.

    python -m pcgcv1_b200.normals cloud.ply cloud_n.ply [--knn 30]

reads ``cloud.ply`` as the D1 / D2 figures read it (``pc_error_wrapper._load_xyz_normals``: file order, float64), estimates one
normal per point on the GPU (``Codec.estimate_normals``, contract in ``include/pcgc_b200.h`` ``pcgc_estimate_normals``) and writes
``cloud_n.ply`` with ``x y z nx ny nz``: the points exactly as read and the normals with 17 significant digits, so both the MPEG
``pc_error`` binary (``-n``) and the built-in figures (``pc_error``, ``DeviceRhoSearch``) read back the device's doubles.

The normal of a point is the smallest-eigenvalue eigenvector of the covariance of its k nearest points (itself included; the lowest
index wins among equidistant points), oriented so that its largest component is positive.  The default k = 30 is this project's
choice; it does not claim parity with any other normal estimator (Open3D, CloudCompare, MeshLab or the tools behind published
``_n.ply`` files), whose neighbourhoods, tie rules and orientations differ."""
from __future__ import annotations

import argparse

import numpy as np

DEFAULT_K = 30


def estimate_normals(xyz, k: int = DEFAULT_K, codec=None) -> np.ndarray:
    """Normals of the points ``xyz`` ([n,3] array or tensor, taken as float64) -> float64 [n,3] NumPy array."""
    import torch
    from . import runtime
    c = codec or runtime.get_codec("voxception", "")
    pts = c.to_device(xyz, torch.float64)
    if pts.dim() != 2 or pts.shape[1] != 3:
        raise ValueError("estimate_normals: points must be [n,3], got %s" % (tuple(pts.shape),))
    return c.estimate_normals(pts.contiguous(), k).cpu().numpy()


def write_ply_normals(path, xyz, normals) -> None:
    """ASCII .ply with ``property float x y z nx ny nz``.  Integer-valued coordinates are written as integers, others with the
    shortest text that reads back to the same double; normals with 17 significant digits (read back exactly)."""
    xyz = np.asarray(xyz, np.float64).reshape(-1, 3)
    normals = np.asarray(normals, np.float64).reshape(-1, 3)
    if len(xyz) != len(normals):
        raise ValueError("write_ply_normals: %d points but %d normals" % (len(xyz), len(normals)))
    if np.all(np.isfinite(xyz)) and np.array_equal(xyz, np.rint(xyz)) and (len(xyz) == 0 or np.abs(xyz).max() < 2.0 ** 53):
        coords = ["%d %d %d" % tuple(p) for p in xyz.astype(np.int64).tolist()]
    else:
        coords = ["%r %r %r" % tuple(p) for p in xyz.tolist()]
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
                "property float nx\nproperty float ny\nproperty float nz\nend_header\n" % len(xyz))
        f.write("".join("%s %.17g %.17g %.17g\n" % (p, n[0], n[1], n[2]) for p, n in zip(coords, normals.tolist())))


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="pcgcv1_b200.normals", formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                 description="Estimate point normals on the GPU and write CLOUD_N (x y z nx ny nz).")
    ap.add_argument("input", help="point cloud (.ply)")
    ap.add_argument("output", help=".ply written with the points of INPUT in the same order and their normals")
    ap.add_argument("--knn", type=int, default=DEFAULT_K, help="neighbours per point, the point itself included (1 .. 64)")
    args = ap.parse_args(argv)
    if not 1 <= args.knn <= 64:
        ap.error("--knn must be in 1 .. 64")
    return args


def make_normals_file(input_file, output_file, k: int = DEFAULT_K, codec=None) -> np.ndarray:
    """Reads ``input_file`` as the D1 / D2 figures do, estimates the normals and writes ``output_file``; returns the normals."""
    from .myutils.pc_error_wrapper import _load_xyz_normals
    xyz, _ = _load_xyz_normals(input_file)
    normals = estimate_normals(xyz, k, codec)
    write_ply_normals(output_file, xyz, normals)
    return normals


def main(argv=None):
    args = parse_args(argv)
    make_normals_file(args.input, args.output, args.knn)


if __name__ == "__main__":
    main()
