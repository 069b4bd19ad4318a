"""Training data from meshes: sample each surface on the GPU, voxelise it and write the per-cube point files ``train_hyper`` reads.

    python -m pcgcv1_b200.dataset 'shapenet/**/*.obj' points64/ [--points 1000000] [--resolution 256] [--cube_size 64]
                                  [--min_num 64] [--seed 0] [--no-rotate]

This is the job of the reference's ``dataprocess/mesh2pc.py`` (surface samples, a random rotation, scaling into a grid, voxelisation,
duplicates dropped) and ``generate_dataset.py`` (64^3 cubes, one ``.h5`` per cube), in one pass per mesh:

* ``load_mesh`` reads OBJ, OFF or PLY (ascii / binary_little_endian) with the library's C++ reader (``pcgc_mesh_parse``); every polygon
  becomes a triangle fan.
* ``Codec.sample_mesh`` (``pcgc_mesh_sample``; the exact rule is in ``include/pcgc_b200.h``) draws ``--points`` samples uniformly
  over the surface, rotates them, scales the box of the rotated mesh onto ``[0, resolution - 1]`` along its longest axis, rounds to
  the grid and keeps the distinct grid points.
* ``inout_points.partition_points`` cuts the cloud into cubes with the reference's ``load_points`` rule (cube order, the ``min_num``
  filter and its single-point quirk); each kept cube becomes ``<out>/<stem>_<k:04d>.npy``, int16 [n,3] cube-local points, which
  ``train_hyper.load_cube_points`` / ``CubeFiles.voxels`` read.
* ``<out>/manifest.csv`` gets one row per input mesh; a mesh that cannot be read or sampled is recorded there with its error and the
  run goes on.  The exit status is 1 when any mesh failed.

Naming and seeds: the *stem* of an input is its path relative to the deepest directory common to all inputs, without the extension
and with ``/`` replaced by ``__`` (ShapeNet names every mesh ``model_normalized.obj``).  The mesh seed is
``(seed * 2^32 + crc32(stem)) mod 2^64``; it drives both the rotation (``random_rotation``) and the sample stream.  So a mesh's files
depend only on the mesh, its stem and the options, not on the other inputs or their order.

The defaults (10^6 points, a 256^3 grid, ``min_num`` 64) are this project's choice.  They do not claim parity with ``mesh2pc.py``,
whose sampling libraries (pyntcloud / open3d) are not used here; the sampling rule, the rotation and the grid scaling are this
project's own."""
from __future__ import annotations

import argparse
import csv
import ctypes as C
import glob
import os
import sys
import zlib
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import _lib

DEFAULT_POINTS = 1_000_000
DEFAULT_RESOLUTION = 256
DEFAULT_CUBE_SIZE = 64
DEFAULT_MIN_NUM = 64
MANIFEST_FIELDS = ["stem", "seed", "vertices", "triangles", "samples", "unique_points", "cubes", "error"]
_FORMATS = {".obj": _lib.MESH_OBJ, ".off": _lib.MESH_OFF, ".ply": _lib.MESH_PLY}


def load_mesh(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """OBJ / OFF / PLY file (format from the extension, case-insensitive) -> (verts float64 [V,3], tris int32 [F,3], 0-based)."""
    ext = os.path.splitext(path)[1].lower()
    if ext not in _FORMATS:
        raise ValueError("%s: unknown mesh format %r (.obj, .off or .ply)" % (path, ext))
    with open(path, "rb") as f:
        data = f.read()
    nv, nt = C.c_int64(), C.c_int64()
    vcap = tcap = max(data.count(b"\n"), len(data) // 12 if ext == ".ply" else 0) + 16     # a first guess; too small -> retried
    while True:
        verts = np.empty((vcap, 3), np.float64)
        tris = np.empty((tcap, 3), np.int32)
        rc = _lib.lib().pcgc_mesh_parse(data, len(data), _FORMATS[ext], verts.ctypes.data, vcap, tris.ctypes.data, tcap, C.byref(nv),
                                        C.byref(nt))
        if rc != _lib.ERR_OVERFLOW:
            break
        vcap, tcap = max(nv.value, 1), max(nt.value, 1)
    if rc == _lib.ERR_CORRUPT:
        raise ValueError("%s: malformed %s mesh" % (path, ext[1:].upper()))
    if rc == _lib.ERR_BAD_ARG and ext == ".ply":
        raise ValueError("%s: unsupported PLY format (ascii 1.0 and binary_little_endian 1.0 are read)" % path)
    _lib.check(rc)
    return verts[:nv.value].copy(), tris[:nt.value].copy()


def random_rotation(seed: int) -> np.ndarray:
    """A uniform random rotation: the normalised Gaussian quaternion drawn from ``np.random.default_rng(seed)`` -> float64 [3,3]."""
    w, x, y, z = np.random.default_rng(seed).standard_normal(4)
    n = np.sqrt(w * w + x * x + y * y + z * z)
    w, x, y, z = w / n, x / n, y / n, z / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]], np.float64)


def stems(paths: Sequence[str]) -> List[str]:
    """Each path relative to the deepest directory common to all, without its extension, ``/`` replaced by ``__``."""
    if not paths:
        return []
    absp = [os.path.abspath(p) for p in paths]
    root = os.path.commonpath([os.path.dirname(p) for p in absp])
    out = [os.path.splitext(os.path.relpath(p, root))[0].replace(os.sep, "__") for p in absp]
    dup = sorted({s for s in out if out.count(s) > 1})
    if dup:
        raise ValueError("several inputs map to the same output name: %s" % ", ".join(dup))
    return out


def mesh_seed(seed: int, stem: str) -> int:
    return (int(seed) * 2 ** 32 + zlib.crc32(stem.encode("utf-8"))) % 2 ** 64


def mesh_cloud(path: str, seed: int, points: int = DEFAULT_POINTS, resolution: int = DEFAULT_RESOLUTION, rotate: bool = True,
               codec=None) -> Tuple[np.ndarray, Dict[str, int]]:
    """One mesh -> (distinct grid points int32 [m,3] in lexicographic order, counts for the manifest).  ``seed`` is the mesh seed."""
    import torch
    from . import runtime
    verts, tris = load_mesh(path)
    info = {"vertices": len(verts), "triangles": len(tris)}
    c = codec or runtime.get_codec("voxception", "")
    rot = random_rotation(seed) if rotate else None
    pts = c.sample_mesh(c.to_device(verts, torch.float64), c.to_device(tris, torch.int32), points, seed, resolution, rot)
    cloud = pts.cpu().numpy()
    info.update(samples=int(points), unique_points=len(cloud))
    return cloud, info


def write_cubes(cloud: np.ndarray, out_dir: str, stem: str, cube_size: int = DEFAULT_CUBE_SIZE, min_num: int = DEFAULT_MIN_NUM) -> int:
    """Cut ``cloud`` with ``partition_points`` and write one int16 [n,3] ``<stem>_<k:04d>.npy`` per kept cube -> cubes written."""
    from .dataprocess import inout_points
    local, offsets, _, _ = inout_points.partition_points(cloud, cube_size, min_num)
    for k in range(len(offsets) - 1):
        np.save(os.path.join(out_dir, "%s_%04d.npy" % (stem, k)), local[offsets[k]:offsets[k + 1]])
    return len(offsets) - 1


def generate(paths: Sequence[str], out_dir: str, points: int = DEFAULT_POINTS, resolution: int = DEFAULT_RESOLUTION,
             cube_size: int = DEFAULT_CUBE_SIZE, min_num: int = DEFAULT_MIN_NUM, seed: int = 0, rotate: bool = True, log=print) -> int:
    """Every mesh of ``paths`` -> cube files and a manifest row in ``out_dir``.  Returns the number of meshes that failed."""
    os.makedirs(out_dir, exist_ok=True)
    names = stems(paths)
    failed = 0
    with open(os.path.join(out_dir, "manifest.csv"), "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=MANIFEST_FIELDS)
        w.writeheader()
        for path, stem in zip(paths, names):
            s = mesh_seed(seed, stem)
            row = {"stem": stem, "seed": s, "error": ""}
            try:
                cloud, info = mesh_cloud(path, s, points, resolution, rotate)
                row.update(info)
                row["cubes"] = write_cubes(cloud, out_dir, stem, cube_size, min_num)
            except (ValueError, RuntimeError, OSError) as e:
                failed += 1
                row["error"] = str(e).replace("\n", " ")
                log("%s: %s" % (path, row["error"]))
            w.writerow(row)
            f.flush()
    return failed


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="pcgcv1_b200.dataset", formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                 description="Sample meshes on the GPU and write the per-cube point files of train_hyper.")
    ap.add_argument("inputs", help="glob of mesh files (.obj / .off / .ply; '**' recurses); quote it")
    ap.add_argument("out_dir", help="directory for the <stem>_<k>.npy cube files and manifest.csv")
    ap.add_argument("--points", type=int, default=DEFAULT_POINTS, help="surface samples per mesh (1 .. 2^28)")
    ap.add_argument("--resolution", type=int, default=DEFAULT_RESOLUTION, help="grid size along the longest axis (2 .. 4096)")
    ap.add_argument("--cube_size", type=int, default=DEFAULT_CUBE_SIZE)
    ap.add_argument("--min_num", type=int, default=DEFAULT_MIN_NUM, help="cubes with fewer points are dropped")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-rotate", dest="rotate", action="store_false", help="keep the meshes' orientation")
    a = ap.parse_args(argv)
    if not 1 <= a.points <= 2 ** 28:
        ap.error("--points must be in 1 .. 2^28")
    if not 2 <= a.resolution <= 4096:
        ap.error("--resolution must be in 2 .. 4096")
    if not 1 <= a.cube_size <= 32767:
        ap.error("--cube_size must be in 1 .. 32767")
    if not 0 <= a.seed < 2 ** 32:
        ap.error("--seed must be in 0 .. 2^32 - 1")
    return a


def main(argv=None) -> int:
    a = parse_args(argv)
    paths = sorted(glob.glob(a.inputs, recursive=True))
    if not paths:
        print("no files match %s" % a.inputs, file=sys.stderr)
        return 1
    failed = generate(paths, a.out_dir, a.points, a.resolution, a.cube_size, a.min_num, a.seed, a.rotate,
                      log=lambda m: print(m, file=sys.stderr))
    print("%d meshes, %d failed; manifest: %s" % (len(paths), failed, os.path.join(a.out_dir, "manifest.csv")))
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main())
