"""Command line of the codec with the reference's surface (``test.py:24-115``): the same positional arguments, option names,
defaults and file naming (``./compressed/<name>.*`` on the way in, ``<name>_rec.ply`` on the way out), so scripts written for the
reference run unchanged:

    python -m pcgcv1_b200.test compress   cloud.ply          [--mode hyper|factorized] [--modelname models.model_voxception] [--ckpt_dir DIR]
    python -m pcgcv1_b200.test decompress compressed/cloud   [... the same options ...]

``--modelname`` takes the reference's module paths; ``--gpu 0`` is refused instead of silently falling back (there is no CPU path)."""
from __future__ import annotations

import argparse
import importlib
import os

# (flag, type, default, help) -- names and defaults are the reference's (test.py:33-42)
_OPTIONS = [
    ("--mode", str, "hyper", "entropy model: 'hyper' (hyperprior + conditional model) or 'factorized'"),
    ("--modelname", str, "models.model_voxception", "transform module: models.model_voxception or models.model_simple"),
    ("--ckpt_dir", str, "", "directory with weights.npz or a TF-1.13 checkpoint ('' = seeded synthetic weights)"),
    ("--scale", float, 1.0, "geometry scaling applied before coding and undone after decoding"),
    ("--cube_size", int, 64, "edge of the cubes the cloud is partitioned into"),
    ("--min_num", int, 64, "cubes with fewer points are dropped"),
    ("--rho", float, 1.0, "output points per input point (top-k classification)"),
    ("--gpu", int, 1, "kept for compatibility; must be 1"),
]

CUBE_SIZE_MESSAGE = "the transforms are built for 64^3 cubes (the reference's default and its checkpoints)"


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="pcgcv1_b200.test", formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    ap.add_argument("command", choices=["compress", "decompress"], help="compress: .ply -> ./compressed/<name>.*; decompress: the reverse")
    ap.add_argument("input", nargs="?", help="point cloud (.ply) to compress, or compressed/<name> to decompress")
    ap.add_argument("output", nargs="?", help="name of the compressed set / of the reconstructed .ply")
    for flag, typ, default, text in _OPTIONS:
        ap.add_argument(flag, type=typ, default=default, dest=flag.lstrip("-"), help=text)
    args = ap.parse_args(argv)
    print(args)
    return args


class _Session:
    """Everything one invocation needs: the model module, its codec and the mode-specific pairs of functions."""

    def __init__(self, args):
        from . import runtime, transform
        from .dataprocess import inout_bitstream as ibs
        name = args.modelname if args.modelname.startswith("pcgcv1_b200.") else "pcgcv1_b200." + args.modelname
        self.args = args
        self.model = importlib.import_module(name)
        self.codec = runtime.get_codec(self.model, args.ckpt_dir)
        if args.mode == "hyper":
            self.encode, self.decode = transform.compress_hyper, transform.decompress_hyper
            self.store, self.fetch = ibs.write_binary_files_hyper, ibs.read_binary_files_hyper
        elif args.mode == "factorized":
            self.encode, self.decode = transform.compress_factorized, transform.decompress_factorized
            self.store, self.fetch = ibs.write_binary_files_factorized, ibs.read_binary_files_factorized
        else:
            raise SystemExit("--mode must be 'hyper' or 'factorized'")

    def compress(self):
        from .process import preprocess
        a = self.args
        name = a.output or os.path.split(a.input)[-1][:-4]
        cubes, cube_positions, points_numbers = preprocess(a.input, a.scale, a.cube_size, a.min_num, codec=self.codec)
        coded = [v.numpy() for v in self.encode(cubes, self.model, a.ckpt_dir)]
        if a.mode == "hyper":
            y_strings, y_min_vs, y_max_vs, y_shape, z_strings, z_min_v, z_max_v, z_shape = coded
            self.store(name, y_strings, z_strings, points_numbers, cube_positions, y_min_vs, y_max_vs, y_shape, z_min_v, z_max_v, z_shape,
                       rootdir="./compressed")
        else:
            strings, min_v, max_v, shape = coded
            self.store(name, strings, points_numbers, cube_positions, min_v, max_v, shape, rootdir="./compressed")

    def decompress(self):
        from .process import postprocess
        a = self.args
        rootdir, name = os.path.split(a.input)
        target = a.output or name + "_rec.ply"
        if a.mode == "hyper":
            y_strings, z_strings, points_numbers, cube_positions, y_min_vs, y_max_vs, y_shape, z_min_v, z_max_v, z_shape = self.fetch(name, rootdir)
            logits = self.decode(y_strings, y_min_vs, y_max_vs, y_shape, z_strings, z_min_v, z_max_v, z_shape, self.model, a.ckpt_dir)
        else:
            strings, points_numbers, cube_positions, min_v, max_v, shape = self.fetch(name, rootdir)
            logits = self.decode(strings, min_v, max_v, shape, self.model, a.ckpt_dir)
        postprocess(target, logits, points_numbers, cube_positions, a.scale, a.cube_size, a.rho, codec=self.codec)


def main(argv=None):
    args = parse_args(argv)
    if args.gpu != 1:
        raise SystemExit("pcgcv1_b200 has no CPU path (--gpu 0): the codec is the CUDA library")
    if args.cube_size != 64:
        raise SystemExit(CUBE_SIZE_MESSAGE)
    session = _Session(args)
    getattr(session, args.command)()


if __name__ == "__main__":
    main()
