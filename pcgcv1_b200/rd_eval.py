"""Rate-distortion evaluation of one point cloud over the rate points of an ``.ini``: bits per input point against D1 / D2 PSNR.

    python -m pcgcv1_b200.rd_eval cloud.ply cloud_n.ply rates.ini rd.csv [--mode hyper|factorized]
                                  [--modelname models.model_voxception] [--rates R1,R3] [--knn K]

With ``--knn K`` and no file at ``cloud_n.ply``, the normals of ``cloud.ply`` are first estimated on the GPU from its K nearest
neighbours (``pcgcv1_b200.normals``) and written to ``cloud_n.ply``; later runs, and the MPEG binary, then read that file.  Without
``--knn``, or when the file exists, the normals file is read as given.

``rates.ini`` has the layout of the reference's rate-point files: ``[DEFAULT]`` with ``cube_size``, ``min_num`` and ``resolution``,
then one section per rate point (``[R1]`` .. ``[Rn]``) with ``scale``, ``ckpt_dir`` and optionally ``rho_d1`` / ``rho_d2``.  For every
rate section (all of them, or those named by ``--rates``):

1. ``preprocess`` + the mode's ``compress_*``; the container is written through ``inout_bitstream`` into ``<rd>_files/<rate>/``;
2. bpp = 8 * (bytes of the container's files, ``.cubepos`` included) / points of the input cloud;
3. the container is read back and decoded: the stream on disk is the one scored;
4. ``cfg_post_process`` with the GPU-resident search (``eval_ablation_studies.DeviceRhoSearch``) finds ``rho_d1`` / ``rho_d2`` when
   the section lacks them and writes them back to the ``.ini``; a later run reads them instead of searching;
5. D1 is scored at ``rho_d1``, D2 at ``rho_d2`` (the built-in figures, ``geometry_metrics_device``); the ``rho_d1`` reconstruction is
   kept as ``<rate>/<cloud>_rec.ply``;
6. one row is appended to the CSV (columns in ``COLUMNS``; stage times in seconds).

This is this project's driver, not a drop-in for the reference's ``eval.py`` (which is not available here): the command line and the
CSV columns are its own, and it scores with the built-in D1 / D2 figures even when the MPEG ``pc_error`` binary is present."""
from __future__ import annotations

import argparse
import configparser
import csv
import os
import time

COLUMNS = ["rate", "scale", "ckpt_dir", "points", "bytes", "bpp", "rho_d1", "rho_d2",
           "d1_mseF_psnr", "d1_h_psnr", "d2_mseF_psnr", "d2_h_psnr",
           "t_compress", "t_decompress", "t_rho_search", "t_score"]


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="pcgcv1_b200.rd_eval", formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    ap.add_argument("input", help="point cloud (.ply)")
    ap.add_argument("normals", help=".ply with the points of INPUT in the same order and their normals (nx ny nz)")
    ap.add_argument("ini", help="rate points: [DEFAULT] cube_size, min_num, resolution; [R1..Rn] scale, ckpt_dir[, rho_d1, rho_d2]")
    ap.add_argument("csv", help="CSV the rows are appended to; the containers go to <csv without .csv>_files/<rate>/")
    ap.add_argument("--mode", default="hyper", help="entropy model: 'hyper' or 'factorized'")
    ap.add_argument("--modelname", default="models.model_voxception", help="models.model_voxception or models.model_simple")
    ap.add_argument("--rates", default="", help="comma-separated sections to evaluate ('' = every section)")
    ap.add_argument("--knn", type=int, default=None,
                    help="when NORMALS does not exist: estimate the normals of INPUT from K nearest neighbours (1 .. 64) and write NORMALS")
    args = ap.parse_args(argv)
    if args.knn is not None and not 1 <= args.knn <= 64:
        ap.error("--knn must be in 1 .. 64")
    return args


def _container_bytes(name, rootdir):
    from .dataprocess.inout_bitstream import _paths
    p = _paths(name, rootdir)
    return sum(os.path.getsize(f) for f in (p.strings, p.head, p.hyper, p.pointnums, p.cubepos) if os.path.exists(f))


def evaluate_rate(config, ini, rate, args, search, n_points, workroot):
    """Steps 1-6 of the module docstring for one section; returns the CSV row as a dict."""
    from . import test
    from .eval_ablation_studies import ITEM_D1, ITEM_D2, cfg_post_process
    from .process import preprocess
    cube_size, min_num = config.getint(rate, "cube_size"), config.getint(rate, "min_num")
    res = config.getint(rate, "resolution")
    scale, ckpt_dir = config.getfloat(rate, "scale"), config.get(rate, "ckpt_dir", fallback="")
    s = test._Session(argparse.Namespace(mode=args.mode, modelname=args.modelname, ckpt_dir=ckpt_dir))
    search.codec = s.codec
    name = os.path.split(args.input)[-1][:-4]
    rootdir = os.path.join(workroot, rate)

    t0 = time.time()
    cubes, cube_positions, points_numbers = preprocess(args.input, scale, cube_size, min_num, codec=s.codec)
    coded = [v.numpy() for v in s.encode(cubes, s.model, ckpt_dir)]
    if args.mode == "hyper":
        y_strings, y_min_vs, y_max_vs, y_shape, z_strings, z_min_v, z_max_v, z_shape = coded
        s.store(name, y_strings, z_strings, points_numbers, cube_positions, y_min_vs, y_max_vs, y_shape, z_min_v, z_max_v, z_shape,
                rootdir=rootdir)
    else:
        strings, min_v, max_v, shape = coded
        s.store(name, strings, points_numbers, cube_positions, min_v, max_v, shape, rootdir=rootdir)
    t1 = time.time()
    nbytes = _container_bytes(name, rootdir)

    if args.mode == "hyper":
        y_strings, z_strings, points_numbers, cube_positions, y_min_vs, y_max_vs, y_shape, z_min_v, z_max_v, z_shape = s.fetch(name, rootdir)
        logits = s.decode(y_strings, y_min_vs, y_max_vs, y_shape, z_strings, z_min_v, z_max_v, z_shape, s.model, ckpt_dir)
    else:
        strings, points_numbers, cube_positions, min_v, max_v, shape = s.fetch(name, rootdir)
        logits = s.decode(strings, min_v, max_v, shape, s.model, ckpt_dir)
    logits = s.codec.to_device(logits)             # resident for the whole search
    t2 = time.time()

    rec = os.path.join(rootdir, name + "_rec.ply")
    rho_d1, rho_d2 = cfg_post_process(config, ini, rate, args.input, rec, args.normals, logits, points_numbers, cube_positions, scale,
                                      cube_size, res, post=search.post, metric=search.metric)
    t3 = time.time()

    search.post(rec, logits, points_numbers, cube_positions, scale, cube_size, rho_d1)
    d1 = search.metric(args.input, rec, args.normals, res)
    search.write(rec)
    search.post(rec, logits, points_numbers, cube_positions, scale, cube_size, rho_d2)
    d2 = search.metric(args.input, rec, args.normals, res)
    t4 = time.time()
    return {"rate": rate, "scale": scale, "ckpt_dir": ckpt_dir, "points": n_points, "bytes": nbytes, "bpp": 8.0 * nbytes / n_points,
            "rho_d1": rho_d1, "rho_d2": rho_d2, "d1_mseF_psnr": d1[ITEM_D1], "d1_h_psnr": d1["h.,PSNR   (p2point)"],
            "d2_mseF_psnr": d2.get(ITEM_D2, float("nan")), "d2_h_psnr": d2.get("h.,PSNR   (p2plane)", float("nan")),
            "t_compress": round(t1 - t0, 4), "t_decompress": round(t2 - t1, 4), "t_rho_search": round(t3 - t2, 4),
            "t_score": round(t4 - t3, 4)}


def main(argv=None):
    from . import test
    from .dataprocess.inout_points import load_ply_data
    from .eval_ablation_studies import DeviceRhoSearch
    args = parse_args(argv)
    config = configparser.ConfigParser()
    if not config.read(args.ini):
        raise SystemExit("cannot read %s" % args.ini)
    rates = [r for r in args.rates.split(",") if r] or config.sections()
    for rate in rates:
        if not config.has_section(rate):
            raise SystemExit("%s has no section [%s]" % (args.ini, rate))
        if config.getint(rate, "cube_size") != 64:
            raise SystemExit(test.CUBE_SIZE_MESSAGE)
    n_points = len(load_ply_data(args.input))
    if args.knn is not None and not os.path.exists(args.normals):
        from .normals import make_normals_file
        make_normals_file(args.input, args.normals, args.knn)
    search = DeviceRhoSearch(args.input, args.normals)
    workroot = (args.csv[:-4] if args.csv.endswith(".csv") else args.csv) + "_files"
    rows = []
    for rate in rates:
        row = evaluate_rate(config, args.ini, rate, args, search, n_points, workroot)
        new = not os.path.exists(args.csv)
        with open(args.csv, "a", newline="") as f:
            w = csv.DictWriter(f, fieldnames=COLUMNS)
            if new:
                w.writeheader()
            w.writerow(row)
        print(", ".join("%s %s" % (k, row[k]) for k in COLUMNS))
        rows.append(row)
    return rows


if __name__ == "__main__":
    main()
