"""Drop-in for ``myutils/pc_error_wrapper.py``: ``pc_error(infile1, infile2, normal1, res, show=False)`` -> one-row table of
the geometry-distortion figures the rho search and the RD scripts read (``eval_ablation_studies.py:152-205``).

The reference shells out to a prebuilt MPEG ``pc_error`` 0.13.4 binary, ``myutils/pc_error_d`` relative to the working directory
(pc_error_wrapper.py:48-53), and greps its report for 24 headers (:29-46).  No source for that tool exists in the reference, so it
is not rebuilt.  When the binary is present it is called with the reference's exact command line.  When it is absent the same 24
keys are computed here from the tool's published definitions (MPEG document N18665 "Common test conditions", metrics D1 / D2):

    direction 1 (A -> B): for every point a of A, its nearest neighbour b in B, e = a - b;
        point-to-point  d = |e|^2;  point-to-plane  d = (e . n_a)^2  with n_a the normal of a (file ``normal1``)
    direction 2 (B -> A): the same from B, the plane taken at the nearest point of A (its normal)
    mse = mean d, h. = max d (Hausdorff), symmetric figure = max of the two directions,
    PSNR = 10 log10(3 p^2 / value) with p = ``res - 1`` (the ``--resolution`` the reference passes).

Parity of the built-in figures against the binary is UNPINNED (the binary is absent here); they are pinned on a brute-force
restatement of these formulas in tests/test_rho_search.py."""
from __future__ import annotations

import os
import subprocess
import time

import numpy as np

PC_ERROR = "myutils/pc_error_d"

_KINDS = ("h.       %s(p2point)", "h.,PSNR  %s(p2point)", "h.       %s(p2plane)", "h.,PSNR  %s(p2plane)",
          "mse%s      (p2point)", "mse%s,PSNR (p2point)", "mse%s      (p2plane)", "mse%s,PSNR (p2plane)")
HEADERS = [k % "1" for k in _KINDS] + [k % "2" for k in _KINDS] + \
          ["h.        (p2point)", "h.,PSNR   (p2point)", "h.        (p2plane)", "h.,PSNR   (p2plane)",
           "mseF      (p2point)", "mseF,PSNR (p2point)", "mseF      (p2plane)", "mseF,PSNR (p2plane)"]


def have_pc_error() -> bool:
    return os.path.isfile(PC_ERROR) and os.access(PC_ERROR, os.X_OK)


def get_points_number(filedir):
    """``element vertex N`` of a .ply header (pc_error_wrapper.py:6-14)."""
    with open(filedir) as f:
        line = f.readline()
        while line.find("element vertex") == -1:
            if not line:
                raise ValueError("%s: no 'element vertex' line" % filedir)
            line = f.readline()
    return int(line.split(" ")[-1][:-1])


def number_in_line(line):
    """The last token of a report line that parses as a float (pc_error_wrapper.py:16-24)."""
    number = None
    for item in line.split(" "):
        try:
            number = float(item)
        except ValueError:
            continue
    return number


def _load_xyz_normals(filename):
    """ASCII .ply -> (xyz float64 [n,3], normals float64 [n,3] or None).  Normals = properties nx ny nz when the header names them."""
    props, n, body = [], None, 0
    with open(filename, "rb") as f:
        data = f.read()
    pos = 0
    while True:
        end = data.index(b"\n", pos)
        line = data[pos:end].decode("ascii", "replace").strip()
        pos = end + 1
        if line.startswith("element vertex"):
            n = int(line.split()[-1])
        elif line.startswith("property") and n is not None:
            props.append(line.split()[-1])
        elif line == "end_header":
            body = pos
            break
    arr = np.loadtxt(data[body:].decode("ascii").splitlines()[:n], dtype=np.float64, ndmin=2)
    cols = {p: i for i, p in enumerate(props)}
    xyz = arr[:, [cols.get("x", 0), cols.get("y", 1), cols.get("z", 2)]]
    normals = arr[:, [cols["nx"], cols["ny"], cols["nz"]]] if all(k in cols for k in ("nx", "ny", "nz")) else None
    return xyz, normals


def _figures(stats, peak):
    """``stats[kind][side] = (mse, h)`` for kind in p2point[, p2plane] and side "1" / "2" -> the dict of HEADERS keys."""
    psnr = lambda v: float("inf") if v == 0 else 10.0 * np.log10(3.0 * peak * peak / v)
    out = {}
    for kind in stats:
        for side in ("1", "2"):
            mse, h = stats[kind][side]
            out["h.       %s(%s)" % (side, kind)], out["h.,PSNR  %s(%s)" % (side, kind)] = h, psnr(h)
            out["mse%s      (%s)" % (side, kind)], out["mse%s,PSNR (%s)" % (side, kind)] = mse, psnr(mse)
        hf = max(out["h.       1(%s)" % kind], out["h.       2(%s)" % kind])
        mf = max(out["mse1      (%s)" % kind], out["mse2      (%s)" % kind])
        out["h.        (%s)" % kind], out["h.,PSNR   (%s)" % kind] = hf, psnr(hf)
        out["mseF      (%s)" % kind], out["mseF,PSNR (%s)" % kind] = mf, psnr(mf)
    return out


def geometry_metrics(a, b, normals_a=None, peak=1023.0):
    """The 24 figures of ``pc_error -a A -b B -n N --hausdorff=1 --resolution=peak`` from their definitions (module docstring).
    ``a`` [n,3], ``b`` [m,3]; ``normals_a`` [n,3] or None (then the p2plane keys are absent, as when the tool runs without -n)."""
    from scipy.spatial import cKDTree
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if len(a) == 0 or len(b) == 0:
        raise ValueError("geometry_metrics: empty point cloud")
    _, ia = cKDTree(b).query(a)                       # nearest point of B for every a
    _, ib = cKDTree(a).query(b)                       # nearest point of A for every b
    e1, e2 = a - b[ia], b - a[ib]
    d = {"1": {"p2point": (e1 * e1).sum(1)}, "2": {"p2point": (e2 * e2).sum(1)}}
    if normals_a is not None:
        na = np.asarray(normals_a, np.float64)
        d["1"]["p2plane"] = ((e1 * na).sum(1)) ** 2
        d["2"]["p2plane"] = ((e2 * na[ib]).sum(1)) ** 2
    return _figures({kind: {side: (float(d[side][kind].mean()), float(d[side][kind].max())) for side in ("1", "2")} for kind in d["1"]},
                    peak)


def geometry_metrics_device(a, b, normals_a=None, peak=1023.0, codec=None):
    """``geometry_metrics`` on the GPU (``Codec.geometry_sums``: exact grid search, lowest index of the searched set on ties):
    the same keys and the same mean / max / PSNR expressions.  ``a``, ``b``, ``normals_a``: [n,3] torch tensors (moved to the
    codec's device as float64 if they are not there) or arrays.  For integer coordinates the p2point figures equal
    ``geometry_metrics``' bit for bit; the p2plane figures can differ where the nearest neighbour is not unique (the k-d tree's
    tie order is unspecified)."""
    import torch
    from .. import runtime
    c = codec or runtime.get_codec("voxception", "")
    a, b = c.to_device(a, torch.float64), c.to_device(b, torch.float64)
    n = None if normals_a is None else c.to_device(normals_a, torch.float64)
    if len(a) == 0 or len(b) == 0:
        raise ValueError("geometry_metrics: empty point cloud")
    s = runtime.to_host(c.geometry_sums(a, b, n), "geometry_sums").reshape(2, 2, 2).astype(np.float64)
    count = {"1": len(a), "2": len(b)}
    kinds = ("p2point",) if n is None else ("p2point", "p2plane")
    return _figures({kind: {side: (float(s[int(side) - 1, k, 0]) / count[side], float(s[int(side) - 1, k, 1])) for side in ("1", "2")}
                     for k, kind in enumerate(kinds)}, peak)


def pc_error(infile1, infile2, normal1, res, show=False):
    """One-row pandas DataFrame keyed by the reference's 24 headers (pc_error_wrapper.py:26-74)."""
    import pandas as pd
    start = time.time()
    results = {}
    if have_pc_error():
        command = str(PC_ERROR + " -a " + infile1 + " -b " + infile2 + " -n " + normal1 + " --hausdorff=1 " + " --resolution=" + str(res - 1))
        subp = subprocess.Popen(command, shell=True, stdout=subprocess.PIPE)
        c = subp.stdout.readline()
        while c:
            line = str(c, encoding="utf8")
            if show:
                print(line)
            for key in HEADERS:
                if line.find(key) != -1:
                    results[key] = number_in_line(line)
            c = subp.stdout.readline()
        subp.wait()
    else:
        a, _ = _load_xyz_normals(infile1)
        b, _ = _load_xyz_normals(infile2)
        normals = None
        if normal1 and os.path.isfile(normal1):
            an, normals = _load_xyz_normals(normal1)
            if normals is not None and (len(an) != len(a) or not np.array_equal(an, a)):
                raise ValueError("%s does not list the points of %s in the same order" % (normal1, infile1))
        results = geometry_metrics(a, b, normals, peak=float(res - 1))
        if show:
            for k in HEADERS:
                if k in results:
                    print("%s: %s" % (k, results[k]))
    print("===== measure PCC quality using `pc_error` version 0.13.4", round(time.time() - start, 4))
    return pd.DataFrame([results])
