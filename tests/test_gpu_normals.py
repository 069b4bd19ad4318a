"""k-nearest-neighbour PCA normals on the GPU (pcgc_estimate_normals, Codec.estimate_normals, pcgcv1_b200.normals) and the normals
file they produce for D2 (rd_eval --knn).

Oracle: ``_knn_lowest`` restates the neighbourhood rule (the k smallest (d2, index), d2 = (e0*e0 + e1*e1) + e2*e2), by brute force for
small clouds and through a k-d tree for large ones; ``_oracle_cov`` restates the two-pass covariance on coordinates relative to the
point, in the same order, and ``numpy.linalg.eigh`` gives the reference eigen-decomposition."""
import configparser
import csv
import os

import numpy as np
import pytest

from pcgcv1_b200 import normals as nm
from pcgcv1_b200 import rd_eval
from pcgcv1_b200.myutils import pc_error_wrapper as pw


def _d2(q, p):
    e = q[:, None, :] - p[None, :, :] if p.ndim == 2 else q[:, None, :] - p
    return (e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]


def _knn_brute(pts, k, queries=None):
    queries = np.arange(len(pts)) if queries is None else queries
    m = min(k, len(pts))
    out = np.empty((len(queries), m), np.int64)
    idx = np.arange(len(pts))
    for i in range(0, len(queries), 256):
        d = _d2(pts[queries[i:i + 256]], pts)
        order = np.lexsort((np.broadcast_to(idx, d.shape), d), axis=-1)
        out[i:i + 256] = order[:, :m]
    return out


def _knn_tree(pts, k, queries=None):
    from scipy.spatial import cKDTree
    queries = np.arange(len(pts)) if queries is None else queries
    m = min(k, len(pts))
    tree = cKDTree(pts)
    dk, _ = tree.query(pts[queries], k=m)
    rk = (dk.reshape(len(queries), m)[:, -1]) * (1 + 1e-9) + 1e-9      # the k-th distance, widened past any rounding
    out = np.empty((len(queries), m), np.int64)
    for row, (qi, cand) in enumerate(zip(queries, tree.query_ball_point(pts[queries], rk))):
        cand = np.asarray(cand, np.int64)
        d = _d2(pts[qi][None], pts[cand])[0]
        out[row] = cand[np.lexsort((cand, d))[:m]]
    return out


def _knn_lowest(pts, k, queries=None):
    """Indices of the min(k, n) points with the smallest (d2, index) for every query, in that order."""
    pts = np.asarray(pts, np.float64)
    return _knn_brute(pts, k, queries) if len(pts) <= 6000 else _knn_tree(pts, k, queries)


def _oracle_cov(pts, nbr, queries):
    """Two-pass covariance of every neighbourhood on u = p - q, running sums in neighbour order (the kernel's arithmetic)."""
    U = pts[nbr] - pts[queries][:, None, :]
    m = nbr.shape[1]
    mu = np.zeros((len(queries), 3))
    for j in range(m):
        mu = mu + U[:, j]
    mu = mu / m
    C = np.zeros((len(queries), 3, 3))
    for j in range(m):
        e = U[:, j] - mu
        C = C + e[:, :, None] * e[:, None, :]
    return C / m


def _check_normals(n, C):
    """The accuracy bar: a clear smallest eigenvalue pins the eigenvector to 1e-8; otherwise n lies in the low eigenspace."""
    w, v = np.linalg.eigh(C)
    assert np.all(np.abs(np.linalg.norm(n, axis=1) - 1.0) <= 1e-12)
    a = np.argmax(np.abs(n), axis=1)                                 # first maximum: lowest axis on a tie
    assert np.all(n[np.arange(len(n)), a] > 0)
    zero = np.all(C.reshape(len(C), 9) == 0, axis=1)
    assert np.array_equal(n[zero], np.tile([0.0, 0.0, 1.0], (int(zero.sum()), 1)))
    l0, l1, l2 = w[:, 0], w[:, 1], w[:, 2]
    clear = (l1 - l0 > 1e-6 * l2) & ~zero
    v0 = v[:, :, 0]
    err = np.minimum(np.linalg.norm(n - v0, axis=1), np.linalg.norm(n + v0, axis=1))
    assert np.all(err[clear] <= 1e-8), err[clear].max()
    Cn = np.einsum("pij,pj->pi", C, n)
    r = np.einsum("pi,pi->p", n, Cn)
    res = np.linalg.norm(Cn - r[:, None] * n, axis=1)
    low = ~clear & ~zero
    assert np.all(res[low] <= 1e-9 * l2[low]) and np.all(r[low] <= l0[low] + 1e-9 * l2[low])
    return int(clear.sum())


# ---- clouds ----------------------------------------------------------------------------------------------------------------------
def _cloud(name):
    rng = np.random.default_rng(17)
    if name == "ties":
        return np.unique(rng.integers(0, 24, (3000, 3)), axis=0).astype(np.float64)
    if name == "lattice16":
        return np.stack(np.meshgrid(*[np.arange(16.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
    if name == "off_grid":
        return rng.uniform(0, 50, (3000, 3))
    if name == "negative":
        return rng.integers(-6000, -5970, (3000, 3)).astype(np.float64)      # duplicates included
    if name == "vox12_extent":
        corners = np.array(np.meshgrid([0, 4095], [0, 4095], [0, 4095])).reshape(3, -1).T
        return np.concatenate([rng.integers(0, 4096, (5000, 3)), corners]).astype(np.float64)
    if name == "cluster_and_outliers":                                   # far queries go through the coarse level
        a = np.unique(rng.integers(0, 40, (2000, 3)), axis=0)
        return np.concatenate([a, [[3000, 20, 20], [3001, 22, 20], [20, 2500, 2600], [-900, -900, 4000]]]).astype(np.float64)
    if name == "single":
        return np.array([[3.0, 4.0, 5.0]])
    if name == "identical":
        return np.repeat([[5.0, 5.0, 5.0]], 100, axis=0)
    if name == "small":
        return rng.uniform(-3, 3, (10, 3))
    raise ValueError(name)


def _gpu(codec, pts, k):
    n, idx = codec.estimate_normals(codec.to_device(np.ascontiguousarray(pts, np.float64)), k, return_knn=True)
    return n.cpu().numpy(), idx.cpu().numpy()


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k", [("ties", 30), ("ties", 64), ("lattice16", 30), ("lattice16", 1), ("negative", 30),
                                    ("vox12_extent", 30)])
def test_tree_oracle_equals_brute_oracle(name, k):
    pts = _cloud(name)
    q = np.random.default_rng(1).choice(len(pts), 600, replace=False)
    assert np.array_equal(_knn_tree(pts, k, q), _knn_brute(pts, k, q))


@pytest.mark.parametrize("kind", ["integer", "float"])
def test_write_ply_normals_round_trips_bit_for_bit(tmp_path, kind):
    rng = np.random.default_rng(4)
    if kind == "integer":
        xyz = rng.integers(-5000, 5000, (500, 3)).astype(np.float64)
    else:
        xyz = rng.normal(0, 1e3, (500, 3)) * 10.0 ** rng.integers(-8, 3, (500, 1))
    n = rng.normal(size=(500, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    n[0] = [0.0, 0.0, 1.0]
    path = str(tmp_path / "c_n.ply")
    nm.write_ply_normals(path, xyz, n)
    got_xyz, got_n = pw._load_xyz_normals(path)
    assert np.array_equal(got_xyz.view(np.int64), xyz.view(np.int64))
    assert np.array_equal(got_n.view(np.int64), n.view(np.int64))
    if kind == "integer":
        assert open(path).read().split("end_header\n")[1].split("\n")[0].split()[:3] == ["%d" % v for v in xyz[0]]


def test_command_lines():
    a = nm.parse_args(["c.ply", "c_n.ply"])
    assert (a.input, a.output, a.knn) == ("c.ply", "c_n.ply", nm.DEFAULT_K) and nm.DEFAULT_K == 30
    assert nm.parse_args(["c.ply", "c_n.ply", "--knn", "64"]).knn == 64
    for bad in ("0", "65"):
        with pytest.raises(SystemExit):
            nm.parse_args(["c.ply", "c_n.ply", "--knn", bad])
    assert rd_eval.parse_args(["c.ply", "c_n.ply", "r.ini", "rd.csv"]).knn is None
    assert rd_eval.parse_args(["c.ply", "c_n.ply", "r.ini", "rd.csv", "--knn", "30"]).knn == 30
    with pytest.raises(SystemExit):
        rd_eval.parse_args(["c.ply", "c_n.ply", "r.ini", "rd.csv", "--knn", "65"])


# ---- GPU: neighbourhoods and normals ---------------------------------------------------------------------------------------------
CASES = [("ties", 30), ("ties", 1), ("ties", 64), ("lattice16", 30), ("off_grid", 30), ("off_grid", 64), ("negative", 30),
         ("vox12_extent", 30), ("cluster_and_outliers", 30), ("single", 1), ("single", 30), ("identical", 30), ("small", 20),
         ("small", 10)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,k", CASES)
def test_neighbours_and_normals_match_oracle(codec, name, k):
    pts = _cloud(name)
    n, idx = _gpu(codec, pts, k)
    want = _knn_lowest(pts, k)
    m = min(k, len(pts))
    assert idx.shape == (len(pts), k) and n.shape == (len(pts), 3)
    assert np.array_equal(idx[:, :m], want)
    assert np.all(idx[:, m:] == -1)
    _check_normals(n, _oracle_cov(pts, want, np.arange(len(pts))))
    if name in ("single", "identical"):
        assert np.array_equal(n, np.tile([0.0, 0.0, 1.0], (len(pts), 1)))


@pytest.mark.gpu
def test_collinear_neighbourhoods(codec):
    t = np.arange(200.0)[:, None]
    pts = np.concatenate([t * [1.0, 2.0, -1.0] + [5.0, -3.0, 7.0], t * [0.0, 0.0, 1.0] + [1000.0, 0.0, 0.0]])
    n, _ = _gpu(codec, pts, 12)
    d = np.where(np.arange(len(pts))[:, None] < 200, np.array([1.0, 2.0, -1.0]) / np.sqrt(6.0), [0.0, 0.0, 1.0])
    assert np.all(np.abs((n * d).sum(1)) <= 1e-12)
    assert np.all(np.abs(np.linalg.norm(n, axis=1) - 1.0) <= 1e-12)


def _share_within(n, truth, deg):
    cos = np.abs((n * truth).sum(1)) / np.linalg.norm(truth, axis=1)
    return float((cos >= np.cos(np.radians(deg))).mean())


@pytest.mark.gpu
def test_voxelised_sphere_and_plane(codec):
    g = np.arange(-102, 103)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    r = np.sqrt(x * x + y * y + z * z)
    sphere = np.stack([x, y, z], -1)[np.abs(r - 100.0) < 0.5].astype(np.float64)
    n = nm.estimate_normals(sphere, 30, codec)
    assert len(sphere) > 100_000 and _share_within(n, sphere, 10.0) >= 0.99
    u, v = np.meshgrid(np.arange(300.0), np.arange(300.0), indexing="ij")
    plane = np.stack([u.ravel(), v.ravel(), np.rint(0.3 * u.ravel() + 0.2 * v.ravel())], -1)
    n = nm.estimate_normals(plane, 30, codec)
    assert _share_within(n, np.tile([-0.3, -0.2, 1.0], (len(plane), 1)), 10.0) >= 0.99


@pytest.mark.gpu
def test_full_vox10_cloud_sample_and_determinism(codec):
    import torch
    from pcgcv1_b200 import synthetic
    pts = synthetic.cloud_vox10(0).astype(np.float64)
    assert len(pts) > 700_000
    t = codec.to_device(pts)
    n1, i1 = codec.estimate_normals(t, 30, return_knn=True)
    n2, i2 = codec.estimate_normals(t, 30, return_knn=True)
    assert torch.equal(n1.view(torch.int64), n2.view(torch.int64)) and torch.equal(i1, i2)
    assert torch.equal(codec.estimate_normals(t, 30).view(torch.int64), n1.view(torch.int64))
    q = np.sort(np.random.default_rng(0).choice(len(pts), 20_000, replace=False))
    want = _knn_tree(pts, 30, q)
    n, idx = n1.cpu().numpy()[q], i1.cpu().numpy()[q]
    assert np.array_equal(idx, want)
    assert _check_normals(n, _oracle_cov(pts, want, q)) > 0.9 * len(q)


@pytest.mark.gpu
def test_bad_arguments_raise(codec):
    import torch
    t = codec.to_device(np.zeros((8, 3)))
    for k in (0, 65):
        with pytest.raises(ValueError):
            codec.estimate_normals(t, k)
    out = torch.empty((8, 3), dtype=torch.float64, device=codec.dev)
    for k, n in ((0, 8), (65, 8), (30, 0)):
        assert codec.lib.pcgc_estimate_normals(codec.ctx, t.data_ptr(), n, k, out.data_ptr(), None) != 0
    assert codec.lib.pcgc_estimate_normals(codec.ctx, t.data_ptr(), 8, 30, None, None) != 0
    bad = [torch.zeros((0, 3), dtype=torch.float64, device=codec.dev), t.float(), codec.to_device(np.zeros((8, 2))),
           codec.to_device(np.zeros((3, 8))).t(), torch.zeros((8, 3), dtype=torch.float64)]
    for b in bad:
        with pytest.raises(ValueError):
            codec.estimate_normals(b, 30)


@pytest.mark.gpu
def test_geometry_sums_unchanged_by_normals_in_the_same_workspace(codec):
    import torch
    rng = np.random.default_rng(2)
    a = codec.to_device(rng.uniform(0, 1000, (50_000, 3)))
    b = codec.to_device(rng.uniform(0, 1000, (40_000, 3)))
    n = codec.estimate_normals(a, 30)
    s1 = codec.geometry_sums(a, b, n).cpu()
    codec.estimate_normals(codec.to_device(rng.uniform(0, 1000, (300_000, 3))), 64)          # grows the shared workspace
    s2 = codec.geometry_sums(a, b, n).cpu()
    assert torch.equal(s1.view(torch.int64), s2.view(torch.int64))


# ---- GPU: the normals file, the CPU metric and the RD driver ---------------------------------------------------------------------
def _write_xyz(path, pts):
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\nend_header\n" % len(pts))
        f.write("".join("%r %r %r\n" % tuple(p) for p in np.asarray(pts, np.float64).tolist()))


@pytest.mark.gpu
def test_cli_file_and_cpu_metric_agree_with_device(codec, tmp_path, monkeypatch):
    from pcgcv1_b200 import synthetic
    from pcgcv1_b200.dataprocess import inout_points as iop
    monkeypatch.chdir(tmp_path)                                      # no MPEG binary here: pc_error takes its CPU path
    pts = synthetic.cloud_vox10(seed=3, target_points=20000)
    src, srcn, rec = (str(tmp_path / f) for f in ("src.ply", "src_n.ply", "rec.ply"))
    iop.write_ply_data(src, pts)
    nm.main([src, srcn])
    xyz, n_file = pw._load_xyz_normals(srcn)
    n_dev = codec.estimate_normals(codec.to_device(pts.astype(np.float64)), 30)
    assert np.array_equal(xyz, pts.astype(np.float64))
    assert np.array_equal(n_file.view(np.int64), n_dev.cpu().numpy().view(np.int64))
    rng = np.random.default_rng(8)
    b = pts[::2] + rng.uniform(-1.3, 1.3, pts[::2].shape)             # off-grid: every nearest neighbour is unique
    _write_xyz(rec, b)
    cpu = pw.pc_error(src, rec, srcn, 1024).iloc[0].to_dict()
    dev = pw.geometry_metrics_device(pts, b, n_dev, peak=1023.0, codec=codec)
    keys = [h for h in pw.HEADERS if "p2plane" in h]
    assert all(k in cpu and k in dev for k in keys)
    for k in keys:
        assert abs(cpu[k] - dev[k]) <= 1e-12 * max(abs(cpu[k]), 1e-300), (k, cpu[k], dev[k])


@pytest.mark.gpu
def test_rd_driver_estimates_missing_normals_once(codec, tmp_path, monkeypatch):
    from pcgcv1_b200 import synthetic
    from pcgcv1_b200.dataprocess import inout_points as iop
    pts = synthetic.cloud_vox10(seed=1, target_points=30000)
    src, srcn = str(tmp_path / "cloud.ply"), str(tmp_path / "missing_n.ply")
    iop.write_ply_data(src, pts)
    ini = str(tmp_path / "rates.ini")
    with open(ini, "w") as f:
        f.write("[DEFAULT]\ncube_size = 64\nmin_num = 20\nresolution = 1024\n\n[R1]\nscale = 1.0\nckpt_dir = \n")
    out = str(tmp_path / "rd.csv")
    monkeypatch.chdir(tmp_path)
    assert not os.path.exists(srcn)
    rows = rd_eval.main([src, srcn, ini, out, "--knn", "30"])
    assert os.path.exists(srcn)
    xyz, n_file = pw._load_xyz_normals(srcn)
    assert np.array_equal(xyz, pts.astype(np.float64)) and n_file is not None
    with open(out) as f:
        got = list(csv.DictReader(f))
    assert len(got) == 1 and np.isfinite(float(got[0]["d2_mseF_psnr"])) and np.isfinite(float(got[0]["d2_h_psnr"]))
    cfg = configparser.ConfigParser()
    cfg.read(ini)
    assert float(cfg.get("R1", "rho_d2")) == rows[0]["rho_d2"]

    def no_estimate(*a, **k):
        raise AssertionError("estimated although the normals file exists")
    monkeypatch.setattr(nm, "make_normals_file", no_estimate)
    again = rd_eval.main([src, srcn, ini, out, "--knn", "30"])
    assert [(r["rho_d2"], r["d2_mseF_psnr"]) for r in again] == [(r["rho_d2"], r["d2_mseF_psnr"]) for r in rows]
