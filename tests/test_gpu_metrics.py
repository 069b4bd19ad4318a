"""D1 / D2 figures on the GPU (pcgc_geometry_sums, myutils/pc_error_wrapper.geometry_metrics_device), the GPU-resident rho search
(eval_ablation_studies.DeviceRhoSearch) and the RD driver (rd_eval).

The device search resolves equidistant neighbours to the LOWEST index of the searched set; ``_brute_lowest`` restates the figures
with that rule (np.argmin returns the first minimum).  p2point figures do not depend on which equidistant neighbour is taken, so for
integer clouds they must equal the k-d tree path bit for bit; p2plane figures are pinned on the restatement."""
import configparser
import csv
import os

import numpy as np
import pytest

from pcgcv1_b200 import eval_ablation_studies as ev
from pcgcv1_b200.myutils import pc_error_wrapper as pw


def _nearest_lowest(q, s):
    """Index of the nearest point of s for every q (lowest index among equidistant ones), |e|^2 as (e0^2 + e1^2) + e2^2."""
    out = np.empty(len(q), np.int64)
    for i in range(0, len(q), 512):
        e = q[i:i + 512, None, :] - s[None, :, :]
        d = (e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]
        out[i:i + 512] = d.argmin(1)
    return out


def _brute_lowest(a, b, na, peak):
    """All 24 figures by brute force with the lowest-index tie rule."""
    ia, ib = _nearest_lowest(a, b), _nearest_lowest(b, a)
    e1, e2 = a - b[ia], b - a[ib]
    sq = lambda e: (e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]
    dot = lambda e, n: (e[:, 0] * n[:, 0] + e[:, 1] * n[:, 1]) + e[:, 2] * n[:, 2]
    d = {"p2point": {"1": sq(e1), "2": sq(e2)}}
    if na is not None:
        d["p2plane"] = {"1": dot(e1, na) ** 2, "2": dot(e2, na[ib]) ** 2}
    psnr = lambda v: float("inf") if v == 0 else 10 * np.log10(3 * peak * peak / v)
    out = {}
    for kind, v in d.items():
        for side in ("1", "2"):
            out["mse%s      (%s)" % (side, kind)] = v[side].mean()
            out["h.       %s(%s)" % (side, kind)] = v[side].max()
        mf, hf = max(v["1"].mean(), v["2"].mean()), max(v["1"].max(), v["2"].max())
        out["mseF      (%s)" % kind], out["h.        (%s)" % kind] = mf, hf
        for side in ("1", "2", "F"):
            out["mse%s,PSNR (%s)" % (side, kind)] = psnr(out["mse%s      (%s)" % (side, kind)])
        for side in ("1", "2"):
            out["h.,PSNR  %s(%s)" % (side, kind)] = psnr(out["h.       %s(%s)" % (side, kind)])
        out["h.,PSNR   (%s)" % kind] = psnr(hf)
    return out


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _close(got, want, rel):
    if want == float("inf") or got == float("inf"):
        return got == want
    return abs(got - want) <= rel * max(abs(want), 1e-300)


def _check(got, want, exact_p2point):
    assert set(got) == set(want)
    for k, v in want.items():
        if exact_p2point and "p2point" in k:
            assert got[k] == v, (k, got[k], v)
        else:
            assert _close(got[k], v, 1e-12), (k, got[k], v)


def test_brute_lowest_matches_brute_on_tie_free_input():
    from test_rho_search import _brute
    rng = np.random.default_rng(5)
    a = np.unique(rng.integers(0, 64, (400, 3)), axis=0).astype(np.float64)
    b = a[::2] + rng.uniform(-1.2, 1.2, a[::2].shape)
    na = _unit(rng, len(a))
    got = _brute_lowest(a, b, na, 1023.0)
    assert set(got) == set(pw.HEADERS)
    for k, v in _brute(a, b, na, 1023.0).items():
        assert abs(got[k] - v) <= 1e-12 * max(abs(v), 1.0), k


def _voxels_with_ties(seed, n=3000, extent=48):
    rng = np.random.default_rng(seed)
    a = np.unique(rng.integers(0, extent, (n, 3)), axis=0).astype(np.float64)
    b = a[rng.random(len(a)) < 0.6]
    b = b + rng.integers(-1, 2, b.shape)                 # a subset of A with +-1 jitter: many equidistant neighbours
    return a, b, _unit(rng, len(a))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_integer_clouds_with_ties(codec, seed):
    a, b, na = _voxels_with_ties(seed)
    got = pw.geometry_metrics_device(a, b, na, peak=1023.0, codec=codec)
    cpu = pw.geometry_metrics(a, b, na, peak=1023.0)
    for k in cpu:
        if "p2point" in k:
            assert got[k] == cpu[k], k
    _check(got, _brute_lowest(a, b, na, 1023.0), exact_p2point=True)


@pytest.mark.gpu
def test_off_grid_float_clouds(codec):
    rng = np.random.default_rng(11)
    a = np.unique(rng.integers(0, 200, (20000, 3)), axis=0).astype(np.float64)
    b = a[::3] + rng.uniform(-1.2, 1.2, a[::3].shape)
    na = _unit(rng, len(a))
    got = pw.geometry_metrics_device(a, b, na, peak=1023.0, codec=codec)
    want = pw.geometry_metrics(a, b, na, peak=1023.0)
    assert set(got) == set(want) == set(pw.HEADERS)
    for k, v in want.items():
        assert _close(got[k], v, 1e-12), (k, got[k], v)
    assert set(pw.geometry_metrics_device(a, b, None, codec=codec)) == {h for h in pw.HEADERS if "p2point" in h}


def _adversarial(name):
    rng = np.random.default_rng(7)
    if name == "identical":
        a = np.unique(rng.integers(0, 100, (2000, 3)), axis=0).astype(np.float64)
        return a, a.copy()
    if name == "single_point_a":
        return np.array([[3.0, 4.0, 5.0]]), rng.integers(0, 50, (500, 3)).astype(np.float64)
    if name == "single_point_b":
        return rng.integers(0, 50, (500, 3)).astype(np.float64), np.array([[3.0, 4.0, 5.0]])
    if name == "sizes_5000_vs_7":
        return rng.uniform(0, 300, (5000, 3)), rng.uniform(0, 300, (7, 3))
    if name == "one_cell":
        return rng.uniform(0, 40, (800, 3)), np.repeat([[10.0, 10.0, 10.0]], 64, axis=0)
    if name == "lattice_faces":
        g = np.stack(np.meshgrid(*[np.arange(16.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
        return g, g[::5] + 0.5                      # queries equidistant from 8 lattice points, on cell faces of any grid step
    if name == "negative":
        a = rng.integers(-6000, -5900, (3000, 3)).astype(np.float64)
        return a, a[::2] + rng.integers(-1, 2, a[::2].shape)
    if name == "hausdorff_outlier":
        a = np.unique(rng.integers(0, 100, (3000, 3)), axis=0).astype(np.float64)
        b = a[::2] + rng.integers(-1, 2, a[::2].shape)
        return np.concatenate([a, [[4100.0, 50.0, 60.0]]]), b
    if name == "vox12_extent":
        a = np.concatenate([rng.integers(0, 4096, (5000, 3)), np.array(np.meshgrid([0, 4095], [0, 4095], [0, 4095])).reshape(3, -1).T])
        b = np.concatenate([a[::3] + rng.integers(-3, 4, a[::3].shape), rng.integers(0, 4096, (500, 3))])
        return a.astype(np.float64), b.astype(np.float64)
    raise ValueError(name)


ADVERSARIAL = ["identical", "single_point_a", "single_point_b", "sizes_5000_vs_7", "one_cell", "lattice_faces", "negative",
               "hausdorff_outlier", "vox12_extent"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ADVERSARIAL)
def test_adversarial_inputs(codec, name):
    a, b = _adversarial(name)
    na = _unit(np.random.default_rng(3), len(a))
    integer = np.array_equal(a, np.rint(a)) and np.array_equal(b, np.rint(b))
    peak = 4095.0 if name == "vox12_extent" else 1023.0
    got = pw.geometry_metrics_device(a, b, na, peak=peak, codec=codec)
    _check(got, _brute_lowest(a, b, na, peak), exact_p2point=integer)
    cpu = pw.geometry_metrics(a, b, na, peak=peak)
    for k in cpu:
        if "p2point" in k:
            assert got[k] == cpu[k] if integer else _close(got[k], cpu[k], 1e-12), k
    if name == "identical":
        assert got["mseF,PSNR (p2point)"] == float("inf") and got["h.,PSNR   (p2point)"] == float("inf")
    if name == "hausdorff_outlier":
        assert got["h.       1(p2point)"] >= 3900.0 ** 2


@pytest.mark.gpu
def test_empty_sets_raise(codec):
    import torch
    a = torch.zeros((0, 3), dtype=torch.float64, device=codec.dev)
    b = torch.ones((4, 3), dtype=torch.float64, device=codec.dev)
    with pytest.raises(ValueError):
        codec.geometry_sums(a, b)
    with pytest.raises(ValueError):
        pw.geometry_metrics_device(np.ones((4, 3)), np.zeros((0, 3)), codec=codec)


@pytest.mark.gpu
def test_two_calls_give_the_same_bits(codec):
    import torch
    rng = np.random.default_rng(2)
    a = torch.tensor(rng.uniform(0, 1000, (200000, 3)), device=codec.dev)
    b = torch.tensor(rng.uniform(0, 1000, (150000, 3)), device=codec.dev)
    n = torch.tensor(_unit(rng, 200000), device=codec.dev)
    s1 = codec.geometry_sums(a, b, n).cpu()
    s2 = codec.geometry_sums(a, b, n).cpu()
    assert torch.equal(s1.view(torch.int64), s2.view(torch.int64))


def _decoded(max_cubes):
    from pcgcv1_b200 import synthetic, transform
    from pcgcv1_b200.models import model_voxception
    cubes, pos, nums = synthetic.workload("vox10", seed=0, max_cubes=max_cubes)
    pos = np.asarray(pos)[:len(cubes)]
    out = transform.compress_hyper(cubes, model_voxception, "")
    xs = transform.decompress_hyper(*[o.numpy() for o in out], model_voxception, "")
    pts = np.concatenate([np.argwhere(cubes[i, ..., 0] > 0) + pos[i] * 64 for i in range(len(cubes))]).astype(np.int32)
    return xs, nums[:len(cubes)], pos, pts


@pytest.mark.gpu
def test_full_vox10_cloud_against_decoded_reconstruction(codec, tmp_path):
    from pcgcv1_b200.dataprocess import inout_points as iop
    xs, nums, pos, pts = _decoded(None)
    src = str(tmp_path / "in.ply")
    iop.write_ply_data(src, pts)
    search = ev.DeviceRhoSearch(src, "", codec=codec)
    search.post("unused.ply", xs, nums, pos, 1, 64, 1.0)
    rec = search.points.cpu().numpy()
    assert len(pts) > 700_000 and len(rec) == int(np.asarray(nums, np.int64).sum())
    got = pw.geometry_metrics_device(pts, rec, None, codec=codec)
    want = pw.geometry_metrics(pts, rec, None)
    assert got == want


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1, 0.5])
def test_device_search_matches_file_search(codec, tmp_path, scale):
    from pcgcv1_b200.dataprocess import inout_points as iop
    xs, nums, pos, pts = _decoded(12)
    src = str(tmp_path / "in.ply")
    iop.write_ply_data(src, pts)
    rhos = ev.RHOS_D1
    seen_file, seen_dev = [], []

    def file_metric(a, b, n, res, show=False):
        r = pw.pc_error(a, b, n, res, show)
        seen_file.append(float(r[ev.ITEM_D1].iloc[0]))
        return r
    rec = str(tmp_path / "rec.ply")
    best_file = ev.select_optimal_rho(ev.ITEM_D1, rhos, src, rec, "", xs, nums, pos, scale, 64, 1024, metric=file_metric)

    search = ev.DeviceRhoSearch(src, "", codec=codec)

    def dev_metric(a, b, n, res, show=False):
        r = search.metric(a, b, n, res, show)
        seen_dev.append(r[ev.ITEM_D1])
        return r
    dev_rec = str(tmp_path / "dev_rec.ply")
    best_dev = ev.select_optimal_rho(ev.ITEM_D1, rhos, src, dev_rec, "", xs, nums, pos, scale, 64, 1024, post=search.post, metric=dev_metric)
    assert not os.path.exists(dev_rec)
    assert best_dev == best_file and len(seen_dev) == len(seen_file) >= 2
    if scale == 1:
        assert seen_dev == seen_file
    else:
        assert np.allclose(seen_dev, seen_file, rtol=0, atol=1e-4)
    # write() stores the last candidate as postprocess did
    search.write(dev_rec)
    assert open(dev_rec).read() == open(rec).read()


def _write_ply(name, pts, normals=None):
    with open(name, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n" % len(pts))
        if normals is not None:
            f.write("property float nx\nproperty float ny\nproperty float nz\n")
        f.write("end_header\n")
        for i, p in enumerate(pts):
            f.write(" ".join(repr(float(x)) for x in (list(p) + (list(normals[i]) if normals is not None else []))) + "\n")


@pytest.mark.gpu
def test_rd_driver_two_rate_points(codec, tmp_path, monkeypatch):
    from pcgcv1_b200 import rd_eval, synthetic
    from pcgcv1_b200.dataprocess import inout_points as iop
    from pcgcv1_b200.dataprocess.inout_bitstream import _paths
    pts = synthetic.cloud_vox10(seed=1, target_points=30000)
    src, srcn = str(tmp_path / "cloud.ply"), str(tmp_path / "cloud_n.ply")
    iop.write_ply_data(src, pts)
    _write_ply(srcn, pts, _unit(np.random.default_rng(0), len(pts)))
    ini = str(tmp_path / "rates.ini")
    with open(ini, "w") as f:
        f.write("[DEFAULT]\ncube_size = 64\nmin_num = 20\nresolution = 1024\n\n[R1]\nscale = 1.0\nckpt_dir = \n\n[R2]\nscale = 0.5\nckpt_dir = \n")
    out = str(tmp_path / "rd.csv")
    monkeypatch.chdir(tmp_path)
    rows = rd_eval.main([src, srcn, ini, out])
    with open(out) as f:
        got = list(csv.DictReader(f))
    assert [r["rate"] for r in got] == ["R1", "R2"] and list(got[0]) == rd_eval.COLUMNS
    for r in got:
        p = _paths("cloud", str(tmp_path / "rd_files" / r["rate"]))
        nbytes = sum(os.path.getsize(x) for x in (p.strings, p.head, p.hyper, p.pointnums, p.cubepos))
        assert int(r["bytes"]) == nbytes and float(r["bpp"]) == 8.0 * nbytes / len(pts)
        assert np.isfinite(float(r["d1_mseF_psnr"])) and np.isfinite(float(r["d2_mseF_psnr"]))
    cfg = configparser.ConfigParser()
    cfg.read(ini)
    for r in rows:
        assert float(cfg.get(r["rate"], "rho_d1")) == r["rho_d1"] and float(cfg.get(r["rate"], "rho_d2")) == r["rho_d2"]
    # a second run reads the stored rhos instead of searching
    def no_search(*a, **k):
        raise AssertionError("searched although the .ini holds the rhos")
    monkeypatch.setattr(ev, "select_optimal_rho", no_search)
    again = rd_eval.main([src, srcn, ini, out])
    assert [(r["rho_d1"], r["rho_d2"], r["d1_mseF_psnr"]) for r in again] == [(r["rho_d1"], r["rho_d2"], r["d1_mseF_psnr"]) for r in rows]
    with open(out) as f:
        assert len(list(csv.DictReader(f))) == 4
    # cube sizes other than 64 are refused as by the codec's command line
    cfg.set("DEFAULT", "cube_size", "32")
    with open(ini, "w") as f:
        cfg.write(f)
    with pytest.raises(SystemExit, match="64\\^3"):
        rd_eval.main([src, srcn, ini, out])
