"""Training data from meshes: the mesh reader (pcgc_mesh_parse), the surface sampler (pcgc_mesh_sample, Codec.sample_mesh) against
its NumPy restatement (oracle/meshsample.py), and the generator CLI (python -m pcgcv1_b200.dataset) feeding train_hyper."""
import csv
import ctypes as C
import os
import struct

import numpy as np
import pytest

from oracle import meshsample as om
from pcgcv1_b200 import _lib
from pcgcv1_b200 import dataset as ds


def _write(tmp_path, name, data):
    p = tmp_path / name
    p.parent.mkdir(parents=True, exist_ok=True)
    p.write_bytes(data if isinstance(data, bytes) else data.encode())
    return str(p)


def _write_obj(path, v, f):
    with open(path, "w") as fh:
        fh.write("".join("v %r %r %r\n" % tuple(p) for p in v.tolist()))
        fh.write("".join("f %d %d %d\n" % tuple(t) for t in (f + 1).tolist()))


# ------------------------------------------------------------------------------------------------ reader (CPU)
SQUARE_PYRAMID = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [0.5, 0.5, 1]], np.float64)


def test_obj_every_face_form(tmp_path):
    p = _write(tmp_path, "m.OBJ", """# comment
mtllib m.mtl
o thing
v 0 0 0
v 1 0 0 1.0
v 1 1 0
vt 0.5 0.5
vn 0 0 1
v 0 1 0
v 0.5 0.5 1
g side
usemtl red
s 1
f 1 2 3
f 1/1 3/1 4/1
f -5//1 -4//1 -2//1
f 1/1/1 2/1/1 3/1/1 4/1/1 5/1/1
l 1 2
p 3
""")
    v, t = ds.load_mesh(p)
    assert v.dtype == np.float64 and t.dtype == np.int32
    np.testing.assert_array_equal(v, SQUARE_PYRAMID)
    np.testing.assert_array_equal(t, [[0, 1, 2], [0, 2, 3], [0, 1, 3], [0, 1, 2], [0, 2, 3], [0, 3, 4]])


def test_off_glued_header_and_colours(tmp_path):
    glued = "OFF5 3 0\n# a comment\n" + "".join("%r %r %r\n" % tuple(x) for x in SQUARE_PYRAMID.tolist()) + \
        "3 0 1 4\n4 0 1 2 3\n5 0 1 2 3 4\n"
    v, t = ds.load_mesh(_write(tmp_path, "a.off", glued))
    np.testing.assert_array_equal(v, SQUARE_PYRAMID)
    np.testing.assert_array_equal(t, [[0, 1, 4], [0, 1, 2], [0, 2, 3], [0, 1, 2], [0, 2, 3], [0, 3, 4]])
    coloured = "COFF\n5 2 0\n" + "".join("%r %r %r 255 0 0 255\n" % tuple(x) for x in SQUARE_PYRAMID.tolist()) + \
        "3 0 1 4 10 20 30\n4 0 1 2 3 1 2 3\n"
    v, t = ds.load_mesh(_write(tmp_path, "b.off", coloured))
    np.testing.assert_array_equal(v, SQUARE_PYRAMID)
    np.testing.assert_array_equal(t, [[0, 1, 4], [0, 1, 2], [0, 2, 3]])


PLY_FACES = [[0, 1, 4], [0, 1, 2, 3], [1, 2, 4]]
PLY_TRIS = [[0, 1, 4], [0, 1, 2], [0, 2, 3], [1, 2, 4]]


def _ply_header(fmt, count_t, index_t):
    return ("ply\nformat %s 1.0\ncomment made by hand\nelement vertex 5\nproperty double x\nproperty float y\nproperty float z\n"
            "property float nx\nproperty uchar red\nelement material 2\nproperty float shine\nproperty int id\n"
            "element face 3\nproperty list %s %s vertex_indices\nproperty uchar flag\nend_header\n" % (fmt, count_t, index_t))


def test_ply_ascii(tmp_path):
    body = "".join("%r %r %r 0.5 200\n" % tuple(x) for x in SQUARE_PYRAMID.tolist()) + "0.25 7\n1.5 8\n" + \
        "".join("%d %s 1\n" % (len(f), " ".join(map(str, f))) for f in PLY_FACES)
    v, t = ds.load_mesh(_write(tmp_path, "a.ply", _ply_header("ascii", "uchar", "int") + body))
    np.testing.assert_array_equal(v, SQUARE_PYRAMID)
    np.testing.assert_array_equal(t, PLY_TRIS)


@pytest.mark.parametrize("count_t,index_t", [("uchar", "int"), ("int", "uint")])
def test_ply_binary_little_endian(tmp_path, count_t, index_t):
    cf, inf = {"uchar": "<B", "int": "<i"}[count_t], {"int": "<i", "uint": "<I"}[index_t]
    body = b"".join(struct.pack("<dfffB", x[0], x[1], x[2], 0.5, 200) for x in SQUARE_PYRAMID)
    body += struct.pack("<fi", 0.25, 7) + struct.pack("<fi", 1.5, 8)
    for f in PLY_FACES:
        body += struct.pack(cf, len(f)) + b"".join(struct.pack(inf, i) for i in f) + struct.pack("<B", 1)
    v, t = ds.load_mesh(_write(tmp_path, "b.PLY", _ply_header("binary_little_endian", count_t, index_t).encode() + body))
    np.testing.assert_array_equal(v, SQUARE_PYRAMID)
    np.testing.assert_array_equal(t, PLY_TRIS)
    with pytest.raises(ValueError, match="malformed"):                 # truncated binary body
        ds.load_mesh(_write(tmp_path, "c.ply", _ply_header("binary_little_endian", count_t, index_t).encode() + body[:-3]))


@pytest.mark.parametrize("name,text", [
    ("zero.obj", "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 0 1 2\n"),
    ("range.obj", "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 4\n"),
    ("range.off", "OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 3\n"),
    ("two.obj", "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2\n"),
    ("two.off", "OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n2 0 1\n"),
    ("short.off", "OFF\n3 2 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n"),
    ("junk.obj", "\x00\x01binary junk\n"),
])
def test_reader_rejects_malformed(tmp_path, name, text):
    with pytest.raises(ValueError, match="malformed"):
        ds.load_mesh(_write(tmp_path, name, text))


def test_ply_big_endian_is_unsupported(tmp_path):
    hdr = "ply\nformat binary_big_endian 1.0\nelement vertex 3\nproperty float x\nproperty float y\nproperty float z\n" \
          "element face 1\nproperty list uchar int vertex_indices\nend_header\n"
    body = b"".join(struct.pack(">fff", *x) for x in SQUARE_PYRAMID[:3]) + struct.pack(">Biii", 3, 0, 1, 2)
    with pytest.raises(ValueError, match="unsupported PLY format"):
        ds.load_mesh(_write(tmp_path, "be.ply", hdr.encode() + body))


def test_parse_overflow_reports_counts():
    data = b"v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1 2 3 4\n"
    L = _lib.lib()
    nv, nt = C.c_int64(), C.c_int64()
    v = np.empty((1, 3), np.float64)
    t = np.empty((1, 3), np.int32)
    assert L.pcgc_mesh_parse(data, len(data), _lib.MESH_OBJ, v.ctypes.data, 1, t.ctypes.data, 1, C.byref(nv), C.byref(nt)) == _lib.ERR_OVERFLOW
    assert (nv.value, nt.value) == (4, 2)
    v = np.empty((4, 3), np.float64)
    t = np.empty((2, 3), np.int32)
    assert L.pcgc_mesh_parse(data, len(data), _lib.MESH_OBJ, v.ctypes.data, 4, t.ctypes.data, 2, C.byref(nv), C.byref(nt)) == 0
    np.testing.assert_array_equal(t, [[0, 1, 2], [0, 2, 3]])


# ------------------------------------------------------------------------------------------------ oracle (CPU)
def _area_mesh():
    """Right triangles of areas 1 : 2 : 4 : 8 (a2 = 2, 4, 8, 16) and one degenerate face."""
    v, f = [], []
    for k, a2 in enumerate([2.0, 4.0, 8.0, 16.0]):
        o = np.array([3.0 * k, 0.0, 0.0])
        v += [o, o + [a2, 0, 0], o + [0, 1, 0]]
        f.append([3 * k, 3 * k + 1, 3 * k + 2])
    v += [np.array([0.0, 0.0, 1.0]), np.array([1.0, 1.0, 1.0]), np.array([2.0, 2.0, 1.0])]      # collinear: a2 = 0
    f.append([12, 13, 14])
    return np.array(v, np.float64), np.array(f, np.int32)


def test_oracle_samples_on_their_faces():
    v, f = om.icosphere(2)
    v = v * [3.0, 1.0, 0.5] + [10.0, -4.0, 2.0]
    _, samples, faces, _ = om.sample_mesh(v, f, 20000, seed=7, resolution=64)
    A, B, Cc = v[f[faces, 0]], v[f[faces, 1]], v[f[faces, 2]]
    nrm = np.cross(B - A, Cc - A)
    scale = np.abs(samples).max()
    assert np.all(np.abs(np.einsum("ij,ij->i", samples - A, nrm)) <= 1e-12 * scale * np.linalg.norm(nrm, axis=1))
    # barycentric coordinates inside [0, 1] (to rounding)
    M = np.stack([B - A, Cc - A], -1)
    for i in range(0, len(samples), 997):
        lam = np.linalg.lstsq(M[i], samples[i] - A[i], rcond=None)[0]
        assert lam.min() >= -1e-9 and lam.sum() <= 1 + 1e-9


def test_oracle_face_counts_chi2():
    from scipy import stats
    v, f = _area_mesh()
    _, _, faces, _ = om.sample_mesh(v, f, 1_000_000, seed=11, resolution=64)
    counts = np.bincount(faces, minlength=5)
    assert counts[4] == 0
    expected = 1_000_000 * np.array([1, 2, 4, 8]) / 15.0
    chi2 = float((((counts[:4] - expected) ** 2) / expected).sum())
    assert stats.chi2.sf(chi2, 3) > 1e-3, (counts, chi2)


def test_oracle_weight_threshold():
    # largest a2 = 1 -> frexp e = 1 -> threshold 2^-31
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [2.0 ** -31 * (1 - 2.0 ** -20), 0, 1], [0, 1, 1], [2.0 ** -31, 0, 1]])
    f = np.array([[0, 1, 2], [3, 4, 5], [3, 6, 5]], np.int32)
    a2, w, P = om.face_weights(v, f)
    assert a2[0] == 1.0 and a2[1] < 2.0 ** -31 <= a2[2]
    assert w[1] == 0 and w[2] == 1
    # the face just above the threshold owns the target P[2] (largest f with P[f] <= target); the one below owns none
    assert np.searchsorted(P[:-1], P[2], side="right") - 1 == 2
    assert not np.any(np.searchsorted(P[:-1], np.arange(P[1], P[2] + 1, dtype=np.uint64), side="right") - 1 == 1)


def test_mulhi64():
    rng = np.random.default_rng(0)
    a = rng.integers(0, 2 ** 64, 1000, dtype=np.uint64)
    for b in (1, 2 ** 32 - 1, 2 ** 32, 2 ** 63 + 12345, 2 ** 64 - 1):
        ref = np.array([(int(x) * b) >> 64 for x in a], dtype=np.uint64)
        np.testing.assert_array_equal(om.mulhi64(a, b), ref)


# ------------------------------------------------------------------------------------------------ rotation, names, seeds (CPU)
def test_random_rotation_orthonormal():
    for seed in (0, 1, 2 ** 40 + 3, 2 ** 64 - 1):
        R = ds.random_rotation(seed)
        assert np.abs(R @ R.T - np.eye(3)).max() <= 1e-15
        assert abs(np.linalg.det(R) - 1.0) <= 1e-15
    assert not np.array_equal(ds.random_rotation(1), ds.random_rotation(2))


def test_stems_and_seeds():
    a = ["/d/shapenet/02691156/x1/models/model_normalized.obj", "/d/shapenet/02958343/y2/models/model_normalized.obj",
         "/d/shapenet/02691156/x3/models/model_normalized.obj"]
    s = ds.stems(a)
    assert s[0] == "02691156__x1__models__model_normalized" and s[0] != s[1]
    # the same file in another list order: same stem, same seed
    s2 = ds.stems(a[::-1])
    assert s2[::-1] == s
    assert [ds.mesh_seed(5, x) for x in s2[::-1]] == [ds.mesh_seed(5, x) for x in s]
    assert ds.mesh_seed(0, s[0]) != ds.mesh_seed(1, s[0]) and ds.mesh_seed(0, s[0]) < 2 ** 32
    assert ds.mesh_seed(2 ** 32 - 1, "z") < 2 ** 64
    with pytest.raises(ValueError, match="same output name"):
        ds.stems(["/d/a.obj", "/d/a.off"])


# ------------------------------------------------------------------------------------------------ device against oracle (GPU)
def _device(codec, v, f, n, seed, R, rot):
    import torch
    pts, samples, faces = codec.sample_mesh(codec.to_device(np.asarray(v, np.float64), torch.float64),
                                            codec.to_device(np.asarray(f, np.int32), torch.int32), n, seed, R, rot, return_samples=True)
    return pts.cpu().numpy(), samples.cpu().numpy(), faces.cpu().numpy()


def _far_vertices():
    v, f = om.icosphere(1)
    v = np.concatenate([v, [[1e4, -1e4, 5e3], [-3e3, 2e3, 1e5]]])        # never referenced: the box must ignore them
    return v, f


def _sliver():
    return np.array([[0, 0, 0], [1, 0, 0], [0.5, 1e-9, 0], [0.2, 0.3, 0.4]]), np.array([[0, 1, 2], [0, 1, 3]], np.int32)


CASES = {
    "one_triangle": lambda: (np.array([[0.0, 0, 0], [1, 0.2, 0], [0.3, 1, 0.5]]), np.array([[0, 1, 2]], np.int32)),
    "areas_1248": _area_mesh,
    "icosphere_20k": lambda: om.icosphere(5),
    "far_unreferenced": _far_vertices,
    "offset_1e6": lambda: ((lambda v, f: (v + 1e6, f))(*om.icosphere(2))),
    "sliver": _sliver,
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("rotated", [False, True])
def test_device_matches_oracle(codec, case, rotated):
    v, f = CASES[case]()
    rot = ds.random_rotation(99) if rotated else None
    for n, R in ((1, 64), (1000 + 37, 2), (100_003, 64), (100_003, 1024)):
        pts, samples, faces = _device(codec, v, f, n, 1234567 + n, R, rot)
        opts, osamples, ofaces, okeys = om.sample_mesh(v, f, n, 1234567 + n, R, rot)
        np.testing.assert_array_equal(samples.view(np.uint64), osamples.view(np.uint64))
        np.testing.assert_array_equal(faces, ofaces)
        np.testing.assert_array_equal(pts, opts)
        u = np.unique(okeys)
        np.testing.assert_array_equal((pts[:, 0].astype(np.int64) * R + pts[:, 1]) * R + pts[:, 2], u)


@pytest.mark.gpu
def test_device_matches_oracle_large(codec):
    v, f = om.icosphere(5)
    rot = ds.random_rotation(3)
    for n, R in ((3_000_000, 4096), (3_000_000, 1024)):
        pts, samples, faces = _device(codec, v, f, n, 77, R, rot)
        opts, osamples, ofaces, _ = om.sample_mesh(v, f, n, 77, R, rot)
        np.testing.assert_array_equal(samples.view(np.uint64), osamples.view(np.uint64))
        np.testing.assert_array_equal(faces, ofaces)
        np.testing.assert_array_equal(pts, opts)


@pytest.mark.gpu
def test_box_ignores_unreferenced_vertices(codec):
    v, f = _far_vertices()
    pts = _device(codec, v, f, 200_000, 5, 64, None)[0]
    assert pts.min(0).tolist() == [0, 0, 0] and pts.max() == 63          # the sphere spans the grid, the far vertices do not count


@pytest.mark.gpu
def test_device_deterministic(codec):
    v, f = om.icosphere(4)
    rot = ds.random_rotation(8)
    a = _device(codec, v, f, 500_000, 42, 256, rot)
    b = _device(codec, v, f, 500_000, 42, 256, rot)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


@pytest.mark.gpu
def test_device_bad_arguments(codec):
    import torch
    from pcgcv1_b200._lib import PcgcError
    v, f = om.icosphere(1)
    dv = codec.to_device(v, torch.float64)
    df = codec.to_device(f, torch.int32)

    def bad(verts, tris, n=1000, R=64):
        with pytest.raises(PcgcError) as e:
            ptr = C.c_int64()
            pts = torch.empty((max(min(n, 1000), 1), 3), dtype=torch.int32, device=codec.dev)     # the arguments fail before any write
            codec._stream()
            codec._check(codec.lib.pcgc_mesh_sample(codec.ctx, verts.data_ptr(), len(verts), tris.data_ptr(), len(tris),
                                                    np.eye(3).ctypes.data, n, 1, R, pts.data_ptr(), C.byref(ptr), None, None))
        assert e.value.code == _lib.ERR_BAD_ARG

    flat = np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2]], np.float64)
    bad(codec.to_device(flat, torch.float64), codec.to_device(np.array([[0, 1, 2], [2, 1, 0]], np.int32), torch.int32))   # all degenerate
    bad(dv, codec.to_device(np.concatenate([f, [[0, 1, len(v)]]]).astype(np.int32), torch.int32))                        # index >= nv
    bad(dv, codec.to_device(np.concatenate([f, [[0, -1, 2]]]).astype(np.int32), torch.int32))                             # index < 0
    vn = v.copy()
    vn[f[3, 1]] = np.nan
    bad(codec.to_device(vn, torch.float64), df)                                                                            # NaN vertex
    for n, R in ((0, 64), (2 ** 28 + 1, 64), (100, 1), (100, 4097)):
        bad(dv, df, n, R)
    # the context stays usable after each failure
    assert len(_device(codec, v, f, 1000, 1, 64, None)[0]) > 0
    with pytest.raises(ValueError):
        codec.sample_mesh(dv, df, 0, 1, 64)


# ------------------------------------------------------------------------------------------------ end to end (GPU)
@pytest.mark.gpu
def test_cli_end_to_end(codec, tmp_path):
    from pcgcv1_b200 import train_hyper
    from pcgcv1_b200.dataprocess import inout_points
    src = tmp_path / "meshes"
    v1, f1 = om.icosphere(3)
    v2, f2 = om.icosphere(2)
    v2 = v2 * [2.0, 1.0, 0.7]
    (src / "c1" / "m").mkdir(parents=True)
    (src / "c2" / "m").mkdir(parents=True)
    _write_obj(str(src / "c1" / "m" / "model_normalized.obj"), v1, f1)
    _write_obj(str(src / "c2" / "m" / "model_normalized.obj"), v2, f2)
    _write(src, "box.off", "OFF\n8 6 0\n" + "".join("%d %d %d\n" % ((i >> 2) & 1, (i >> 1) & 1, i & 1) for i in range(8)) +
           "4 0 1 3 2\n4 4 6 7 5\n4 0 4 5 1\n4 2 3 7 6\n4 0 2 6 4\n4 1 5 7 3\n")
    hdr = "ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty double x\nproperty double y\nproperty double z\n" \
          "element face %d\nproperty list uchar int vertex_indices\nend_header\n" % (len(v2), len(f2))
    _write(src, "sphere.ply", hdr.encode() + v2.astype("<f8").tobytes() +
           b"".join(struct.pack("<Biii", 3, *t) for t in f2.tolist()))
    _write(src, "broken.obj", "v 0 0 0\nf 1 2 3\n")
    out = tmp_path / "cubes"
    argv = [str(src / "**" / "*.*"), str(out), "--points", "300000", "--resolution", "160", "--min_num", "32", "--seed", "4"]
    assert ds.main(argv) == 1
    rows = {r["stem"]: r for r in csv.DictReader(open(out / "manifest.csv"))}
    assert sorted(rows) == ["box", "broken", "c1__m__model_normalized", "c2__m__model_normalized", "sphere"]
    assert rows["broken"]["error"] and all(not rows[s]["error"] for s in rows if s != "broken")
    first = {p: (out / p).read_bytes() for p in sorted(os.listdir(out))}
    paths = {s: ["%s" % (out / p) for p in sorted(first) if p.startswith(s + "_")] for s in rows}
    assert not paths["broken"]
    for stem in ("c1__m__model_normalized", "sphere", "box"):
        mesh = {"c1__m__model_normalized": (v1, f1), "sphere": (v2, f2)}.get(stem) or ds.load_mesh(str(src / "box.off"))
        seed = ds.mesh_seed(4, stem)
        assert int(rows[stem]["seed"]) == seed
        cloud = om.sample_mesh(mesh[0], mesh[1], 300000, seed, 160, ds.random_rotation(seed))[0]
        assert int(rows[stem]["unique_points"]) == len(cloud)
        local, offsets, _, _ = inout_points.partition_points(cloud, 64, 32)
        assert int(rows[stem]["cubes"]) == len(offsets) - 1 == len(paths[stem]) > 0
        ref = inout_points.points2voxels([local[offsets[k]:offsets[k + 1]] for k in range(len(offsets) - 1)], 64)
        np.testing.assert_array_equal(train_hyper.CubeFiles.voxels(paths[stem]), ref)
        assert np.load(paths[stem][0]).dtype == np.int16
    # a second run writes the same bytes
    assert ds.main(argv) == 1
    assert {p: (out / p).read_bytes() for p in sorted(os.listdir(out))} == first
    # and the training loop runs on the files
    files = sorted(str(out / p) for p in first if p.endswith(".npy"))
    ckpt = str(tmp_path / "ckpt")
    train_hyper.train(files, ckpt, num_iteration=2, batch_size=2, display_step=1, save_step=10 ** 6, log=lambda *a: None)
    import json
    recs = [json.loads(x) for x in open(os.path.join(ckpt, "log.jsonl"))]
    assert len(recs) == 2 and all(np.isfinite(r["loss"]) for r in recs)
