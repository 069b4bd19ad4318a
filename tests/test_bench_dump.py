"""bench.py --dump-outputs: what the timed path computed in its last step, written as float32 / float64 .npy files (long outputs
as a seeded sample) so that two builds run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(directory):
    return {name: np.load(os.path.join(directory, name + ".npy")) for name in bench.DUMP_ARRAYS}


def test_dump_writes_float_arrays_and_samples_the_long_ones_at_fixed_positions(tmp_path):
    import torch
    assert sum(np.dtype(d).itemsize * cap for d, cap in bench.DUMP_ARRAYS.values()) <= bench.DUMP_LIMIT_BYTES
    lengths = {name: 11 for name in bench.DUMP_ARRAYS}
    lengths["occupancy_logits"] = bench.DUMP_ARRAYS["occupancy_logits"][1] + 1000
    lengths["occupied_voxels"] = 3 * bench.DUMP_ARRAYS["occupied_voxels"][1]
    arrays = {name: torch.arange(n, dtype=torch.int64).reshape(-1, 1) for name, n in lengths.items()}   # value = position
    bench.dump_outputs(arrays, str(tmp_path / "a"))
    bench.dump_outputs(arrays, str(tmp_path / "b"))
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sum(v.nbytes for v in a.values()) <= bench.DUMP_LIMIT_BYTES
    for name, (dtype, cap) in bench.DUMP_ARRAYS.items():
        v = a[name]
        assert v.dtype == dtype and v.ndim == 1 and len(v) == min(lengths[name], cap)
        assert np.array_equal(v, b[name])                                   # the same positions every time
        if lengths[name] <= cap:
            assert np.array_equal(v, np.arange(lengths[name]))
        else:                                                               # distinct positions, in order, inside the array
            assert (np.diff(v) > 0).all() and v[0] >= 0 and v[-1] < lengths[name]


@pytest.mark.gpu
def test_dump_holds_what_the_public_api_returns_for_the_same_cubes(tmp_path, codec):
    """7 cubes of the benchmark's cloud: every dumped array equals what compress_hyper / decompress_hyper / select_voxels give
    for those cubes (the whole of each array: nothing is long enough to be sampled), and --steps sets the timed steps."""
    import torch
    from pcgcv1_b200 import synthetic, transform
    from pcgcv1_b200.dataprocess import inout_points
    from pcgcv1_b200.models import model_voxception
    B = 7
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cubes", str(B), "--steps", "2", "--warmup", "1", "--no-cpu",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["cubes_per_gpu"] == B
    got = _load(str(tmp_path))

    cubes, _, nums = synthetic.workload("vox10", seed=0, max_cubes=B)
    host = [o.numpy() for o in transform.compress_hyper(cubes, model_voxception, "")]
    strings = [bytes(s) for s in host[0]]
    assert np.array_equal(got["y_strings"], np.frombuffer(b"".join(strings), np.uint8))
    assert np.array_equal(got["y_string_offsets"], np.concatenate([[0], np.cumsum([len(s) for s in strings])]))
    assert np.array_equal(got["y_minmax"], np.stack([host[1], host[2]], -1).reshape(-1))
    eb = transform._bottleneck(codec, 8)
    z_hat, _, _, _ = codec.factorized(eb._slot, codec.hyper_encode(codec.analysis(codec.to_device(cubes))), want_p=False, want_bits=False)
    assert np.array_equal(got["z_hat"], z_hat.cpu().numpy().reshape(-1))
    xs = transform.decompress_hyper(*host, model_voxception, "")
    logits = xs.tensor.cpu().numpy()
    mask = inout_points.select_voxels(xs, nums, 1.0, codec=codec, dtype="uint8")
    torch.cuda.synchronize()
    assert np.array_equal(got["occupancy_logits"], logits.reshape(-1))
    assert np.array_equal(got["occupied_voxels"], np.flatnonzero(mask))
    assert np.array_equal(got["voxel_counts"], mask.reshape(B, -1).sum(1))
