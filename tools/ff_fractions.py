"""Far-field tile fractions of the analysis 64^3 stage for a workload, as the encoder meets them in steady state (DESIGN 4.1).

Per layer (receptive radius 1 .. 7: X0, T1a, X1, T1b, X2, T1c, X3) and per 8 (x) x 32 (y) x 1 (z) tile of each cube: near (computed),
restore (far now, near for the cube the same sub-batch slot held before) or skip (far for both).  The bench encodes the same cloud every
step in sub-batches of 64, so slot s of sub-batch k follows slot s of the sub-batch before it (the last one of the previous step for k = 0).
K_a16 decides per 16-slice segment: a segment with any near or restore tile is computed whole.  X3 has no previous state (every far tile is
copied).  CPU only: the masks are a function of the cubes.

    python tools/ff_fractions.py [--workload vox10] [--sub-batch 64]
"""
import argparse
import json
import os
import sys

import numpy as np
from scipy import ndimage

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pcgcv1_b200 import synthetic  # noqa: E402

LAYERS = ["X0 conv_in", "T1a K_a", "X1 K_b", "T1b K_a", "X2 K_b", "T1c K_a", "X3 K_b"]


def near_masks(cubes):
    """[B,64,64,64,1] -> [7][B, z 64, y tile 2, x tile 8] bool."""
    occ = cubes[..., 0] != 0
    out = []
    for r in range(1, 8):
        d = ndimage.maximum_filter(occ, size=(1, 2 * r + 1, 2 * r + 1, 2 * r + 1), mode="constant", cval=0)
        out.append(d.reshape(len(cubes), 64, 2, 32, 8, 8).any(axis=(3, 5)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="vox10")
    ap.add_argument("--sub-batch", type=int, default=64)
    args = ap.parse_args()
    cubes, _, _ = synthetic.workload(args.workload, seed=0)
    sb = args.sub_batch
    masks = near_masks(cubes)
    chunks = [(a, min(a + sb, len(cubes))) for a in range(0, len(cubes), sb)]
    rows = {}
    for L, name in enumerate(LAYERS):
        m = masks[L]
        # steady state: slot s last held cube (previous chunk's start + s); the previous chunk of chunk 0 is the last chunk
        prev = np.ones((sb,) + m.shape[1:], bool)
        for a, b in chunks:                                       # one warm-up step
            prev[: b - a] = m[a:b]
        near = restore = total = seg_comp = segs = 0
        for a, b in chunks:
            cur, old = m[a:b], (prev[: b - a] if L < 6 else np.zeros_like(m[a:b]))
            near += cur.sum()
            restore += (~cur & old).sum()
            total += cur.size
            live = (cur | old).reshape(b - a, 4, 16, 2, 8).any(axis=2)   # 16-slice segments
            seg_comp += live.sum()
            segs += live.size
            prev[: b - a] = cur
        rows[name] = {"compute": round(near / total, 4), "restore": round(restore / total, 4),
                      "skip": round(1 - (near + restore) / total, 4)}
        if L in (1, 3, 5):
            rows[name]["segments_computed"] = round(seg_comp / segs, 4)
    print(json.dumps({"workload": args.workload, "cubes": len(cubes), "sub_batch": sb, "layers": rows}, indent=1))


if __name__ == "__main__":
    main()
