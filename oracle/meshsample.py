"""NumPy restatement of pcgc_mesh_sample (include/pcgc_b200.h): face weights, Philox draws, barycentric samples, rotation, grid and
deduplication, in the same float64 operations and order (test infrastructure only).

Every step is elementwise IEEE arithmetic (+, -, *, sqrt, floor, ldexp, frexp, rint, one division), so the device, built without
FMA contraction, gives the same bits."""
from __future__ import annotations

import numpy as np

from .entropy import philox4x32_10

_M32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def icosphere(level: int):
    """Unit icosphere with 20 * 4^level faces (vertices on the sphere, shared along edges)."""
    t = (1.0 + 5.0 ** 0.5) / 2.0
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], np.float64)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6],
                  [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10], [8, 6, 7],
                  [9, 8, 1]], np.int64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    for _ in range(level):
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
        key = np.minimum(e[:, 0], e[:, 1]) * len(v) + np.maximum(e[:, 0], e[:, 1])
        uk, inv = np.unique(key, return_inverse=True)
        a, b = uk // len(v), uk % len(v)
        mid = v[a] + v[b]
        mid /= np.linalg.norm(mid, axis=1, keepdims=True)
        m = len(v) + inv.reshape(3, -1)
        v = np.concatenate([v, mid])
        f = np.concatenate([np.stack([f[:, 0], m[0], m[2]], 1), np.stack([f[:, 1], m[1], m[0]], 1),
                            np.stack([f[:, 2], m[2], m[1]], 1), np.stack([m[0], m[1], m[2]], 1)])
    return v, f.astype(np.int32)


def face_weights(verts: np.ndarray, tris: np.ndarray):
    """-> (a2 float64 [F], w uint64 [F], P uint64 [F+1] exclusive prefix sum, P[F] = W)."""
    verts = np.asarray(verts, np.float64)
    tris = np.asarray(tris, np.int64)
    A, B, C = verts[tris[:, 0]], verts[tris[:, 1]], verts[tris[:, 2]]
    e1, e2 = B - A, C - A
    cx = e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1]
    cy = e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2]
    cz = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
    a2 = np.sqrt((cx * cx + cy * cy) + cz * cz)
    _, e = np.frexp(a2.max())
    w = np.floor(np.ldexp(a2, 32 - int(e))).astype(np.uint64)
    P = np.zeros(len(w) + 1, np.uint64)
    np.cumsum(w, out=P[1:])
    return a2, w, P


def mulhi64(a: np.ndarray, b: int) -> np.ndarray:
    """High 64 bits of the 128-bit product a * b (uint64 arrays), in 32-bit halves."""
    a = np.asarray(a, np.uint64)
    b = np.uint64(b)
    a_lo, a_hi = a & _M32, a >> _S32
    b_lo, b_hi = b & _M32, b >> _S32
    lo_lo = a_lo * b_lo
    hi_lo = a_hi * b_lo
    lo_hi = a_lo * b_hi
    hi_hi = a_hi * b_hi
    cross = (lo_lo >> _S32) + (hi_lo & _M32) + lo_hi          # <= (2^32 - 1)^2 + 2 (2^32 - 1) = 2^64 - 1: no overflow
    return hi_hi + (hi_lo >> _S32) + (cross >> _S32)


def draw(P: np.ndarray, n: int, seed: int, j0: int = 0):
    """Samples j0 .. j0+n-1 -> (face int64 [n], u1 float64 [n], u2 float64 [n])."""
    j = np.arange(j0, j0 + n, dtype=np.uint64)
    r0, r1, r2, r3 = philox4x32_10(j & _M32, j >> _S32, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    t = (r1.astype(np.uint64) << _S32) | r0.astype(np.uint64)
    W = int(P[-1])
    target = mulhi64(t, W)
    face = np.searchsorted(P[:-1], target, side="right") - 1
    u1 = (r2.astype(np.float64) + 0.5) * 2.0 ** -32
    u2 = (r3.astype(np.float64) + 0.5) * 2.0 ** -32
    return face, u1, u2


def rotate(R: np.ndarray, p: np.ndarray) -> np.ndarray:
    R = np.asarray(R, np.float64)
    return np.stack([(R[r, 0] * p[:, 0] + R[r, 1] * p[:, 1]) + R[r, 2] * p[:, 2] for r in range(3)], -1)


def sample_mesh(verts, tris, n: int, seed: int, resolution: int, rotation=None, chunk: int = 1 << 22):
    """-> (points int32 [m,3] distinct grid points in ascending key order, samples float64 [n,3] (rotated), faces int32 [n],
    keys int64 [n] in sample order)."""
    verts = np.asarray(verts, np.float64)
    tris = np.asarray(tris, np.int64)
    R = np.eye(3) if rotation is None else np.asarray(rotation, np.float64)
    _, _, P = face_weights(verts, tris)
    if int(P[-1]) == 0:
        raise ValueError("every face is degenerate")
    ref = np.unique(tris.reshape(-1))
    qv = rotate(R, verts[ref])
    lo, hi = qv.min(0), qv.max(0)
    E = (hi - lo).max()
    scale = np.float64(resolution - 1) / E
    samples = np.empty((n, 3), np.float64)
    faces = np.empty(n, np.int32)
    keys = np.empty(n, np.int64)
    for j0 in range(0, n, chunk):
        m = min(chunk, n - j0)
        f, u1, u2 = draw(P, m, seed, j0)
        s = np.sqrt(u1)
        a, b, c = 1.0 - s, s * (1.0 - u2), s * u2
        A, B, C = verts[tris[f, 0]], verts[tris[f, 1]], verts[tris[f, 2]]
        p = (a[:, None] * A + b[:, None] * B) + c[:, None] * C
        q = rotate(R, p)
        g = np.clip(np.rint((q - lo) * scale), 0, resolution - 1).astype(np.int64)
        keys[j0:j0 + m] = (g[:, 0] * resolution + g[:, 1]) * resolution + g[:, 2]
        samples[j0:j0 + m] = q
        faces[j0:j0 + m] = f
    u = np.unique(keys)
    points = np.stack([u // (resolution * resolution), (u // resolution) % resolution, u % resolution], -1).astype(np.int32)
    return points, samples, faces, keys
