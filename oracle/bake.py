"""float32 numpy restatement of the material-atlas layout of rise_sdf_b200/csrc/bake.cu (`rsdf_bake_uv`,
`rsdf_bake_texels`), with the same operation order, so that the kernels can be checked bit for bit.  Test-only."""
import math

import numpy as np

f32 = np.float32


def layout(n_faces, T):
    """(C, cols): P = ceil(F / 2) cells, cols = ceil(sqrt(P)) (at least 1), C = T // cols."""
    P = (n_faces + 1) // 2
    cols = max(1, math.isqrt(P - 1) + 1 if P > 0 else 0)
    return T // cols, cols


def corners(C, b):
    """cell-local (x, y) of the three corners of triangle A (b = 0) or B (b = 1), in vertex order"""
    if b == 0:
        return [(0, 0), (C - 3, 0), (0, C - 3)]
    return [(C - 1, C - 1), (1, C - 1), (C - 1, 1)]


def owner(C, i, j):
    """0 (A) or 1 (B): which triangle of a cell owns cell-local texel (i, j)"""
    return np.where(np.asarray(i) + np.asarray(j) <= C - 2, 0, 1)


def barycentrics(C, b, x, y):
    """(b0, b1, b2) float32 of cell-local texel centres (x, y) owned by triangle b (arrays)."""
    x, y = np.asarray(x), np.asarray(y)
    if b == 0:
        L = f32(C - 3)
        s, t = x.astype(f32) / L, y.astype(f32) / L
    else:
        L = f32(C - 2)
        s, t = (C - 1 - x).astype(f32) / L, (C - 1 - y).astype(f32) / L
    e = s + t
    d = (e - f32(1.0)) * f32(0.5)
    over = e > f32(1.0)
    s = np.where(over, s - d, s).astype(f32)
    t = np.where(over, t - d, t).astype(f32)
    s = np.minimum(np.maximum(s, f32(0.0)), f32(1.0))
    t = np.minimum(np.maximum(t, f32(0.0)), f32(1.0))
    b0 = (f32(1.0) - s) - t
    return b0.astype(f32), s.astype(f32), t.astype(f32)


def uv(n_faces, T):
    """float32 [F, 3, 2] per-corner glTF UVs."""
    C, cols = layout(n_faces, T)
    out = np.zeros((n_faces, 3, 2), np.float32)
    for f in range(n_faces):
        p = f // 2
        col0, row0 = (p % cols) * C, (p // cols) * C
        for k, (x, y) in enumerate(corners(C, f & 1)):
            out[f, k, 0] = (f32(col0 + x) + f32(0.5)) / f32(T)
            out[f, k, 1] = (f32(row0 + y) + f32(0.5)) / f32(T)
    return out


def texels(v_pos, t_pos_idx, T, row0, n_rows):
    """(face_id int32 [n_rows * T], points float32 [n_rows * T, 3]) of atlas rows [row0, row0 + n_rows)."""
    v_pos = np.asarray(v_pos, np.float32)
    t_pos_idx = np.asarray(t_pos_idx, np.int64)
    F = len(t_pos_idx)
    C, cols = layout(F, T)
    gj, gi = np.meshgrid(np.arange(row0, row0 + n_rows), np.arange(T), indexing="ij")
    gi, gj = gi.ravel(), gj.ravel()
    cc, cr = gi // C, gj // C
    x, y = gi - cc * C, gj - cr * C
    b = owner(C, x, y)
    face = 2 * (cr * cols + cc) + b
    face = np.where((cc < cols) & (face < F), face, -1)
    pts = np.zeros((len(gi), 3), np.float32)
    for side in (0, 1):
        m = (face >= 0) & (b == side)
        b0, b1, b2 = barycentrics(C, side, x[m], y[m])
        tri = v_pos[t_pos_idx[face[m]]]                     # [n, 3 corners, 3]
        pts[m] = (b0[:, None] * tri[:, 0] + b1[:, None] * tri[:, 1]) + b2[:, None] * tri[:, 2]
    return face.astype(np.int32), pts
