"""float32 numpy restatement of the normal-map kernels of rise_sdf_b200/csrc/bake.cu (`rsdf_bake_tangents`,
`rsdf_normal_pack`), with the same operation order, so that the kernels can be checked bit for bit, and a float64
`decode` that rebuilds the world-space normal from NORMAL, TANGENT and a texel the way a glTF viewer does.  Test-only."""
import numpy as np

from oracle import bake as ob

f32 = np.float32


def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], -1)


def _unit(v):
    """(v / |v|, ok); rows whose length is 0 or not finite are returned unchanged with ok False"""
    with np.errstate(all="ignore"):
        length = np.sqrt(_dot(v, v))
        ok = (length > 0) & np.isfinite(length)
        return np.where(ok[..., None], v / np.where(ok, length, f32(1.0))[..., None], v), ok


def _reject(v, n):
    """v - n (n . v)"""
    return v - n * _dot(n, v)[..., None]


def _bary(b, a):
    """(b0 a0 + b1 a1) + b2 a2 of b [n, 3] and a [n, 3 corners, 3]"""
    return (b[:, 0:1] * a[:, 0] + b[:, 1:2] * a[:, 1]) + b[:, 2:3] * a[:, 2]


def tangents(v_pos, t_pos_idx, v_nrm):
    """float32 [F, 3, 4] glTF TANGENTs per face corner (include/rsdf_b200.h, `rsdf_bake_tangents`)."""
    v_pos, v_nrm = np.asarray(v_pos, np.float32), np.asarray(v_nrm, np.float32)
    t_pos_idx = np.asarray(t_pos_idx, np.int64).reshape(-1, 3)
    F = len(t_pos_idx)
    p, n = v_pos[t_pos_idx], v_nrm[t_pos_idx]                 # [F, 3 corners, 3]
    e1, e2 = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
    u = np.where((np.arange(F) % 2 == 1)[:, None], -e1, e1)  # +u: e1 for A, -e1 for B
    w = np.where(_dot((n[:, 0] + n[:, 1]) + n[:, 2], _cross(e1, e2)) > 0, f32(-1.0), f32(1.0))
    uu = _dot(u, u)
    out = np.empty((F, 3, 4), np.float32)
    for k in range(3):
        nk, has_n = _unit(n[:, k])
        nk = np.where(has_n[:, None], nk, f32(0.0))
        t1 = _reject(u, nk)
        t = _reject(t1, nk)
        fallback = ~has_n | ~(_dot(t1, t1) > f32(1e-6) * uu)
        a = np.abs(nk)
        axis = np.where((a[:, 0] <= a[:, 1]) & (a[:, 0] <= a[:, 2]), 0, np.where(a[:, 1] <= a[:, 2], 1, 2))
        t = np.where(fallback[:, None], _reject(np.eye(3, dtype=np.float32)[axis], nk), t)
        out[:, k, :3] = _unit(t)[0]
        out[:, k, 3] = w
    return out


def texel_barycentrics(n_faces, T, row0, n_rows):
    """(face int64 [n_rows * T] (-1: unowned), barycentrics float32 [n_rows * T, 3]) of atlas rows
    [row0, row0 + n_rows), as `rsdf_bake_texels` computes them (oracle/bake.py `texels`)."""
    C, cols = ob.layout(n_faces, T)
    gj, gi = np.meshgrid(np.arange(row0, row0 + n_rows), np.arange(T), indexing="ij")
    gi, gj = gi.ravel(), gj.ravel()
    cc, cr = gi // C, gj // C
    x, y = gi - cc * C, gj - cr * C
    side = ob.owner(C, x, y)
    face = 2 * (cr * cols + cc) + side
    face = np.where((cc < cols) & (face < n_faces), face, -1)
    b = np.zeros((len(gi), 3), np.float32)
    for s in (0, 1):
        m = (face >= 0) & (side == s)
        b[m] = np.stack(ob.barycentrics(C, s, x[m], y[m]), -1)
    return face, b


def normal_pack(v_nrm, t_pos_idx, t_tangent, T, row0, n_rows, grad):
    """float32 [n_rows * T, 3] tangent-space normals of atlas rows [row0, row0 + n_rows) from the per-texel field
    gradient grad [n_rows * T, 3] (include/rsdf_b200.h, `rsdf_normal_pack`)."""
    v_nrm, t_tangent = np.asarray(v_nrm, np.float32), np.asarray(t_tangent, np.float32)
    t_pos_idx = np.asarray(t_pos_idx, np.int64).reshape(-1, 3)
    grad = np.asarray(grad, np.float32).reshape(-1, 3)
    face, b = texel_barycentrics(len(t_pos_idx), T, row0, n_rows)
    out = np.zeros((len(face), 3), np.float32)
    out[:, 2] = 1.0
    m = face >= 0
    fm, bm = face[m], b[m]
    with np.errstate(all="ignore"):                           # rows that fail are not written
        N, ok_n = _unit(_bary(bm, v_nrm[t_pos_idx[fm]]))
        g, ok_g = _unit(grad[m])
        tg = t_tangent[fm]
        Tp, ok_t = _unit(_reject(_bary(bm, tg[:, :, :3]), N))
        B = tg[:, 0, 3:4] * _cross(N, Tp)
        enc = np.stack([_dot(g, Tp), _dot(g, B), _dot(g, N)], -1)
    ok = ok_g & ok_n & ok_t
    out[np.flatnonzero(m)[ok]] = enc[ok]
    return out


def decode(nrm, tangent, b, enc):
    """float64 [n, 3] world-space unit normals a glTF viewer shades with: NORMAL nrm [n, 3 corners, 3] and TANGENT
    tangent [n, 3 corners, 4] interpolated with barycentrics b [n, 3], N = normalize(N), T = the tangent made orthogonal
    to N and normalised, B = w cross(N, T), and the texel enc [n, 3] (tangent-space, in [-1, 1]) mapped to
    normalize(x T + y B + z N)."""
    nrm, tangent, b, enc = (np.asarray(a, np.float64) for a in (nrm, tangent, b, enc))
    unit = lambda v: v / np.linalg.norm(v, axis=-1, keepdims=True)
    N = unit(np.einsum("nk,nkc->nc", b, nrm))
    t = np.einsum("nk,nkc->nc", b, tangent[:, :, :3])
    T = unit(t - N * np.sum(N * t, -1, keepdims=True))
    B = tangent[:, 0, 3:4] * np.cross(N, T)
    return unit(enc[:, 0:1] * T + enc[:, 1:2] * B + enc[:, 2:3] * N)
