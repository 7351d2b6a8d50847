"""The material-atlas layout (oracle/bake.py, restated from csrc/bake.cu): texel ownership, bilinear footprints,
texel barycentrics and the cell placement of `bake.atlas_layout`.  CPU only."""
import numpy as np
import pytest

from oracle import bake as ob
from rise_sdf_b200.bake import atlas_layout

CELLS = range(4, 13)


def _uv_corners(C, b):
    return np.array(ob.corners(C, b), np.float64)


def _closest_on_triangle(q, P):
    """fp64 closest point to q on the (closed) triangle P [3, 2], as barycentrics"""
    A = np.array([P[1] - P[0], P[2] - P[0]]).T
    lam = np.linalg.solve(A, q - P[0])
    bary = np.array([1 - lam.sum(), lam[0], lam[1]])
    if (bary >= -1e-12).all():
        return bary
    best, bb = np.inf, None
    for a, b in ((0, 1), (1, 2), (2, 0)):
        d = P[b] - P[a]
        u = np.clip(np.dot(q - P[a], d) / np.dot(d, d), 0.0, 1.0)
        p = P[a] + u * d
        dist = np.linalg.norm(q - p)
        if dist < best - 1e-12:
            best, bb = dist, np.zeros(3)
            bb[a], bb[b] = 1 - u, u
    return bb


@pytest.mark.parametrize("C", CELLS)
def test_ownership_partitions_the_cell(C):
    j, i = np.meshgrid(np.arange(C), np.arange(C), indexing="ij")
    own = ob.owner(C, i, j)
    a, b = own == 0, own == 1
    assert (a ^ b).all()
    assert a.sum() == C * (C - 1) // 2 and b.sum() == C * (C + 1) // 2
    for side in (0, 1):
        for x, y in ob.corners(C, side):
            assert 0 <= x < C and 0 <= y < C and ob.owner(C, x, y) == side


@pytest.mark.parametrize("C", CELLS)
def test_bilinear_footprint_stays_on_owned_texels(C):
    rng = np.random.default_rng(C)
    for side in (0, 1):
        P = _uv_corners(C, side)
        w = -np.log(rng.random((4000, 3)))
        w /= w.sum(1, keepdims=True)
        w = np.concatenate([w, np.eye(3), [[.5, .5, 0], [0, .5, .5], [.5, 0, .5]]])
        for x, y in w @ P:
            fx, fy = np.floor(x), np.floor(y)
            rx, ry = x - fx, y - fy
            for di, wx in ((0, 1 - rx), (1, rx)):
                for dj, wy in ((0, 1 - ry), (1, ry)):
                    if wx * wy > 0:
                        ti, tj = int(fx) + di, int(fy) + dj
                        assert 0 <= ti < C and 0 <= tj < C, (side, x, y)
                        assert ob.owner(C, ti, tj) == side, (side, x, y, ti, tj)


@pytest.mark.parametrize("C", CELLS)
def test_texel_barycentrics(C):
    j, i = np.meshgrid(np.arange(C), np.arange(C), indexing="ij")
    i, j = i.ravel(), j.ravel()
    own = ob.owner(C, i, j)
    for side in (0, 1):
        P = _uv_corners(C, side)
        m = own == side
        b0, b1, b2 = ob.barycentrics(C, side, i[m], j[m])
        got = np.stack([b0, b1, b2], 1).astype(np.float64)
        assert got.dtype == np.float64 and b0.dtype == np.float32
        for k, (x, y) in enumerate(ob.corners(C, side)):               # corners: one-hot, exactly
            r = np.nonzero((i[m] == x) & (j[m] == y))[0][0]
            assert np.array_equal(got[r], np.eye(3)[k])
        for r, (x, y) in enumerate(zip(i[m], j[m])):
            want = _closest_on_triangle(np.array([x, y], np.float64), P)   # the centre inside, nearest point outside
            assert np.abs(got[r] - want).max() <= 1e-6, (side, x, y, got[r], want)
            assert np.all(got[r] >= -1e-6) and abs(got[r].sum() - 1) <= 1e-6     # b0 = 1 - s - t rounds


@pytest.mark.parametrize("C", CELLS)
def test_atlas_texels_and_uvs(C):
    """An odd face count with a partial last row of cells and unused columns: every face owns its share of its cell,
    corner UVs land on texels of their face whose points are the vertices, and bilinear samples anywhere inside a
    face's UV triangle read only that face's texels."""
    rng = np.random.default_rng(100 + C)
    F, cols = 41, 5
    T = cols * C + 2
    assert ob.layout(F, T) == (C, cols) == atlas_layout(F, T)
    v = rng.standard_normal((30, 3)).astype(np.float32)
    f = rng.integers(0, 30, (F, 3))
    face, pts = ob.texels(v, f, T, 0, T)
    face, pts = face.reshape(T, T), pts.reshape(T, T, 3)
    counts = np.bincount(face[face >= 0], minlength=F)
    assert (counts[0::2] == C * (C - 1) // 2).all() and (counts[1::2] == C * (C + 1) // 2).all()
    assert (face[:, cols * C:] == -1).all() and (face[-((T - 5 * C) or 1):, :] == -1).all()
    assert (pts[face < 0] == 0).all()
    uv = ob.uv(F, T)
    tex = uv.astype(np.float64) * T - 0.5                     # texel-centre coordinates of the corners
    assert np.abs(tex - np.round(tex)).max() <= 1e-5 * T      # (exact when T is a power of two)
    tex = np.round(tex)
    for fi in range(F):
        for k in range(3):
            ti, tj = int(tex[fi, k, 0]), int(tex[fi, k, 1])
            assert face[tj, ti] == fi
            assert np.array_equal(pts[tj, ti], v[f[fi, k]])
        w = -np.log(rng.random((200, 3)))
        w /= w.sum(1, keepdims=True)
        for x, y in w @ tex[fi]:
            fx, fy = int(np.floor(x)), int(np.floor(y))
            rx, ry = x - fx, y - fy
            for di, wx in ((0, 1 - rx), (1, rx)):
                for dj, wy in ((0, 1 - ry), (1, ry)):
                    if wx * wy > 0:
                        assert face[fy + dj, fx + di] == fi
    # bands: any split of the rows gives the same texels
    for n in (1, C + 1, 7):
        parts = [ob.texels(v, f, T, r0, min(n, T - r0)) for r0 in range(0, T, n)]
        assert np.array_equal(np.concatenate([p[0] for p in parts]), face.ravel())
        assert np.array_equal(np.concatenate([p[1] for p in parts]), pts.reshape(-1, 3))


def test_atlas_layout():
    assert atlas_layout(0, 16) == (16, 1)
    assert atlas_layout(1, 16) == (16, 1) and atlas_layout(2, 16) == (16, 1)
    assert atlas_layout(3, 16) == (8, 2)                          # P = 2 -> 2 columns
    assert atlas_layout(8, 64) == (32, 2) and atlas_layout(9, 64) == (21, 3)
    assert atlas_layout(2 * 1024 ** 2, 8192) == (8, 1024)
    assert atlas_layout(2 * 1024 ** 2 + 1, 8192) == (7, 1025)
    for F in range(0, 2000, 7):
        for T in (16, 100, 1024):
            P = (F + 1) // 2
            try:
                C, cols = atlas_layout(F, T)
            except ValueError:
                assert T // max(1, int(np.ceil(np.sqrt(P)))) < 4
                continue
            assert cols * cols >= P and (cols - 1) ** 2 < max(P, 1)
            assert C == T // cols >= 4 and (C, cols) == ob.layout(F, T)
    # the error names the smallest texture that fits, which does fit
    for F, T in ((2 * 1025 ** 2, 4096), (200, 16), (2 * 5000 ** 2, 16384)):
        cols = int(np.ceil(np.sqrt((F + 1) // 2)))
        with pytest.raises(ValueError, match=f"at least {4 * cols} texels"):
            atlas_layout(F, T)
        if 4 * cols <= 16384:
            assert atlas_layout(F, 4 * cols) == (4, cols)
    for T in (15, 16385):
        with pytest.raises(ValueError):
            atlas_layout(1, T)
