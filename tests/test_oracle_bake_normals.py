"""The normal-map restatement in oracle/bake_normals.py (what csrc/bake.cu's `rsdf_bake_tangents` / `rsdf_normal_pack`
are checked against on the GPU): tangent frames, the glTF normal-texture convention (+X along +u, +Y image-up) on
both triangles of a cell, encode / decode round trips and the documented fallbacks.  CPU only."""
import numpy as np
import pytest

from oracle import bake as ob
from oracle import bake_normals as obn

f32 = np.float32


def _random_mesh(rng, V=60, F=91):
    v = (rng.standard_normal((V, 3)) * 2).astype(np.float32)
    f = rng.integers(0, V, (F, 3))
    n = rng.standard_normal((V, 3)).astype(np.float32)
    return v, f, (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32)


def test_tangents_are_unit_orthogonal_and_signed():
    v, f, n = _random_mesh(np.random.default_rng(0))
    t = obn.tangents(v, f, n)
    assert t.shape == (len(f), 3, 4) and t.dtype == np.float32
    assert np.abs(np.linalg.norm(t[..., :3].astype(np.float64), axis=-1) - 1).max() < 1e-6
    assert np.abs(np.sum(t[..., :3].astype(np.float64) * n[f], -1)).max() < 1e-6
    assert set(np.unique(t[..., 3])) <= {-1.0, 1.0}
    assert np.all(t[:, :, 3] == t[:, :1, 3])                    # one w per face


def _planar_pair(rng):
    """two random triangles in the plane z = c (A = face 0, B = face 1), vertex normals +z, agreeing with the winding"""
    while True:
        p = np.concatenate([rng.uniform(-1, 1, (6, 2)), np.full((6, 1), 0.25)], 1).astype(np.float32)
        f = np.arange(6).reshape(2, 3)
        cz = [np.cross(p[a[1]] - p[a[0]], p[a[2]] - p[a[0]])[2] for a in f]
        if min(abs(c) for c in cz) > 0.05:
            break
    for i, c in enumerate(cz):
        if c < 0:
            f[i, 1], f[i, 2] = f[i, 2], f[i, 1]
    n = np.tile(np.array([0.0, 0.0, 1.0], np.float32), (6, 1))
    return p, f, n


def _owned(face, k):
    return np.flatnonzero(face == k)


@pytest.mark.parametrize("seed", range(4))
def test_normal_texture_convention_on_both_triangles(seed):
    rng = np.random.default_rng(seed)
    p, f, n = _planar_pair(rng)
    T = 32
    t = obn.tangents(p, f, n)
    assert np.all(t[..., 3] == -1.0)
    face, b = obn.texel_barycentrics(2, T, 0, T)
    face_ref, pts = ob.texels(p, f, T, 0, T)
    assert np.array_equal(face, face_ref)
    tilt = lambda d: np.tile(np.array(d, np.float32), (T * T, 1))
    for k in (0, 1):
        own = _owned(face, k)
        # the surface point moves along +T one texel to the right and along +B one texel up (texels inside the
        # triangle: A's run to x + y = C - 3, B's from x + y = C; the row between is the dilation)
        C = ob.layout(2, T)[0]
        x, y = own % T, own // T
        ins = np.zeros((T, T), bool)
        keep = (x + y <= C - 3) if k == 0 else (x + y >= C)
        ins[y[keep], x[keep]] = True
        grid = pts.reshape(T, T, 3)
        tk = t[k, 0, :3]
        bk = t[k, 0, 3] * np.cross(n[0], tk)
        d_right = (grid[:, 1:] - grid[:, :-1])[ins[:, 1:] & ins[:, :-1]]
        d_up = (grid[:-1] - grid[1:])[ins[:-1] & ins[1:]]
        assert len(d_right) > 10 and len(d_up) > 10
        assert np.all(d_right @ tk > 0) and np.all(d_up @ bk > 0)
        assert np.abs(d_right @ bk).max() < 1e-5                # (image-up is -e2 or e2, not orthogonal to T)
        # a gradient tilted towards +u encodes red > 0.5, one tilted image-up green > 0.5, one along N flat
        e1, e2 = p[f[k, 1]] - p[f[k, 0]], p[f[k, 2]] - p[f[k, 0]]
        u, imgup = (e1, -e2) if k == 0 else (-e1, e2)
        u, imgup = u / np.linalg.norm(u), imgup / np.linalg.norm(imgup)
        for d, ch in ((u, 0), (imgup, 1)):
            enc = obn.normal_pack(n, f, t, T, 0, T, tilt(0.4 * d + np.array([0, 0, 1])))[own]
            assert np.all(0.5 * enc[:, ch] + 0.5 > 0.5)
        enc = obn.normal_pack(n, f, t, T, 0, T, tilt([0, 0, 3.0]))[own]
        assert np.array_equal(enc, np.tile(np.array([0, 0, 1], np.float32), (len(own), 1)))


def test_encode_decode_round_trip():
    rng = np.random.default_rng(1)
    v, f, n = _random_mesh(rng)
    t = obn.tangents(v, f, n)
    T = 64
    face, b = obn.texel_barycentrics(len(f), T, 0, T)
    g = rng.standard_normal((T * T, 3)).astype(np.float32) * 5
    enc = obn.normal_pack(n, f, t, T, 0, T, g)
    m = face >= 0
    assert np.abs(np.linalg.norm(enc.astype(np.float64), axis=1) - 1).max() < 1e-6
    assert np.all(enc[~m] == np.array([0, 0, 1], np.float32))
    dec = obn.decode(n[f[face[m]]], t[face[m]], b[m], enc[m])
    want = g[m] / np.linalg.norm(g[m].astype(np.float64), axis=1, keepdims=True)
    assert np.abs(dec - want).max() < 1e-5


def test_fallbacks():
    p = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 0, 1], [2, 0, 0]], np.float32)
    n = np.array([[0, 0, 1], [0, 0, 0], [1, 0, 0], [0, 0.6, 0.8], [0, 0, 1], [0, 0, 1]], np.float32)
    # face 0 (A): corner 1 has a zero normal; corner 2 has a normal parallel to +u = e1
    # face 1 (B): e1 = 0 (p3 == p4)
    f = np.array([[0, 1, 2], [3, 4, 5]])
    t = obn.tangents(p, f, n)
    assert np.array_equal(t[0, 0], np.array([1, 0, 0, -1], np.float32))   # ordinary corner: e1, w from the winding
    assert np.array_equal(t[0, 1], np.array([1, 0, 0, -1], np.float32))   # zero normal: the x axis
    assert np.array_equal(t[0, 2], np.array([0, 1, 0, -1], np.float32))   # parallel: least aligned axis y
    assert np.all(t[1, :, 3] == 1.0)                                       # zero cross(e1, e2): w = +1
    assert np.array_equal(t[1, 0, :3], np.array([1, 0, 0], np.float32))   # |n_x| smallest: x axis
    want = np.array([1, 0, 0], np.float32)
    assert np.array_equal(t[1, 2, :3], want) and np.array_equal(t[1, 1, :3], want)
    # normal_pack: zero or non-finite gradient, zero interpolated normal, unowned texels -> (0, 0, 1)
    T = 16
    face, _ = obn.texel_barycentrics(2, T, 0, T)
    flat = np.array([0, 0, 1], np.float32)
    for bad in (0.0, np.nan, np.inf):
        enc = obn.normal_pack(n, f, t, T, 0, T, np.full((T * T, 3), bad, np.float32))
        assert np.all(enc == flat)
    g = np.tile(np.array([0.3, 0.2, 1.0], np.float32), (T * T, 1))
    nz = np.zeros_like(n)
    assert np.all(obn.normal_pack(nz, f, t, T, 0, T, g) == flat)
    enc = obn.normal_pack(n, f, t, T, 0, T, g)
    assert np.all(enc[face < 0] == flat) and not np.all(enc[face == 0] == flat)
    # a tangent along the interpolated normal (T' = 0): flat
    tz = t.copy()
    tz[:, :, :3] = np.array([0, 0, 1], np.float32)
    enc = obn.normal_pack(np.tile(np.array([0, 0, 1], np.float32), (6, 1)), f, tz, T, 0, T, g)
    assert np.all(enc == flat)
