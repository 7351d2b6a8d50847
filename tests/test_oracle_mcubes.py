"""The marching-cubes triangle table (face-walk rule) and the CPU reference mesher (CPU only)."""
import numpy as np
import pytest

from oracle import mcubes as M


def closed_and_oriented(faces):
    """Every directed edge of the triangle soup occurs exactly once and so does its reverse."""
    f = np.asarray(faces, np.int64)
    a = np.concatenate([f[:, 0], f[:, 1], f[:, 2]])
    b = np.concatenate([f[:, 1], f[:, 2], f[:, 0]])
    n = int(f.max()) + 1 if f.size else 1
    key, rev = a * n + b, b * n + a
    _, counts = np.unique(key, return_counts=True)
    return bool((counts == 1).all()) and bool(np.isin(rev, key).all())


def padded_noise(shape, seed):
    f = np.random.default_rng(seed).standard_normal(shape).astype(np.float32)
    f[0] = f[-1] = f[:, 0] = f[:, -1] = f[:, :, 0] = f[:, :, -1] = -1.0     # outside (value <= iso) all round
    return f


def test_committed_table_header_is_the_generator_output():
    with open(M.HEADER) as fh:
        assert fh.read() == M.header_text()


def test_table_size_and_bound():
    assert sum(1 for t in M.TABLE if t) == 254
    assert max(len(t) for t in M.TABLE) == 5
    assert not M.TABLE[0] and not M.TABLE[255]


@pytest.mark.parametrize("case", range(256))
def test_every_case_uses_exactly_its_crossing_edges(case):
    inside = [(case >> c) & 1 for c in range(8)]
    crossing = {e for e, (a, b) in enumerate(M.EDGES) if inside[a] != inside[b]}
    used = {e for t in M.TABLE[case] for e in t}
    assert used == crossing
    for t in M.TABLE[case]:
        assert len(set(t)) == 3


@pytest.mark.parametrize("seed", range(4))
def test_noise_meshes_are_closed_and_oriented(seed):
    v, f = M.marching_cubes(padded_noise((14, 14, 14), seed), 0.0)
    assert len(f) > 100 and closed_and_oriented(f)
    assert np.array_equal(np.unique(f), np.arange(len(v)))                 # every vertex is used


def test_sphere_is_a_closed_outward_genus_0_surface():
    g = np.linspace(-1.0, 1.0, 24)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    sdf = (np.sqrt(x * x + y * y + z * z) - 0.6).astype(np.float32)
    v, f = M.marching_cubes(sdf, 0.0, negate=True)
    assert closed_and_oriented(f)
    assert len(v) - len(f) * 3 // 2 + len(f) == 2
    n = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    c = v[f].mean(1) - 11.5
    assert ((n * c).sum(1) > 0).all()
    # `negate` reads -volume: the same mesh as meshing a negated copy
    v2, f2 = M.marching_cubes(-sdf, 0.0, negate=False)
    assert np.array_equal(v, v2) and np.array_equal(f, f2)
    # negating both the volume and the isovalue keeps the vertex bits (the inside flips, so the faces change)
    v3, f3 = M.marching_cubes(sdf, -0.0)
    assert np.array_equal(v3, v) and closed_and_oriented(f3)
