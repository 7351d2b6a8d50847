"""Marching cubes on the device (csrc/mcubes.cu via rise_sdf_b200.mcubes), `VolumeSDF.isosurface`, `NeuSModel.export`
and the OBJ writer.  Exact agreement with the CPU reference mesher (oracle/mcubes.py) on noise fields; topology,
orientation and vertex placement on analytic fields; determinism, scratch memory and the single read-back at 512^3."""
import numpy as np
import pytest
import torch

from oracle import mcubes as omc
from rise_sdf_b200 import formats
from rise_sdf_b200.mcubes import marching_cubes
from test_oracle_mcubes import closed_and_oriented

gpu = pytest.mark.gpu


def analytic(kind, n):
    """(sdf float32 [n,n,n] over linspace(-1, 1, n)^3, outward gradient function of index-space points)."""
    g = np.linspace(-1.0, 1.0, n)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    to_world = lambda p: p * (2.0 / (n - 1)) - 1.0
    if kind == "sphere":
        sdf = np.sqrt(x * x + y * y + z * z) - 0.6
        grad = lambda p: to_world(p)
    else:                                                   # torus around z, R = 0.5, r = 0.2
        q = np.sqrt(x * x + y * y) - 0.5
        sdf = np.sqrt(q * q + z * z) - 0.2

        def grad(p):
            w = to_world(p)
            rho = np.sqrt(w[:, 0] ** 2 + w[:, 1] ** 2)
            return np.stack([w[:, 0] / rho * (rho - 0.5), w[:, 1] / rho * (rho - 0.5), w[:, 2]], -1)
    return sdf.astype(np.float32), grad


@gpu
@pytest.mark.parametrize("shape", [(48, 33, 2), (40, 40, 40), (2, 2, 2), (17, 5, 70)])
@pytest.mark.parametrize("negate", [False, True])
def test_matches_cpu_reference_exactly(shape, negate):
    f = np.random.default_rng(sum(shape) + negate).standard_normal(shape).astype(np.float32)
    iso = 0.25
    v_ref, f_ref = omc.marching_cubes(f, iso, negate=negate)
    v, fc = marching_cubes(torch.from_numpy(f).cuda(), iso, negate=negate)
    v, fc = v.cpu().numpy(), fc.cpu().numpy()
    assert v.dtype == np.float32 and fc.dtype == np.int64
    assert np.array_equal(fc, f_ref)
    assert v.shape == v_ref.shape and np.abs(v - v_ref).max(initial=0.0) <= 1e-6
    # each vertex sits at the fp64 linear crossing of its edge, up to the fp32 rounding of its coordinate
    val = (-f if negate else f).astype(np.float64)
    lin, axis = np.nonzero(omc.crossing_edges(val > np.float32(iso)).reshape(-1, 3))
    lo = np.stack(np.unravel_index(lin, shape), -1)
    hi = lo.copy()
    hi[np.arange(len(lin)), axis] += 1
    va, vb = val[tuple(lo.T)], val[tuple(hi.T)]
    exact = lo.astype(np.float64)
    exact[np.arange(len(lin)), axis] += (np.float32(iso) - va) / (vb - va)
    assert (np.abs(v - exact) <= 1e-6 + np.spacing(np.abs(v)) / 2).all()


@gpu
@pytest.mark.parametrize("n", [64, 128])
@pytest.mark.parametrize("kind,chi", [("sphere", 2), ("torus", 0)])
def test_analytic_fields(kind, chi, n):
    sdf, grad = analytic(kind, n)
    v, f = marching_cubes(torch.from_numpy(sdf).cuda(), 0.0, negate=True)
    v, f = v.cpu().numpy().astype(np.float64), f.cpu().numpy()
    ins = -sdf > 0
    n_cross = sum(int((ins.take(range(1, n), a) != ins.take(range(n - 1), a)).sum()) for a in range(3))
    assert len(v) == n_cross
    assert np.array_equal(np.unique(f), np.arange(len(v)))
    assert closed_and_oriented(f)
    assert len(v) - len(f) * 3 // 2 + len(f) == chi
    nrm = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    area2 = np.linalg.norm(nrm, axis=1)
    keep = area2 > 1e-6
    assert keep.mean() > 0.9
    dots = (nrm[keep] * grad(v[f[keep]].mean(1))).sum(1)
    assert (dots > 0).all()


@gpu
def test_edge_cases():
    dev = "cuda"
    for fill in (1.0, -1.0):                                # all inside, all outside
        v, f = marching_cubes(torch.full((9, 8, 7), fill, device=dev), 0.0)
        assert v.shape == (0, 3) and f.shape == (0, 3) and v.is_cuda and f.dtype == torch.int64
    # corners exactly at the isovalue: finite vertices (t in {0, 1} allowed), closed mesh
    g = np.random.default_rng(3).integers(-2, 3, (20, 21, 22)).astype(np.float32)
    g[0] = g[-1] = g[:, 0] = g[:, -1] = g[:, :, 0] = g[:, :, -1] = -1.0
    for iso in (0.0, 1.0):
        v, f = marching_cubes(torch.from_numpy(g).cuda(), iso)
        assert len(f) > 0 and bool(torch.isfinite(v).all()) and closed_and_oriented(f.cpu().numpy())
        vr, fr = omc.marching_cubes(g, iso)
        assert np.array_equal(f.cpu().numpy(), fr) and np.array_equal(v.cpu().numpy(), vr)
    # size guard: 3 * nx * ny * nz must fit int32 (1024 * 1024 * 683 does not; 512^3 does)
    big = torch.zeros(1, 1, 1, device=dev).expand(1024, 1024, 683)
    with pytest.raises(ValueError, match="grid edges"):
        marching_cubes(big, 0.0)
    with pytest.raises(ValueError):
        marching_cubes(torch.zeros(4, 4, device=dev), 0.0)


def test_cpu_tensor_raises():
    with pytest.raises(NotImplementedError, match="Only support cuda inputs."):
        marching_cubes(torch.zeros(4, 4, 4), 0.0)


@gpu
def test_512_determinism_memory_and_one_readback():
    g = torch.linspace(-1.0, 1.0, 512, device="cuda")
    x, y, z = torch.meshgrid(g, g, g, indexing="ij")
    vol = (x * x + y * y + z * z).sqrt_() - 0.6
    del g, x, y, z
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    v1, f1 = marching_cubes(vol, 0.0, negate=True)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base - v1.numel() * 4 - f1.numel() * 8
    assert extra <= 512 ** 3, extra
    v2, f2 = marching_cubes(vol, 0.0, negate=True)
    assert len(f1) > 100_000 and torch.equal(v1, v2) and torch.equal(f1, f2)
    assert closed_and_oriented(f1.cpu().numpy())
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        marching_cubes(vol, 0.0, negate=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    d2h = [n for n in names if "DtoH" in n or "Device -> Host" in n or "Device -> Pageable" in n]
    assert len(d2h) == 1, d2h
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        marching_cubes(vol, 0.0, negate=True)
    b.record()
    torch.cuda.synchronize()
    print(f"marching_cubes 512^3 sphere: {a.elapsed_time(b) / 10:.3f} ms per call, V={len(v1)}, F={len(f1)}, "
          f"scratch {extra / 2 ** 20:.1f} MiB")


@gpu
def test_isosurface_and_export_on_the_neus_model():
    from test_gpu_neus import build
    from rise_sdf_b200.geometry import MarchingCubeHelper
    m = build(table_scale=0.002).eval()
    geo = m.geometry
    res = 128
    mesh = geo.isosurface(res)
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    assert v.shape[0] > 1000 and f.dtype == torch.int64
    assert float(v.abs().max()) <= geo.radius
    # the fine grid is placed on the coarse mesh's bounds, padded by 10 % and clamped to the radius
    helper = MarchingCubeHelper(res)
    r = geo.radius
    coarse = helper(geo.isosurface_level(res), 0.0)["v_pos"] * (2 * r) - r
    lo, hi = coarse.amin(0), coarse.amax(0)
    bmin, bmax = (lo - (hi - lo) * 0.1).clamp(-r, r), (hi + (hi - lo) * 0.1).clamp(-r, r)
    fine = helper(geo.isosurface_level(res, bmin, bmax), 0.0)
    assert torch.equal(fine["t_pos_idx"], f) and torch.equal(fine["v_pos"] * (bmax - bmin) + bmin, v)
    assert bool((v >= bmin - 1e-6).all()) and bool((v <= bmax + 1e-6).all())
    # closed and oriented, except where the level set leaves the grid: this model's surface touches the y = -radius
    # face of the box, so the mesh is open there, and only there (every open edge lies on the fine grid's boundary)
    fn, vn = f.cpu().numpy(), v.cpu().numpy()
    a = np.concatenate([fn[:, 0], fn[:, 1], fn[:, 2]])
    b = np.concatenate([fn[:, 1], fn[:, 2], fn[:, 0]])
    key, rev = a * len(vn) + b, b * len(vn) + a
    assert np.unique(key).size == key.size
    open_ = ~np.isin(rev, key)
    eps = 1e-5 * r
    on_box = lambda i: ((np.abs(vn[i] - bmin.cpu().numpy()) <= eps) | (np.abs(vn[i] - bmax.cpu().numpy()) <= eps)).any(1)
    assert bool(on_box(a[open_]).all()) and bool(on_box(b[open_]).all())
    # with the grid's outer layer set outside, the same level grid meshes to a closed, oriented surface
    level = geo.isosurface_level(res, bmin, bmax).clone()
    for d in range(3):
        level.select(d, 0).fill_(1.0)
        level.select(d, res - 1).fill_(1.0)
    assert closed_and_oriented(helper(level, 0.0)["t_pos_idx"].cpu().numpy())
    # vertices lie on the level set to within one fine cell
    cell = float(((bmax - bmin) / (res - 1)).max())
    sdf = geo.forward_level(v)
    _, g, _ = geo(v, with_grad=True, with_feature=True)
    assert float(sdf.abs().max()) <= cell * float(g.norm(dim=-1).max())
    # export: vertex colours = texture(feature, -normal, normal) at the vertices
    out = m.export(chunk_size=5000, resolution=res)
    assert torch.equal(out["v_pos"], v) and torch.equal(out["t_pos_idx"], f)
    rgb = out["v_rgb"]
    assert rgb.shape == v.shape and float(rgb.min()) >= 0.0 and float(rgb.max()) <= 1.0
    idx = torch.arange(0, v.shape[0], 7, device=v.device)[:3000]
    _, g, feat = geo(v[idx], with_grad=True, with_feature=True)
    nrm = torch.nn.functional.normalize(g, p=2, dim=-1)
    with torch.no_grad():
        want = m.texture(feat, -nrm, nrm)
    assert float((rgb[idx] - want).abs().max()) <= 1e-5


def test_save_mesh_obj_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    v = rng.standard_normal((50, 3)).astype(np.float32)
    f = rng.integers(0, 50, (80, 3))
    c = rng.random((50, 3)).astype(np.float32)
    for rgb in (None, c):
        path = formats.save_mesh_obj(str(tmp_path / "m.obj"), torch.from_numpy(v), torch.from_numpy(f), None
                                     if rgb is None else torch.from_numpy(rgb))
        vs, fs = [], []
        for line in open(path):
            tok = line.split()
            if tok[0] == "v":
                vs.append([float(t) for t in tok[1:]])
            elif tok[0] == "f":
                fs.append([int(t) - 1 for t in tok[1:]])
        vs, fs = np.array(vs), np.array(fs)
        assert np.array_equal(fs, f)
        assert vs.shape == (50, 3 if rgb is None else 6)
        assert np.array_equal(vs[:, :3].astype(np.float32), v)
        if rgb is not None:
            assert np.array_equal(vs[:, 3:].astype(np.float32), rgb)
    formats.save_mesh_obj(str(tmp_path / "e.obj"), torch.zeros(0, 3), torch.zeros(0, 3, dtype=torch.int64))
    assert open(tmp_path / "e.obj").read() == ""
