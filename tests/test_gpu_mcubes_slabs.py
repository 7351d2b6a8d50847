"""Streamed marching cubes (`mcubes.marching_cubes_slabs`, `rsdf_mc_slab_count` / `_emit`) and the streamed
`VolumeSDF.isosurface`.  Bit-identical to the dense mesher on noise fields for every slab size; topology, placement,
determinism, memory and read-backs on analytic fields above the dense mesher's 2^31 - 1 edge bound; the neus model's
isosurface and export at 1024^3.  The slab planner and argument checks run without a GPU."""
import numpy as np
import pytest
import torch

from rise_sdf_b200 import mcubes
from rise_sdf_b200.mcubes import marching_cubes, marching_cubes_slab_iter, marching_cubes_slabs, plan_slabs
from test_oracle_mcubes import closed_and_oriented

gpu = pytest.mark.gpu


def slicer(vol):
    return lambda x0, n: vol[x0:x0 + n]


def check_same(vol, iso, negate, slab_layers):
    v0, f0 = marching_cubes(vol, iso, negate=negate)
    v1, f1 = marching_cubes_slabs(slicer(vol), vol.shape, iso, negate=negate, slab_layers=slab_layers)
    assert v1.dtype == torch.float32 and f1.dtype == torch.int64
    assert torch.equal(v0, v1) and torch.equal(f0, f1), (tuple(vol.shape), slab_layers, negate)
    return v0, f0


# ------------------------------------------------------------------------------------------------ planner (CPU)
def test_plan_covers_the_volume_with_halos():
    for shape, layers in [((10, 4, 4), 3), ((10, 4, 4), 1), ((11, 4, 4), 3), ((2, 5, 5), 1), ((7, 3, 3), 7),
                          ((7, 3, 3), 100), ((3, 2, 2), 2)]:
        plan = plan_slabs(shape, layers)
        nx = shape[0]
        assert plan[0][0] == 0 and sum(own for _, own, _ in plan) == nx
        for (x0, own, p), nxt in zip(plan, plan[1:] + [None]):
            assert p >= 2 and 1 <= own <= p and p == min(own + 2, nx - x0)
            if nxt is not None:
                assert nxt[0] == x0 + own
                assert nx - nxt[0] >= 2                      # no one-layer slab
    assert plan_slabs((10, 4, 4), 3) == [(0, 3, 5), (3, 3, 5), (6, 4, 4)]    # a last lone layer is folded in
    assert plan_slabs((7, 3, 3), 100) == [(0, 7, 7)]
    assert plan_slabs((1, 5, 5)) == [] and plan_slabs((5, 0, 5)) == []


def test_plan_respects_the_int32_and_slab_byte_bounds(monkeypatch):
    syz = 2048 * 2048
    plan = plan_slabs((2048, 2048, 2048))
    assert len(plan) > 1
    assert all(3 * p * syz <= mcubes.MAX_EDGES for _, _, p in plan)
    assert max(own for _, own, _ in plan[:-1]) * syz * 4 <= mcubes.SLAB_BYTES
    # a slab size beyond the int32 bound is capped: own + 2 halo layers must fit
    plan = plan_slabs((4096, 2048, 2048), 10 ** 6)
    assert max(p for _, _, p in plan) == mcubes.MAX_EDGES // (3 * syz)
    monkeypatch.setattr(mcubes, "SLAB_BYTES", 5 * 4 * 64 * 64)
    assert [own for _, own, _ in plan_slabs((64, 64, 64))][:3] == [5, 5, 5]
    assert plan_slabs((512, 512, 512), None) != [(0, 512, 512)]
    monkeypatch.undo()
    assert plan_slabs((512, 512, 512)) == [(0, 512, 512)]                  # the 512^3 grid is one slab


def test_rejects_bad_shapes_and_slab_sizes():
    with pytest.raises(ValueError, match="too large"):
        plan_slabs((10, 30000, 30000))                      # 3 * 3 * ny * nz > 2^31 - 1
    plan_slabs((2, 16384, 16384))                           # within the dense bound: one slab of two layers
    for bad in [(4, 4), (4, 4, -1), (4.0, 4, 4), "abc"]:
        with pytest.raises(ValueError, match="shape"):
            plan_slabs(bad)
    with pytest.raises(ValueError, match="2\\^24|exceeds"):
        plan_slabs(((1 << 24) + 1, 2, 2))
    with pytest.raises(ValueError, match="positive"):
        plan_slabs((8, 8, 8), 0)


def test_cpu_layers_raise():
    with pytest.raises(ValueError, match="CUDA float32"):
        marching_cubes_slabs(lambda x0, n: torch.zeros(n, 4, 4), (8, 4, 4), 0.0)


# ------------------------------------------------------------------------------------------------ slab == dense
@gpu
@pytest.mark.parametrize("shape", [(23, 17, 13), (40, 33, 70), (2, 9, 11), (26, 64, 32)])
@pytest.mark.parametrize("negate", [False, True])
def test_slabs_equal_dense_on_noise(shape, negate):
    vol = torch.from_numpy(np.random.default_rng(sum(shape) + negate).standard_normal(shape).astype(np.float32))
    vol = vol.cuda()
    for slab_layers in (1, 2, 3, 5, shape[0]):
        v, f = check_same(vol, 0.25, negate, slab_layers)
        assert len(f) > 0
    # each slab's vertices lie in its own layers, and its faces use its vertices or the next slab's first layer's
    plan = plan_slabs(shape, 3)
    start = 0
    for (x0, own, p), (vs, fs) in zip(plan, marching_cubes_slab_iter(slicer(vol), shape, 0.25, negate, 3)):
        if len(vs):
            assert float(vs[:, 0].min()) >= x0 and float(vs[:, 0].max()) <= x0 + own
        if len(fs):
            assert int(fs.min()) >= start
        start += len(vs)
    assert start == len(v)


@gpu
def test_slabs_equal_dense_at_the_isovalue_and_when_empty():
    # integer field: many corners exactly at iso = 0 or 1, on every layer, so on every slab boundary
    g = torch.from_numpy(np.random.default_rng(3).integers(-2, 3, (20, 21, 22)).astype(np.float32)).cuda()
    for iso in (0.0, 1.0):
        for negate in (False, True):
            for slab_layers in (1, 2, 3, 5, 20):
                v, f = check_same(g, iso, negate, slab_layers)
                assert len(f) > 0 and bool(torch.isfinite(v).all())
    for fill in (1.0, -1.0):                                 # all inside, all outside
        vol = torch.full((9, 8, 7), fill, device="cuda")
        for slab_layers in (1, 3, 9):
            v, f = check_same(vol, 0.0, False, slab_layers)
            assert v.shape == (0, 3) and f.shape == (0, 3)


@gpu
def test_layer_outputs_are_validated():
    vol = torch.randn(8, 6, 5, device="cuda")
    cases = [(lambda x0, n: vol[x0:x0 + n].double(), "CUDA float32"),
             (lambda x0, n: vol[x0:x0 + n, :5], "shape"),
             (lambda x0, n: vol.transpose(1, 2).contiguous().transpose(1, 2)[x0:x0 + n], "contiguous"),
             (lambda x0, n: vol[x0:x0 + n].cpu(), "CUDA float32")]
    for fn, msg in cases:
        with pytest.raises(ValueError, match=msg):
            marching_cubes_slabs(fn, vol.shape, 0.0, slab_layers=3)


# ------------------------------------------------------------------------------------------------ above the old bound
def analytic_layers(kind, n, buf):
    """layers(x0, k) of the sdf of a sphere (radius 0.6) or a torus around z (R = 0.5, r = 0.2) over
    linspace(-1, 1, n)^3, computed into the head of `buf`: no full grid, no full-slab temporaries."""
    g = torch.linspace(-1.0, 1.0, n, device="cuda")

    def layers(x0, k):
        x, y, z = g[x0:x0 + k].view(k, 1, 1), g.view(1, n, 1), g.view(1, 1, n)
        out = buf[:k * n * n].view(k, n, n)
        if kind == "sphere":
            torch.add(x * x + y * y, z * z, out=out)
            return out.sqrt_().sub_(0.6)
        q = (x * x + y * y).sqrt_().sub_(0.5)
        torch.add(q * q, z * z, out=out)
        return out.sqrt_().sub_(0.2)
    return layers


def analytic_sdf(kind, w):
    if kind == "sphere":
        return w.norm(dim=-1) - 0.6
    q = w[:, :2].norm(dim=-1) - 0.5
    return torch.stack([q, w[:, 2]], -1).norm(dim=-1) - 0.2


def crossings(layers, shape):
    """Crossing edges (inside: -sdf > 0) owned by each slab's layers, counted slab by slab."""
    total = 0
    for x0, own, p in plan_slabs(shape):
        ins = layers(x0, p) < 0
        m = min(own, p - 1)
        total += int((ins[:m] != ins[1:m + 1]).sum())
        total += int((ins[:own, :-1] != ins[:own, 1:]).sum()) + int((ins[:own, :, :-1] != ins[:own, :, 1:]).sum())
    return total


def slab_buffer(shape):
    return torch.empty(max(p for _, _, p in plan_slabs(shape)) * shape[1] * shape[2], device="cuda")


@gpu
@pytest.mark.parametrize("kind,n,chi", [("sphere", 1024, 2), ("torus", 1024, 0), ("sphere", 2048, 2)])
def test_analytic_fields_above_the_dense_bound(kind, n, chi):
    shape = (n, n, n)
    assert 3 * n ** 3 > mcubes.MAX_EDGES and len(plan_slabs(shape)) > 1
    layers = analytic_layers(kind, n, slab_buffer(shape))
    v, f = marching_cubes_slabs(layers, shape, 0.0, negate=True)
    nv, nf = v.shape[0], f.shape[0]
    assert nv == crossings(layers, shape)
    assert int(f.min()) == 0 and int(f.max()) == nv - 1
    assert bool((torch.bincount(f.view(-1), minlength=nv) > 0).all())
    assert nf % 2 == 0 and nv - nf * 3 // 2 + nf == chi
    cell = 2.0 / (n - 1)
    w = v.double() * cell - 1.0
    assert float(analytic_sdf(kind, w).abs().max()) <= cell
    if n == 1024:
        assert closed_and_oriented(f.cpu().numpy())
    else:
        v2, f2 = marching_cubes_slabs(layers, shape, 0.0, negate=True)
        assert torch.equal(v, v2) and torch.equal(f, f2)
    print(f"{kind} {n}^3: V={nv}, F={nf}, {len(plan_slabs(shape))} slabs")


@gpu
def test_2048_peak_memory_and_one_readback_per_slab():
    from torch.profiler import ProfilerActivity, profile
    n = 2048
    shape = (n, n, n)
    plan = plan_slabs(shape)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    buf = slab_buffer(shape)
    v, f = marching_cubes_slabs(analytic_layers("sphere", n, buf), shape, 0.0, negate=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    p_max = max(p for _, _, p in plan)
    out = v.numel() * 4 + f.numel() * 8
    bound = 4 * p_max * n * n + mcubes.scratch_bytes((p_max, n, n)) + 2 * out + (64 << 20)
    assert peak <= bound, (peak, bound)
    assert peak < n ** 3 * 4 // 8
    print(f"2048^3 sphere: {len(plan)} slabs, peak {peak / 2 ** 30:.2f} GiB (bound {bound / 2 ** 30:.2f} GiB)")
    del v, f, buf
    shape = (1024, 1024, 1024)
    layers = analytic_layers("sphere", 1024, slab_buffer(shape))
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        marching_cubes_slabs(layers, shape, 0.0, negate=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    d2h = [nm for nm in names if "DtoH" in nm or "Device -> Host" in nm or "Device -> Pageable" in nm]
    assert len(d2h) == len(plan_slabs(shape)) > 1, d2h


# ------------------------------------------------------------------------------------------------ the neus model
@gpu
def test_isosurface_level_layers_match_the_whole_grid():
    from test_gpu_neus import build
    geo = build(table_scale=0.002).eval().geometry
    whole = geo.isosurface_level(48)
    lo = torch.tensor([-1.0, -0.5, -1.2], device="cuda")
    hi = torch.tensor([1.1, 0.7, 0.4], device="cuda")
    part_whole = geo.isosurface_level(48, lo, hi)
    for x0, n in [(0, 48), (0, 1), (10, 7), (47, 1)]:
        assert torch.equal(geo.isosurface_level(48, x0=x0, n_layers=n), whole[x0:x0 + n])
        assert torch.equal(geo.isosurface_level(48, lo, hi, chunk=1000, x0=x0, n_layers=n), part_whole[x0:x0 + n])
    with pytest.raises(ValueError, match="outside"):
        geo.isosurface_level(48, x0=40, n_layers=9)


@gpu
def test_isosurface_with_small_slabs_equals_one_slab(monkeypatch):
    from test_gpu_neus import build
    geo = build(table_scale=0.002).eval().geometry
    one = geo.isosurface(256)
    assert len(plan_slabs((256, 256, 256))) == 1 and one["v_pos"].shape[0] > 1000
    monkeypatch.setattr(mcubes, "SLAB_BYTES", 7 * 4 * 256 * 256)
    assert len(plan_slabs((256, 256, 256))) > 30
    many = geo.isosurface(256)
    assert torch.equal(one["v_pos"], many["v_pos"]) and torch.equal(one["t_pos_idx"], many["t_pos_idx"])


@gpu
def test_isosurface_and_export_at_1024():
    from test_gpu_neus import build
    m = build(table_scale=0.002).eval()
    geo = m.geometry
    res = 1024
    mesh = geo.isosurface(res)
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    assert v.shape[0] > 10000 and f.dtype == torch.int64
    # the fine grid's bounds from the whole coarse mesh (models/geometry.py:104-110)
    r = geo.radius
    cv, _ = marching_cubes_slabs(lambda x0, n: geo.isosurface_level(res, x0=x0, n_layers=n), (res,) * 3, 0.0,
                                 negate=True)
    coarse = cv / (res - 1.0) * (2 * r) - r
    lo, hi = coarse.amin(0), coarse.amax(0)
    del cv, coarse
    bmin, bmax = (lo - (hi - lo) * 0.1).clamp(-r, r), (hi + (hi - lo) * 0.1).clamp(-r, r)
    assert bool((v >= bmin - 1e-6).all()) and bool((v <= bmax + 1e-6).all())
    # open edges only where the level set leaves the fine grid
    fn, vn = f.cpu().numpy(), v.cpu().numpy()
    a = np.concatenate([fn[:, 0], fn[:, 1], fn[:, 2]])
    b = np.concatenate([fn[:, 1], fn[:, 2], fn[:, 0]])
    key, rev = a * len(vn) + b, b * len(vn) + a
    assert np.unique(key).size == key.size
    open_ = ~np.isin(rev, key)
    eps = 1e-5 * r
    on_box = lambda i: ((np.abs(vn[i] - bmin.cpu().numpy()) <= eps) | (np.abs(vn[i] - bmax.cpu().numpy()) <= eps)).any(1)
    assert bool(on_box(a[open_]).all()) and bool(on_box(b[open_]).all())
    # vertices lie on the level set to within one fine cell
    cell = float(((bmax - bmin) / (res - 1)).max())
    for s in range(0, v.shape[0], 1 << 20):
        vs = v[s:s + (1 << 20)]
        sdf = geo.forward_level(vs)
        _, g, _ = geo(vs, with_grad=True, with_feature=True)
        assert float(sdf.abs().max()) <= cell * float(g.norm(dim=-1).max())
    out = m.export(resolution=res)
    assert torch.equal(out["v_pos"], v) and torch.equal(out["t_pos_idx"], f)
    assert out["v_rgb"].shape == v.shape and out["v_rgb"].dtype == torch.float32
    print(f"neus isosurface 1024^3: V={v.shape[0]}, F={f.shape[0]}")
