"""The hash-grid kernels of the training step, one by one, against float64, level by level.

The float64 reference picks exactly the kernel's cells: pos = fl32(fmaf(scale, x, 0.5)) and its floor are taken in
fp32 (as `oracle.fields.hash_encode` emulates), and the weights are rebuilt as `frac + scale * (x - x.detach())`, which
equals the kernel's fp32 weight bit for bit while giving exact first and second derivatives.  Everything after the
cell choice (weights, table, products, sums, derivatives) is float64, so no sample near a cell face has to be excluded.

Errors are measured per level and feature (a whole-table metric is set by the dense levels, whose entries collect
thousands of samples; a hashed entry collects one or two) as max|kernel - fp64| / max|fp64| of that level.  Each bound
is max(K x the same quantity for an fp32 twin of the reference, a floor), the methodology DESIGN.md §5 uses for the
FD-normal configs.  Measured on a B200, the worst level of every comparison sits at or below its fp32 twin; the
numbers are in each test's docstring (NVIDIA B200, 1000 W power limit).

Sample sets: uniform points; ray-ordered points at the neus render step (consecutive samples share coarse cells across
whole warps, the pattern the scatter's run-length aggregation is built for); degenerate tiles (one point repeated,
two points alternating, zero cotangents inside runs, ragged S); and the unit cube's faces, corners, cell faces and
points 1e-4 outside the cube (where the curvature probe lands near the AABB).
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import fields as of
from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import tinycudann as tcnn

pytestmark = pytest.mark.gpu

PLS = 1.447269237440378
PROD = {16: dict(otype="HashGrid", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
                 per_level_scale=PLS),
        32: dict(otype="HashGrid", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=32,
                 per_level_scale=PLS)}
SMALL = dict(otype="HashGrid", n_levels=6, n_features_per_level=2, log2_hashmap_size=12, base_resolution=4,
             per_level_scale=2.0)
K = 4.0                                 # bound = max(K x fp32-twin error, floor), per level and feature
FLOOR_FWD = 2e-6                        # y, dy_dx: a handful of fp32 roundings of the level's largest value
FLOOR_GRAD = 1e-5                       # scattered / reduced gradients
U = 2.0 ** -24                          # fp32 unit roundoff
STEP = 1.732 * 2 * 1.5 / 1024 / 3.0     # the neus render step in unit-cube coordinates (world / 2 radius)
SIZES = (1, 31, 33, 127, 129, 148 * 128 + 5)


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference and its fp32 twin
# ---------------------------------------------------------------------------------------------------------------------
def ref_levels(x, tabs, meta):
    """Per-level encodings [S, 2] of x [S, 3] (fp64 or fp32 holding the kernel's fp32 inputs) from per-level tables
    tabs[l] [size_l, 2]; arithmetic in tabs' dtype, cells exactly the kernel's."""
    dt = tabs[0].dtype
    x32 = x.detach().float()
    xd = x.to(dt)
    out = []
    for l in range(meta.n_levels):
        scale, res, size = meta.scale[l], meta.res[l], meta.size[l]
        pos = (x32.double() * scale + 0.5).float()          # fmaf: exact product, one rounding to fp32
        cell = torch.floor(pos)
        w = (pos - cell).to(dt) + scale * (xd - xd.detach())
        c0 = cell.to(torch.int64) & 0xFFFFFFFF               # (uint32_t)(int)floorf(p): -1 wraps
        idx, wts = [], []
        for k in range(8):
            b = [(k >> d) & 1 for d in range(3)]
            cc = [(c0[:, d] + b[d]) & 0xFFFFFFFF for d in range(3)]
            idx.append(of._grid_index(cc[0], cc[1], cc[2], res, size))
            wts.append((w[:, 0] if b[0] else 1 - w[:, 0]) * (w[:, 1] if b[1] else 1 - w[:, 1])
                       * (w[:, 2] if b[2] else 1 - w[:, 2]))
        corners = tabs[l][torch.stack(idx, 1)]              # [S, 8, 2]
        out.append((torch.stack(wts, 1)[:, :, None] * corners).sum(1))
    return out


def level_tables(flat, meta, dtype):
    t = flat.detach().cpu().view(-1, 2)
    return [t[meta.offset[l]:meta.offset[l + 1]].to(dtype).clone() for l in range(meta.n_levels)]


def split_table(flat, meta):
    t = flat.detach().view(-1, 2)
    return [t[meta.offset[l]:meta.offset[l + 1]] for l in range(meta.n_levels)]


def split_enc(t, meta):
    """[S, n_out] or [S, n_out, 3] -> per-level [S, 2] or [S, 2, 3]."""
    return [t[:, 2 * l:2 * l + 2] for l in range(meta.n_levels)]


def first_order(x, tabs, meta, gy):
    """d/d(x, table) of sum(y * gy)."""
    dt = tabs[0].dtype
    xl = x.detach().to(dt).requires_grad_(True)
    tl = [t.detach().requires_grad_(True) for t in tabs]
    y = torch.cat(ref_levels(xl, tl, meta), -1)
    g = torch.autograd.grad((y * gy.to(dt)).sum(), [xl] + tl)
    return g[0], list(g[1:])


def second_order(x, tabs, meta, gy, v):
    """Q = <v, dy_dx^T gy>: dQ/dx, dQ/dgy and dQ/dtable (what rsdf_hashgrid_bwd_bwd computes)."""
    dt = tabs[0].dtype
    xl = x.detach().to(dt).requires_grad_(True)
    gyl = gy.detach().to(dt).requires_grad_(True)
    tl = [t.detach().requires_grad_(True) for t in tabs]
    y = torch.cat(ref_levels(xl, tl, meta), -1)
    (gx,) = torch.autograd.grad((y * gyl).sum(), xl, create_graph=True)
    g = torch.autograd.grad((gx * v.to(dt)).sum(), [xl, gyl] + tl)
    return g[0], g[1], list(g[2:])


def jacobian(x, tabs, meta):
    """dy/dx [S, n_out, 3] by autograd through the reference (samples are independent: one grad per output)."""
    xl = x.detach().to(tabs[0].dtype).requires_grad_(True)
    cols = []
    for yl in ref_levels(xl, tabs, meta):
        for f in range(2):
            cols.append(torch.autograd.grad(yl[:, f].sum(), xl, retain_graph=True)[0])
    return torch.stack(cols, 1)


def compare(name, got, ref, twin, floor, per_feature=True):
    """Per level (and feature): max|got - ref| / max|ref| <= max(K * same for the fp32 twin, floor).  Lists of
    per-level tensors.  Returns the worst (error, twin error) for the report."""
    worst = (0.0, 0.0)
    for l, (g, r, t) in enumerate(zip(got, ref, twin)):
        g, r, t = g.detach().cpu().double(), r.detach().double(), t.detach().double()
        for f in (range(2) if per_feature else (None,)):
            gf, rf, tf = (g, r, t) if f is None else (g[:, f], r[:, f], t[:, f])
            m = float(rf.abs().max()) if rf.numel() else 0.0
            if m == 0.0:
                assert not torch.any(gf != 0), f"{name} level {l}: reference is 0, kernel is not"
                continue
            err = float((gf - rf).abs().max()) / m
            tw = float((tf - rf).abs().max()) / m
            bound = max(K * tw, floor)
            assert err <= bound, (f"{name}: level {l} feature {f}: error {err:.3g} of max|ref| > bound {bound:.3g} "
                                  f"(fp32 twin {tw:.3g})")
            worst = (max(worst[0], err), max(worst[1], tw))
    print(f"\n[{name}] worst level error {worst[0]:.3g}, fp32 twin {worst[1]:.3g}")
    return worst


def compare_rows(name, got, ref, twin, floor):
    """Per-sample quantities summed over levels ([S, 3] input gradients): same metric over the whole tensor."""
    return compare(name, [got], [ref], [twin], floor, per_feature=False)


def compare_kernels(name, a, b, ref, twin, floor):
    """Two kernel paths that compute the same sums in a different order: |a - b| per level within the bound the fp32
    twin sets around fp64 (the twin is moved onto b so that compare() measures its distance from the reference)."""
    return compare(name, a, b, [bi.double() + (t.double() - r) for bi, t, r in zip(b, twin, ref)], floor)


# ---------------------------------------------------------------------------------------------------------------------
# sample sets
# ---------------------------------------------------------------------------------------------------------------------
def ray_points(n_rays, n_per_ray, gen):
    """Rays through the cube sampled at the neus render step, ray after ray (consecutive samples on one ray)."""
    c = torch.rand(n_rays, 3, generator=gen) * 0.5 + 0.25
    d = F.normalize(torch.randn(n_rays, 3, generator=gen), dim=-1)
    t = (torch.arange(n_per_ray, dtype=torch.float32) - n_per_ray / 2) * STEP
    return (c[:, None, :] + t[None, :, None] * d[:, None, :]).reshape(-1, 3).contiguous()


def edge_points(gen):
    meta = of.HashGridMeta(16, 2, 19, 16, PLS)
    pts = [torch.tensor([[(k >> d) & 1 for d in range(3)] for k in range(8)], dtype=torch.float32)]
    for val in (0.0, 1.0):                                  # one coordinate exactly on a cube face
        for d in range(3):
            p = torch.rand(16, 3, generator=gen)
            p[:, d] = val
            pts.append(p)
    for l in (1, 12):                                       # cell faces of a dense and of a hashed level
        s = meta.scale[l]
        k = torch.randint(1, int(s), (16,), generator=gen).double()
        f = ((k - 0.5) / s).float()
        for d in range(3):
            for q in (f, torch.nextafter(f, torch.ones_like(f)), torch.nextafter(f, torch.zeros_like(f))):
                p = torch.rand(16, 3, generator=gen)
                p[:, d] = q
                pts.append(p)
    for val in (-1e-4, 1.0 + 1e-4):                         # just outside the cube: the curvature probe near the AABB
        for d in range(3):
            p = torch.rand(16, 3, generator=gen)
            p[:, d] = val
            pts.append(p)
    lo, hi = -1e-4, 1.0 + 1e-4
    pts.append(torch.tensor([[hi if (k >> d) & 1 else lo for d in range(3)] for k in range(8)], dtype=torch.float32))
    return torch.cat(pts).contiguous()


def degenerate_points(gen):
    """Four 128-sample tiles: one point repeated; two far-apart points alternating (every run has length 1 on every
    level); two ray segments (their cotangents get zero runs, see cotangent())."""
    rep = torch.rand(1, 3, generator=gen).expand(128, 3)
    alt = torch.tensor([[0.1, 0.15, 0.2], [0.9, 0.85, 0.8]]).repeat(64, 1)
    return torch.cat([rep, alt, ray_points(2, 128, gen)]).contiguous()


def sample_set(name):
    gen = torch.Generator().manual_seed(100 + SETS.index(name))
    if name == "uniform":
        return torch.rand(2048, 3, generator=gen)
    if name == "rays":
        return ray_points(8, 256, gen)
    if name == "degenerate":
        return degenerate_points(gen)
    if name == "edges":
        return edge_points(gen)
    raise KeyError(name)


SETS = ("uniform", "rays", "degenerate", "edges")


def cotangent(S, n_out, seed, degenerate=False):
    g = torch.randn(S, n_out, generator=torch.Generator().manual_seed(seed))
    if degenerate and S >= 512:
        g[384 + 8:384 + 24] = 0.0           # zero lanes in the middle of a run
        g[448:480, 0::2] = 0.0              # a whole warp with feature 0 zero and feature 1 not
    return g


# ---------------------------------------------------------------------------------------------------------------------
# grids
# ---------------------------------------------------------------------------------------------------------------------
_GRIDS = {}


def grid(cfg_key, table_scale):
    """(Encoding on cuda, oracle meta, fp64 level tables, fp32 level tables), cached per module."""
    key = (cfg_key, table_scale)
    if key not in _GRIDS:
        cfg = SMALL if cfg_key == "small" else PROD[cfg_key]
        enc = tcnn.Encoding(3, cfg)
        g = torch.Generator().manual_seed(7)
        with torch.no_grad():
            enc.params.copy_((torch.rand(enc.params.shape, generator=g) * 2 - 1) * table_scale)
        enc = enc.cuda()
        meta = of.HashGridMeta(cfg["n_levels"], 2, cfg["log2_hashmap_size"], cfg["base_resolution"],
                               cfg["per_level_scale"])
        assert meta.offset == enc.meta.offset and meta.res == enc.meta.res
        _GRIDS.clear()                      # one production table in host memory at a time
        _GRIDS[key] = (enc, meta, level_tables(enc.params, meta, torch.float64),
                       level_tables(enc.params, meta, torch.float32))
    return _GRIDS[key]


def test_production_grids_have_the_expected_dense_levels():
    """Levels 0-4 are dense at base 16, levels 0-2 at base 32; the rest are hashed (2^19 entries)."""
    for base, n_dense in ((16, 5), (32, 3)):
        meta = of.HashGridMeta(16, 2, 19, base, PLS)
        dense = [meta.res[l] ** 3 <= meta.size[l] for l in range(16)]
        assert dense == [True] * n_dense + [False] * (16 - n_dense)


def kernel_fwd(enc, x, with_jacobian):
    S, n_out = x.shape[0], enc.meta.n_output_dims
    y = torch.full((S, n_out), float("nan"), device="cuda")
    J = torch.full((S, n_out, 3), float("nan"), device="cuda") if with_jacobian else None
    L.call("rsdf_hashgrid_fwd", L.ptr(x), L.ptr(enc.params.detach()), enc.meta.ref, S, L.ptr(y), L.ptr(J), L.stream())
    return y, J


# ---------------------------------------------------------------------------------------------------------------------
# 1. forward, y and dy_dx
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base,table_scale", [(16, 1.0), (32, 1.0), (16, 1e-4)])
@pytest.mark.parametrize("name", SETS)
def test_forward_y_and_jacobian_per_level(base, table_scale, name):
    """rsdf_hashgrid_fwd with and without dy_dx vs fp64, per level, faces and out-of-cube points included.
    Measured (B200): y <= 2.3e-7, dy_dx <= 2.2e-7 of the level max; fp32 twin 1.5e-7 - 2.3e-7."""
    enc, meta, t64, t32 = grid(base, table_scale)
    x = sample_set(name)
    xc = x.cuda()
    y0, _ = kernel_fwd(enc, xc, False)
    y1, J = kernel_fwd(enc, xc, True)
    assert torch.equal(y0, y1)
    compare(f"fwd y {name} b{base} t{table_scale}", split_enc(y1.cpu(), meta), ref_levels(x, t64, meta),
            ref_levels(x, t32, meta), FLOOR_FWD)
    compare(f"fwd dy_dx {name} b{base} t{table_scale}", split_enc(J.cpu(), meta), split_enc(jacobian(x, t64, meta), meta),
            split_enc(jacobian(x, t32, meta), meta), FLOOR_FWD)


@pytest.mark.parametrize("S", SIZES)
def test_forward_ragged_sizes(S):
    """Partial warps and tiles: every row written (NaN-filled outputs), every level right.  Measured: <= 2.2e-7
    (1.6e-6 at S = 1, where the single sample sets the level max; twin 1.8e-6)."""
    enc, meta, t64, t32 = grid(16, 1.0)
    x = ray_points(S // 256 + 1, 256, torch.Generator().manual_seed(S))[:S].contiguous()
    y, J = kernel_fwd(enc, x.cuda(), True)
    assert not torch.isnan(y).any() and not torch.isnan(J).any()
    compare(f"fwd y S={S}", split_enc(y.cpu(), meta), ref_levels(x, t64, meta), ref_levels(x, t32, meta), FLOOR_FWD)


# ---------------------------------------------------------------------------------------------------------------------
# 2. first-order table and input gradients through `Encoding`
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base,table_scale", [(16, 1.0), (32, 1.0), (16, 1e-4)])
@pytest.mark.parametrize("name", SETS)
def test_first_order_grads_per_level(base, table_scale, name):
    """Encoding under autograd (rsdf_hashgrid_bwd_table, rsdf_hashgrid_bwd_input) vs fp64, per level.
    Measured: table <= 5.0e-7 (twin <= 6.6e-7), input gradient <= 1.9e-7 (twin <= 3.6e-7)."""
    enc, meta, t64, t32 = grid(base, table_scale)
    x = sample_set(name)
    gy = cotangent(x.shape[0], meta.n_output_dims, 3, degenerate=name == "degenerate")
    enc.params.grad = None
    xc = x.cuda().requires_grad_(True)
    (enc(xc) * gy.cuda()).sum().backward()
    rx, rt = first_order(x, t64, meta, gy)
    tx, tt = first_order(x, t32, meta, gy)
    compare(f"bwd_table {name} b{base} t{table_scale}", split_table(enc.params.grad.cpu(), meta), rt, tt, FLOOR_GRAD)
    compare_rows(f"bwd_input {name} b{base} t{table_scale}", xc.grad, rx, tx, FLOOR_GRAD)
    enc.params.grad = None


@pytest.mark.parametrize("S", SIZES)
def test_table_grad_ragged_sizes(S):
    """rsdf_hashgrid_bwd_table on ray-ordered samples at ragged S: inactive lanes (key 0xffffffff) next to active
    lanes of a run.  Measured: <= 2.3e-7 (twin 5.5e-7) at S = 148 x 128 + 5."""
    enc, meta, t64, t32 = grid(16, 1.0)
    x = ray_points(S // 256 + 1, 256, torch.Generator().manual_seed(S))[:S].contiguous()
    gy = cotangent(S, meta.n_output_dims, S)
    xc, gyc = x.cuda(), gy.cuda()          # held: a temporary's block would be handed to the next allocation
    gt = torch.zeros_like(enc.params.detach())
    L.call("rsdf_hashgrid_bwd_table", L.ptr(xc), L.ptr(gyc), enc.meta.ref, S, L.ptr(gt), L.stream())
    compare(f"bwd_table S={S}", split_table(gt.cpu(), meta), first_order(x, t64, meta, gy)[1],
            first_order(x, t32, meta, gy)[1], FLOOR_GRAD)


# ---------------------------------------------------------------------------------------------------------------------
# 3. every bwd_bwd instance
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg_key,name", [(16, "rays"), (16, "degenerate"), (32, "edges"), ("small", "uniform")])
def test_bwd_bwd_every_output_selection(cfg_key, name):
    """rsdf_hashgrid_bwd_bwd with each of the seven non-empty output selections <TO_TABLE, TO_DLDY, TO_X>: each
    requested output matches fp64 per level; requested per-sample outputs are fully written (NaN-filled) and
    unrequested buffers keep their sentinel.  Measured: table <= 7.1e-7 (twin 5.2e-7, reduced grid), dL_dy <= 1.9e-7,
    x <= 1.4e-7 (twins <= 1.9e-7)."""
    enc, meta, t64, t32 = grid(cfg_key, 1.0)
    x = sample_set(name)
    S, n_out = x.shape[0], meta.n_output_dims
    gy = cotangent(S, n_out, 5, degenerate=name == "degenerate")
    v = torch.randn(S, 3, generator=torch.Generator().manual_seed(6))
    r_x, r_gy, r_t = second_order(x, t64, meta, gy, v)
    w_x, w_gy, w_t = second_order(x, t32, meta, gy, v)
    xc, gyc, vc = x.cuda(), gy.cuda(), v.cuda()
    table = enc.params.detach()
    for sel in range(1, 8):
        want_t, want_gy, want_x = bool(sel & 4), bool(sel & 2), bool(sel & 1)
        gt = torch.zeros_like(table) if want_t else torch.full((8,), -7.0, device="cuda")
        ggy = torch.full((S, n_out), float("nan") if want_gy else -7.0, device="cuda")
        gx = torch.full((S, 3), float("nan") if want_x else -7.0, device="cuda")
        L.call("rsdf_hashgrid_bwd_bwd", L.ptr(xc), L.ptr(table), L.ptr(vc), L.ptr(gyc), enc.meta.ref, S,
               L.ptr(gt) if want_t else None, L.ptr(ggy) if want_gy else None, L.ptr(gx) if want_x else None,
               L.stream())
        tag = f"bwd_bwd<{want_t},{want_gy},{want_x}> {name} {cfg_key}"
        if want_t:
            compare(tag + " table", split_table(gt.cpu(), meta), r_t, w_t, FLOOR_GRAD)
        else:
            assert torch.all(gt == -7.0)
        if want_gy:
            compare(tag + " dL_dy", split_enc(ggy.cpu(), meta), split_enc(r_gy, meta), split_enc(w_gy, meta), FLOOR_GRAD)
        else:
            assert torch.all(ggy == -7.0)
        if want_x:
            compare_rows(tag + " x", gx.cpu(), r_x, w_x, FLOOR_GRAD)
        else:
            assert torch.all(gx == -7.0)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the linked analytic-normal path (VolumeSDF._forward_fused_analytic)
# ---------------------------------------------------------------------------------------------------------------------
def smooth_f(n_out, table_scale, dtype, device):
    """A fixed small softplus net R^n_out -> R per sample, scaled so that the hash-grid normal is O(1)."""
    g = torch.Generator().manual_seed(21)
    W1 = (torch.randn(n_out, 16, generator=g) / math.sqrt(n_out)).to(device, dtype)
    b1 = (torch.randn(16, generator=g) * 0.1).to(device, dtype)
    w2 = (torch.randn(16, generator=g) * 1e-3 / table_scale / math.sqrt(16)).to(device, dtype)
    return lambda y: F.softplus(y @ W1 + b1) @ w2


def linked_loss(y, gx, c, gy):
    return (gx * c).sum() + ((gx.norm(dim=-1) - 1.0) ** 2).sum() + (y * gy).sum()


@pytest.mark.parametrize("x_grad", [False, True])
@pytest.mark.parametrize("base,table_scale,name", [(16, 1.0, "rays"), (32, 1e-4, "rays"), (16, 1.0, "edges"),
                                                   (32, 1.0, "degenerate")])
def test_linked_analytic_normal_path(base, table_scale, name, x_grad):
    """hashgrid_with_jacobian -> g2 = df/dy (create_graph) -> hashgrid_input_grad: the table gradient (one
    rsdf_hashgrid_bwd_table2 scatter) and, for the curvature probe, the gradient to x (rsdf_hashgrid_bwd_input +
    bwd_bwd<false,false,true>) vs fp64 autograd of the same loss; and the linked path equals the op-by-op path
    (Encoding double backward: bwd_table + bwd_bwd<TO_TABLE>) to fp32 rounding.  Measured: table <= 7.7e-7 at O(1)
    tables (twin 7.1e-7), 3.9e-6 at the 1e-4 initial scale (twin 4.0e-6); x <= 4.2e-7 (twin 4.1e-7); linked vs
    op-by-op <= 5.6e-7."""
    enc, meta, t64, t32 = grid(base, table_scale)
    x = sample_set(name)
    S, n_out = x.shape[0], meta.n_output_dims
    gen = torch.Generator().manual_seed(8)
    c, gy = torch.randn(S, 3, generator=gen), torch.randn(S, n_out, generator=gen) * table_scale

    def product(linked):
        enc.params.grad = None
        xc = x.cuda().requires_grad_(x_grad)
        f = smooth_f(n_out, table_scale, torch.float32, "cuda")
        if linked:
            y, J, link = tcnn.hashgrid_with_jacobian(enc, xc)
            (g2,) = torch.autograd.grad(f(y).sum(), y, create_graph=True)
            gx = tcnn.hashgrid_input_grad(enc, g2, xc, J, link)
        else:
            xr = xc if x_grad else xc.detach().requires_grad_(True)
            y = enc(xr)
            (g2,) = torch.autograd.grad(f(y).sum(), y, create_graph=True)
            (gx,) = torch.autograd.grad(y, xr, g2, create_graph=True)
        linked_loss(y, gx, c.cuda(), gy.cuda()).backward()
        gt = enc.params.grad.detach().clone()
        enc.params.grad = None
        return gt, (xc.grad.detach().clone() if x_grad else None)

    def reference(tabs):
        dt = tabs[0].dtype
        xl = x.to(dt).requires_grad_(True)
        tl = [t.detach().requires_grad_(True) for t in tabs]
        y = torch.cat(ref_levels(xl, tl, meta), -1)
        (gx,) = torch.autograd.grad(smooth_f(n_out, table_scale, dt, "cpu")(y).sum(), xl, create_graph=True)
        g = torch.autograd.grad(linked_loss(y, gx, c.to(dt), gy.to(dt)), [xl] + tl)
        return list(g[1:]), g[0]

    gt_link, gx_link = product(True)
    gt_op, gx_op = product(False)
    r_t, r_x = reference(t64)
    w_t, w_x = reference(t32)
    tag = f"linked {name} b{base} t{table_scale} x_grad={x_grad}"
    compare(tag + " table", split_table(gt_link.cpu(), meta), r_t, w_t, FLOOR_GRAD)
    compare(tag + " op-by-op table", split_table(gt_op.cpu(), meta), r_t, w_t, FLOOR_GRAD)
    compare_kernels(tag + " linked vs op-by-op", split_table(gt_link.cpu(), meta), split_table(gt_op.cpu(), meta),
                    r_t, w_t, FLOOR_GRAD)
    if x_grad:
        compare_rows(tag + " x", gx_link.cpu(), r_x, w_x, FLOOR_GRAD)
        compare_rows(tag + " op-by-op x", gx_op.cpu(), r_x, w_x, FLOOR_GRAD)


# ---------------------------------------------------------------------------------------------------------------------
# 5. table2 directly
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base,name", [(16, "rays"), (16, "degenerate"), (32, "uniform"), (32, "edges")])
def test_table2_equals_bwd_table_plus_bwd_bwd_table(base, name):
    """rsdf_hashgrid_bwd_table2(x, dL_dy, v, g2) == rsdf_hashgrid_bwd_table(x, dL_dy) + bwd_bwd<TO_TABLE>(x, v, g2)
    into one buffer, to fp32 atomic-order rounding, and both == fp64 per level.  Measured: table2 <= 7.4e-7, the
    two-pass sum <= 4.6e-7, table2 vs two-pass <= 7.2e-7 (twin <= 9.8e-7)."""
    enc, meta, t64, t32 = grid(base, 1.0)
    x = sample_set(name)
    S, n_out = x.shape[0], meta.n_output_dims
    gy = cotangent(S, n_out, 9, degenerate=name == "degenerate")
    g2 = cotangent(S, n_out, 10, degenerate=name == "degenerate") * 1e-3
    v = torch.randn(S, 3, generator=torch.Generator().manual_seed(11))
    xc, gyc, g2c, vc, table = x.cuda(), gy.cuda(), g2.cuda(), v.cuda(), enc.params.detach()
    a = torch.zeros_like(table)
    L.call("rsdf_hashgrid_bwd_table2", L.ptr(xc), L.ptr(gyc), L.ptr(vc), L.ptr(g2c), enc.meta.ref, S, L.ptr(a),
           L.stream())
    b = torch.zeros_like(table)
    L.call("rsdf_hashgrid_bwd_table", L.ptr(xc), L.ptr(gyc), enc.meta.ref, S, L.ptr(b), L.stream())
    L.call("rsdf_hashgrid_bwd_bwd", L.ptr(xc), L.ptr(table), L.ptr(vc), L.ptr(g2c), enc.meta.ref, S, L.ptr(b), None,
           None, L.stream())

    def reference(tabs):
        return [p + q for p, q in zip(first_order(x, tabs, meta, gy)[1], second_order(x, tabs, meta, g2, v)[2])]

    r, w = reference(t64), reference(t32)
    compare(f"table2 {name} b{base}", split_table(a.cpu(), meta), r, w, FLOOR_GRAD)
    compare(f"table+bwd_bwd {name} b{base}", split_table(b.cpu(), meta), r, w, FLOOR_GRAD)
    compare_kernels(f"table2 vs table+bwd_bwd {name} b{base}", split_table(a.cpu(), meta), split_table(b.cpu(), meta),
                    r, w, FLOOR_GRAD)


# ---------------------------------------------------------------------------------------------------------------------
# 6. jvp and bwd_input on the stored Jacobian
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_out", [12, 32, 48])
@pytest.mark.parametrize("S", (1, 7, 33, 1029))
def test_jvp_and_bwd_input_contractions(n_out, S):
    """g[s,f] = sum_d J[s,f,d] v[s,d] (rsdf_hashgrid_jvp) and dL_dx[s,d] = sum_f J[s,f,d] g[s,f]
    (rsdf_hashgrid_bwd_input) vs the fp64 contractions, elementwise within the fp32 summation bound
    (roundings on a term's path) x u x sum|terms|: 3 fmas for the jvp; ceil(n_out / 32) fmas per lane and a
    5-level shuffle tree for bwd_input."""
    gen = torch.Generator().manual_seed(100 * n_out + S)
    scale = torch.logspace(0, 3.5, n_out)[None, :, None]    # level scales: fine-level columns dominate
    J = (torch.randn(S, n_out, 3, generator=gen) * scale).contiguous()
    v = torch.randn(S, 3, generator=gen)
    g = torch.randn(S, n_out, generator=gen)
    Jc, vc, gc = J.cuda(), v.cuda(), g.cuda()
    out = torch.full((S, n_out), float("nan"), device="cuda")
    L.call("rsdf_hashgrid_jvp", L.ptr(Jc), L.ptr(vc), S, n_out, L.ptr(out), L.stream())
    terms = J.double() * v.double()[:, None, :]
    err = (out.cpu().double() - terms.sum(-1)).abs()
    assert torch.all(err <= 4 * U * terms.abs().sum(-1)), float((err / terms.abs().sum(-1)).max())
    dx = torch.full((S, 3), float("nan"), device="cuda")
    L.call("rsdf_hashgrid_bwd_input", L.ptr(Jc), L.ptr(gc), S, n_out, L.ptr(dx), L.stream())
    terms = J.double() * g.double()[:, :, None]
    err = (dx.cpu().double() - terms.sum(1)).abs()
    assert torch.all(err <= (math.ceil(n_out / 32) + 6) * U * terms.abs().sum(1)), float((err / terms.abs().sum(1)).max())


# ---------------------------------------------------------------------------------------------------------------------
# 7. the finite-difference training node
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eps", [1e-3, 2 * 1.5 / 8180.0])
def test_fd6_train_table_grad(eps):
    """hashgrid_fd6_train's table gradient == the fp64 scatter of the cotangent over the node's own x01 output (whose
    positions test_fd6_neighbours_bit_identical_to_six_forward_passes pins); points at +-radius make neighbours clamp
    onto the same position.  Measured: <= 5.7e-7 (twin 7.8e-7)."""
    enc, meta, t64, t32 = grid(32, 1.0)
    r = 1.5
    gen = torch.Generator().manual_seed(12)
    p = (torch.rand(1024, 3, generator=gen) * 2 - 1) * r
    p[:8] = torch.tensor([[r if (k >> d) & 1 else -r for d in range(3)] for k in range(8)], dtype=torch.float32)
    p[8:40, 0] = r
    p[40:72, 1] = -r
    p[72:104] = p[72]                                       # one point repeated: 6 x 32 neighbour rows, 6 positions
    enc.params.grad = None
    x01, y = tcnn.hashgrid_fd6_train(enc, p.cuda(), eps, r)
    gy = cotangent(y.shape[0], meta.n_output_dims, 13)
    (y * gy.cuda()).sum().backward()
    x = x01.cpu()
    compare(f"fd6 train eps={eps:.3g}", split_table(enc.params.grad.cpu(), meta), first_order(x, t64, meta, gy)[1],
            first_order(x, t32, meta, gy)[1], FLOOR_GRAD)
    enc.params.grad = None


# ---------------------------------------------------------------------------------------------------------------------
# 8. conservation at production scale
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", [16, 32])
def test_scatter_conservation_at_training_scale(base):
    """3.3 M ray-ordered samples (one neus step's worth; coarse entries take millions of same-entry atomics).
    Per level and feature: sum of the first-order table gradient == sum of dL_dy (the trilinear weights sum to one),
    and the second-order part of rsdf_hashgrid_bwd_table2 (table2 - bwd_table) sums to 0 (the weight derivatives sum
    to zero over the 8 corners).  Bounds are relative to the sum of |terms|: sum|dL_dy| and
    sum 2 scale |v|_1 |g2| >= sum_c |coef_c g2|.  Measured: first order <= 1.9e-8, second order <= 8.1e-10."""
    enc, meta, _, _ = grid(base, 1.0)
    gen = torch.Generator(device="cuda").manual_seed(14)
    n_rays, n_per = 12900, 256
    c = torch.rand(n_rays, 3, device="cuda", generator=gen) * 0.5 + 0.25
    d = F.normalize(torch.randn(n_rays, 3, device="cuda", generator=gen), dim=-1)
    t = (torch.arange(n_per, device="cuda", dtype=torch.float32) - n_per / 2) * STEP
    x = (c[:, None, :] + t[None, :, None] * d[:, None, :]).reshape(-1, 3).contiguous()
    S, n_out = x.shape[0], meta.n_output_dims
    gy = torch.randn(S, n_out, device="cuda", generator=gen) + 0.25
    g2 = torch.randn(S, n_out, device="cuda", generator=gen)
    v = torch.randn(S, 3, device="cuda", generator=gen)
    a = torch.zeros_like(enc.params.detach())
    L.call("rsdf_hashgrid_bwd_table", L.ptr(x), L.ptr(gy), enc.meta.ref, S, L.ptr(a), L.stream())
    b = torch.zeros_like(a)
    L.call("rsdf_hashgrid_bwd_table2", L.ptr(x), L.ptr(gy), L.ptr(v), L.ptr(g2), enc.meta.ref, S, L.ptr(b), L.stream())
    v1 = v.double().abs().sum(1, keepdim=True)
    worst1 = worst2 = 0.0
    for l in range(meta.n_levels):
        ga = a.view(-1, 2)[meta.offset[l]:meta.offset[l + 1]].double()
        gb = b.view(-1, 2)[meta.offset[l]:meta.offset[l + 1]].double()
        want = gy[:, 2 * l:2 * l + 2].double().sum(0)
        abs1 = gy[:, 2 * l:2 * l + 2].double().abs().sum(0)
        abs2 = (2 * meta.scale[l] * v1 * g2[:, 2 * l:2 * l + 2].double().abs()).sum(0)
        e1 = ((ga.sum(0) - want).abs() / abs1).max().item()
        e2 = ((gb - ga).sum(0).abs() / (abs1 + abs2)).max().item()
        assert e1 <= 2e-7, f"first order, level {l}: |sum grad - sum dL_dy| = {e1:.3g} of sum|dL_dy|"
        assert e2 <= 2e-7, f"second order, level {l}: |sum| = {e2:.3g} of sum|terms|"
        worst1, worst2 = max(worst1, e1), max(worst2, e2)
    print(f"\n[conservation b{base}] first order {worst1:.3g}, second order {worst2:.3g} (of sum|terms|)")


# ---------------------------------------------------------------------------------------------------------------------
# 9. the _Link hand-off
# ---------------------------------------------------------------------------------------------------------------------
def test_link_park_is_not_consumed_by_another_backward():
    """A backward that reaches the input-grad node but not the linked forward node (here: a gradient to g2 only)
    parks (v, g2) on the link.  A later backward through the forward node alone must not scatter that stale
    second-order term: its table gradient equals the plain first-order gradient.  (Before the park was tagged with
    its backward sweep, the stale term put the gradient 46 off at a max of 8.8.)"""
    enc, meta, _, _ = grid(16, 1.0)
    x = sample_set("rays").cuda()
    S, n_out = x.shape[0], meta.n_output_dims
    gen = torch.Generator().manual_seed(15)
    gy = torch.randn(S, n_out, generator=gen).cuda()
    c = torch.randn(S, 3, generator=gen).cuda()
    g2 = (torch.randn(S, n_out, generator=gen) * 1e-3).cuda().requires_grad_(True)
    y, J, link = tcnn.hashgrid_with_jacobian(enc, x)
    gx = tcnn.hashgrid_input_grad(enc, g2, x, J, link)
    loss = (gx * c).sum() + (y * gy).sum()
    torch.autograd.grad(loss, [g2], retain_graph=True)
    (got,) = torch.autograd.grad((y * gy).sum(), enc.params, retain_graph=True)
    want = torch.zeros_like(got)
    L.call("rsdf_hashgrid_bwd_table", L.ptr(x), L.ptr(gy), enc.meta.ref, S, L.ptr(want), L.stream())
    assert float((got - want).abs().max()) <= 1e-6 * float(want.abs().max())
    # a whole-loss backward still gets both orders, in one table2 scatter: first order + bwd_bwd<TO_TABLE>(v = c)
    (full,) = torch.autograd.grad(loss, enc.params)
    want2 = want.clone()
    L.call("rsdf_hashgrid_bwd_bwd", L.ptr(x), L.ptr(enc.params.detach()), L.ptr(c), L.ptr(g2.detach()), enc.meta.ref, S,
           L.ptr(want2), None, None, L.stream())
    for l in range(meta.n_levels):
        a, b = split_table(full, meta)[l], split_table(want2, meta)[l]
        assert float((a - b).abs().max()) <= 1e-5 * float(b.abs().max()), l
