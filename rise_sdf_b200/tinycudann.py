"""Drop-in for `tinycudann.Encoding` as RISE-SDF uses it (models/network_utils.py:50,99):
`HashGrid` and `SphericalHarmonics` encodings backed by librsdf_b200.so, with the full
autograd surface the reference relies on -- `torch.autograd.grad(out, x, create_graph=True)`
followed by a backward through that result to `params` and `x` (models/geometry.py:224-228,
266-273).  tiny-cuda-nn itself is third-party and absent from the reference tree; the
arithmetic follows its published algorithm (SURVEY.md Appendix A.1/A.2), in fp32 (the
reference build runs fp16 params/outputs and up-casts: models/geometry.py:217).
"""
import numpy as np
import torch
from torch import nn

from . import _lib as L


class HashGridMeta:
    """grid_scale()/grid_resolution()/offset table of tcnn's GridEncoding, evaluated on the host in
    float32: scale_l = exp2f(l*log2f(pls))*base - 1, res_l = ceil(scale_l)+1,
    n_l = min(next_multiple(res_l^3, 8), 2^log2_hashmap_size)."""

    def __init__(self, n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
                 per_level_scale=2.0):
        if n_features_per_level != 2:
            raise NotImplementedError("n_features_per_level must be 2 (both RISE-SDF configs)")
        if n_levels > L.MAX_LEVELS:
            raise ValueError("too many levels")
        self.n_levels, self.n_features = n_levels, n_features_per_level
        log2_pls = np.float32(np.log2(per_level_scale))
        self.scale, self.res, self.size, self.offset = [], [], [], [0]
        for l in range(n_levels):
            s = np.float32(np.exp2(np.float32(np.float32(l) * log2_pls))) * np.float32(base_resolution) - np.float32(1.0)
            s = np.float32(s)
            r = int(np.ceil(s)) + 1
            n = min(r ** 3, (2 ** 32 - 1) // 2)
            n = (n + 7) // 8 * 8
            n = min(n, 1 << log2_hashmap_size)
            self.scale.append(float(s)); self.res.append(r); self.size.append(n)
            self.offset.append(self.offset[-1] + n)
        self.n_params = self.offset[-1] * n_features_per_level
        self.n_output_dims = n_levels * n_features_per_level
        c = L.HashGridMetaC()
        c.n_levels, c.n_features = n_levels, n_features_per_level
        for l in range(n_levels):
            c.scale[l], c.res[l], c.offset[l] = self.scale[l], self.res[l], self.offset[l]
        c.offset[n_levels] = self.offset[n_levels]
        self.c = c

    @property
    def ref(self):
        import ctypes
        return ctypes.byref(self.c)


class _HashGridBackward(torch.autograd.Function):
    """(dL_dy, x, table, dy_dx) -> (dL_dx, dL_dtable); itself differentiable once more."""

    @staticmethod
    def forward(ctx, gy, x, table, dy_dx, meta, need_x, need_table):
        S, n_out = gy.shape
        gx = gt = None
        if need_x:
            gx = torch.empty(S, 3, device=gy.device, dtype=torch.float32)
            L.call("rsdf_hashgrid_bwd_input", L.ptr(dy_dx), L.ptr(gy), S, n_out, L.ptr(gx), L.stream())
        if need_table:
            gt = torch.zeros_like(table)
            L.call("rsdf_hashgrid_bwd_table", L.ptr(x), L.ptr(gy), meta.ref, S, L.ptr(gt), L.stream())
        ctx.save_for_backward(gy, x, table)
        ctx.meta = meta
        return gx, gt

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, ggx, ggt):
        gy, x, table = ctx.saved_tensors
        # ggt (a cotangent on the table gradient) never occurs on the render path
        if ggx is None:
            return None, None, None, None, None, None, None
        S, n_out = gy.shape
        v = ggx.contiguous()
        need_gy, need_x, need_t = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        g_gy = torch.empty_like(gy) if need_gy else None
        g_x = torch.empty_like(x) if need_x else None
        g_t = torch.zeros_like(table) if need_t else None
        L.call("rsdf_hashgrid_bwd_bwd", L.ptr(x), L.ptr(table), L.ptr(v), L.ptr(gy), ctx.meta.ref, S,
               L.ptr(g_t), L.ptr(g_gy), L.ptr(g_x), L.stream())
        return g_gy, g_x, g_t, None, None, None, None


class _HashGridForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, table, meta):
        S = x.shape[0]
        need_x = x.requires_grad
        y = torch.empty(S, meta.n_output_dims, device=x.device, dtype=torch.float32)
        dy_dx = torch.empty(S, meta.n_output_dims, 3, device=x.device, dtype=torch.float32) if need_x else None
        L.call("rsdf_hashgrid_fwd", L.ptr(x), L.ptr(table), meta.ref, S, L.ptr(y), L.ptr(dy_dx), L.stream())
        ctx.save_for_backward(x, table, dy_dx)
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, gy):
        x, table, dy_dx = ctx.saved_tensors
        gx, gt = _HashGridBackward.apply(gy.contiguous(), x, table, dy_dx, ctx.meta,
                                         ctx.needs_input_grad[0] and dy_dx is not None,
                                         ctx.needs_input_grad[1])
        return gx, gt, None


class _Link:
    """Shared by the two autograd nodes of the fused analytic-normal path.  The second-order node runs
    first in the backward sweep (its output feeds the MLP node) and, instead of scattering its table
    gradient right away, parks (v, g2) here; the first-order node then adds both contributions to the
    table with ONE scatter pass (rsdf_hashgrid_bwd_table2).

    The pair is tagged with the autograd graph task (one backward sweep) that parked it, and only that sweep may
    consume it: a backward that reaches the second-order node but not the first-order one (a gradient to g2 alone,
    say) would otherwise leave a pair behind for a later, unrelated backward through the forward node to scatter."""
    __slots__ = ("v", "g2", "task")

    def __init__(self):
        self.v = self.g2 = self.task = None

    def park(self, v, g2):
        self.v, self.g2, self.task = v, g2, torch._C._current_graph_task_id()

    def take(self):
        """(v, g2) parked by the running backward sweep, else None; the link is empty afterwards either way."""
        pair = (self.v, self.g2) if self.v is not None and self.task == torch._C._current_graph_task_id() else None
        self.v = self.g2 = self.task = None
        return pair


class _HashGridForwardJ(torch.autograd.Function):
    """(x, table) -> (y, dy_dx) with the Jacobian as an explicit, non-differentiable output: the fused
    SDF-field path (rise_sdf_b200/sdf_field.py) contracts it with d sdf/d enc itself instead of
    going through torch.autograd.grad."""

    @staticmethod
    def forward(ctx, x, table, meta, link):
        S = x.shape[0]
        y = torch.empty(S, meta.n_output_dims, device=x.device, dtype=torch.float32)
        dy_dx = torch.empty(S, meta.n_output_dims, 3, device=x.device, dtype=torch.float32)
        L.call("rsdf_hashgrid_fwd", L.ptr(x), L.ptr(table), meta.ref, S, L.ptr(y), L.ptr(dy_dx), L.stream())
        ctx.save_for_backward(x, table, dy_dx)
        ctx.meta, ctx.link = meta, link
        ctx.mark_non_differentiable(dy_dx)
        return y, dy_dx

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy, _g_dy_dx):
        x, table, dy_dx = ctx.saved_tensors
        S, n_out = gy.shape
        gy = gy.contiguous()
        gx, gt = None, None
        parked = ctx.link.take() if ctx.link is not None else None
        if ctx.needs_input_grad[0]:
            gx = torch.empty(S, 3, device=gy.device, dtype=torch.float32)
            L.call("rsdf_hashgrid_bwd_input", L.ptr(dy_dx), L.ptr(gy), S, n_out, L.ptr(gx), L.stream())
        if ctx.needs_input_grad[1]:
            gt = torch.zeros_like(table)
            if parked is not None:
                v, g2 = parked
                L.call("rsdf_hashgrid_bwd_table2", L.ptr(x), L.ptr(gy), L.ptr(v), L.ptr(g2), ctx.meta.ref, S,
                       L.ptr(gt), L.stream())
            else:
                L.call("rsdf_hashgrid_bwd_table", L.ptr(x), L.ptr(gy), ctx.meta.ref, S, L.ptr(gt), L.stream())
        return gx, gt, None, None


class _HashGridInputGrad(torch.autograd.Function):
    """(g2, dy_dx; x, table) -> dy_dx^T g2 [S,3] for the fused path.  Backward (the second-order pass):
    d/d g2 = dy_dx . v from the stored Jacobian; the table leg is deferred to the linked first-order
    node (see _Link).  When x requires grad (the curvature probe of models/geometry.py:246-282 sits at
    x + 1e-4 tangent(theta)) its leg -- d/dx of (dy_dx^T g2) . v, the mixed second derivatives of the trilinear
    interpolation -- comes from rsdf_hashgrid_bwd_bwd; on the render path proper sample positions are data."""

    @staticmethod
    def forward(ctx, g2, dy_dx, x, table, meta, link):
        S, n_out = g2.shape
        g2 = g2.contiguous()
        gx = torch.empty(S, 3, device=g2.device, dtype=torch.float32)
        L.call("rsdf_hashgrid_bwd_input", L.ptr(dy_dx), L.ptr(g2), S, n_out, L.ptr(gx), L.stream())
        ctx.save_for_backward(g2, dy_dx, x, table)
        ctx.meta, ctx.link = meta, link
        return gx

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, v):
        g2, dy_dx, x, table = ctx.saved_tensors
        S, n_out = g2.shape
        v = v.contiguous()
        g_g2 = None
        if ctx.needs_input_grad[0]:
            g_g2 = torch.empty_like(g2)
            L.call("rsdf_hashgrid_jvp", L.ptr(dy_dx), L.ptr(v), S, n_out, L.ptr(g_g2), L.stream())
        g_x = None
        if ctx.needs_input_grad[2]:
            g_x = torch.empty_like(x)
            L.call("rsdf_hashgrid_bwd_bwd", L.ptr(x), L.ptr(table), L.ptr(v), L.ptr(g2), ctx.meta.ref, S,
                   None, None, L.ptr(g_x), L.stream())
        if table.requires_grad:
            ctx.link.park(v, g2)
        return g_g2, None, g_x, None, None, None


def hashgrid_with_jacobian(enc, x):
    """enc: a HashGrid `Encoding`; x [S,3] in [0,1] -> (y [S,n_out], dy_dx [S,n_out,3], link)."""
    L.require_cuda(x)
    link = _Link()
    y, dy_dx = _HashGridForwardJ.apply(x, enc.params, enc.meta, link)
    return y, dy_dx, link


def hashgrid_input_grad(enc, g2, x, dy_dx, link):
    """dy_dx^T g2 -> [S,3]; differentiable w.r.t. g2 and (through the linked forward node) the table."""
    return _HashGridInputGrad.apply(g2, dy_dx, x, enc.params, enc.meta, link)


@torch.no_grad()
def hashgrid_fd6(enc, points, eps, radius):
    """Six finite-difference neighbours per point (inference only): points [S,3] in world units ->
    (x01 [6S,3], y [6S,n_out]), rows ordered 6 s + k with k = +x,-x,+y,-y,+z,-z."""
    L.require_cuda(points)
    points = points.contiguous().float()
    S = points.shape[0]
    x01 = torch.empty(6 * S, 3, device=points.device, dtype=torch.float32)
    y = torch.empty(6 * S, enc.meta.n_output_dims, device=points.device, dtype=torch.float32)
    L.call("rsdf_hashgrid_fd6", L.ptr(points), L.ptr(enc.params.detach()), enc.meta.ref, S, float(eps), float(radius),
           L.ptr(x01), L.ptr(y), L.stream())
    return x01, y


class _HashGridFD6(torch.autograd.Function):
    """The training-time twin of `hashgrid_fd6`: (points, table) -> (x01 [6S,3] non-differentiable, y [6S,n_out]); the
    backward is the ordinary table scatter over the 6S neighbour positions (the points are data on the render path).
    The forward shares corner gathers between the six neighbours of a sample, which the generic forward over 6S
    independent points cannot (8.8 M points per split-sum step: 2.3 -> 1.2 ms)."""

    @staticmethod
    def forward(ctx, points, table, enc, eps, radius):
        points = points.contiguous().float()
        S = points.shape[0]
        x01 = torch.empty(6 * S, 3, device=points.device, dtype=torch.float32)
        y = torch.empty(6 * S, enc.meta.n_output_dims, device=points.device, dtype=torch.float32)
        L.call("rsdf_hashgrid_fd6", L.ptr(points), L.ptr(table), enc.meta.ref, S, float(eps), float(radius), L.ptr(x01),
               L.ptr(y), L.stream())
        ctx.save_for_backward(x01, table)
        ctx.meta = enc.meta
        ctx.mark_non_differentiable(x01)
        return x01, y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, _gx, gy):
        x01, table = ctx.saved_tensors
        gt = None
        if ctx.needs_input_grad[1]:
            gt = torch.zeros_like(table)
            L.call("rsdf_hashgrid_bwd_table", L.ptr(x01), L.ptr(gy.contiguous().float()), ctx.meta.ref, x01.shape[0], L.ptr(gt),
                   L.stream())
        return None, gt, None, None, None


def hashgrid_fd6_train(enc, points, eps, radius):
    """`hashgrid_fd6` with autograd to the hash table (points [S,3] carry no gradient)."""
    L.require_cuda(points)
    return _HashGridFD6.apply(points.detach(), enc.params, enc, eps, radius)


class _SHForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u, degree):
        S = u.shape[0]
        out = torch.empty(S, degree * degree, device=u.device, dtype=torch.float32)
        L.call("rsdf_sh_fwd", L.ptr(u), S, degree, L.ptr(out), L.stream())
        ctx.save_for_backward(u)
        ctx.degree = degree
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, go):
        (u,) = ctx.saved_tensors
        gu = torch.empty_like(u)
        L.call("rsdf_sh_bwd", L.ptr(u), L.ptr(go.contiguous()), u.shape[0], ctx.degree, L.ptr(gu), L.stream())
        return gu, None


class Encoding(nn.Module):
    """tinycudann.Encoding(n_input_dims, encoding_config, seed=1337).  Unknown config keys
    (include_xyz, start_level, ...: models/network_utils.py:47-50,99) are ignored like tcnn does.
    `params` is one flat fp32 Parameter in tcnn's level-major order, so reference checkpoints load."""

    def __init__(self, n_input_dims, encoding_config, seed=1337, dtype=torch.float32):
        super().__init__()
        cfg = dict(encoding_config)
        self.n_input_dims = n_input_dims
        self.encoding_config = cfg
        otype = cfg["otype"]
        if n_input_dims != 3:
            raise NotImplementedError("3-D inputs only")
        if otype in ("HashGrid", "Grid"):
            self.kind = "hashgrid"
            self.meta = HashGridMeta(cfg.get("n_levels", 16), cfg.get("n_features_per_level", 2),
                                     cfg.get("log2_hashmap_size", 19), cfg.get("base_resolution", 16),
                                     cfg.get("per_level_scale", 2.0))
            self.n_output_dims = self.meta.n_output_dims
            g = torch.Generator().manual_seed(seed)
            self.params = nn.Parameter((torch.rand(self.meta.n_params, generator=g) * 2 - 1) * 1e-4)
        elif otype == "SphericalHarmonics":
            self.kind = "sh"
            self.degree = int(cfg["degree"])
            self.n_output_dims = self.degree ** 2
            self.params = nn.Parameter(torch.zeros(0))
        else:
            raise NotImplementedError(f"encoding otype {otype!r} is not used by RISE-SDF's render path")

    def forward(self, x):
        L.require_cuda(x)
        x = x.contiguous().float()
        if x.shape[0] == 0:
            return x.new_zeros(0, self.n_output_dims)
        if self.kind == "hashgrid":
            return _HashGridForward.apply(x, self.params, self.meta)
        return _SHForward.apply(x, self.degree)


def free_temporary_memory():
    """tinycudann.free_temporary_memory(): nothing is cached outside torch's allocator here."""
    return None


class Network(nn.Module):
    def __init__(self, *a, **k):
        raise NotImplementedError("tcnn.Network is never constructed under RISE-SDF's configs "
                                  "(all MLPs are VanillaMLP; README.md:56 builds tcnn --no-networks)")


NetworkWithInputEncoding = Network
