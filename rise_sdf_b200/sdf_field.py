"""Host side of the fused SDF-field MLP kernels (csrc/sdf_train.cu): the `VanillaMLP` of
`VolumeSDF` (models/geometry.py:206-228; 35 -> 128 -> 128 -> 48, Softplus(beta=100), weight-norm folded
on the host) evaluated TOGETHER with g0 = d sdf / d h0 -- what the reference obtains through
`torch.autograd.grad(sdf, points, create_graph=True)` -- as ONE autograd node whose backward is ONE
kernel that also carries the second-order terms (eikonal loss, normal-dependent shading).

    out, g0 = fused_sdf(mlp, in0, scale0, shift0, in1)        h0 = cat(in0 * scale0 + shift0, in1)

`out`/`g0` are differentiable w.r.t. in0, in1 and every MLP parameter (first order in `out`, and through
`g0` second order in the network); the node itself is once-differentiable, which is all the render
path needs (no third-order terms exist in the reference's losses).
"""
import ctypes

import torch

from . import _lib as L
from .fused_mlp import fp16_variant, pack_weight

HID, KP = 128, 48


def supports(mlp, dim_in=None):
    """True when `mlp` is the SDF-shaped VanillaMLP the fused kernels are built for."""
    return (getattr(mlp, "sphere_init", False) and mlp.n_hidden_layers == 2 and mlp.n_neurons == HID
            and (dim_in or mlp.dim_in) <= KP and mlp.dim_out <= KP)


def _net_struct(W1, b1, W2, b2, W3, b3):
    keep = [pack_weight(W1, HID, KP), pack_weight(W2, HID, HID), pack_weight(W3, KP, HID),
            b1.detach().contiguous().float(), b2.detach().contiguous().float(), b3.detach().contiguous().float(),
            W3.detach()[0].contiguous().float()]
    c = L.SdfMlpC()
    c.w1_blob, c.w2_blob, c.w3_blob = (k.data_ptr() for k in keep[:3])
    c.b1, c.b2, c.b3, c.w3_row0 = (k.data_ptr() for k in keep[3:])
    c.n_in, c.n_out = W1.shape[1], W3.shape[0]
    c.precision = fp16_variant()
    return c, keep


def _forward(net, in0, scale0, shift0, in1, out, sdf, g0a=None, g0b=None):
    """Launch the forward of S > 0 samples: sdf-only (out is None) in fp32 on the TMEM-operand kernel
    (rsdf_sdf_mlp_eval), everything else on rsdf_sdf_mlp_fwd.  Measured at 3.34 M evaluations on a B200 (DESIGN.md
    §4): sdf-only 0.79 ms on the TMEM-operand kernel vs 1.14 ms on the shared-memory-operand one; the full 48-wide
    output 1.50 vs 1.38 ms."""
    S, w0 = in0.shape
    w1 = 0 if in1 is None else in1.shape[1]
    if out is None and not net.precision:
        L.call("rsdf_sdf_mlp_eval", ctypes.byref(net), L.ptr(in0), w0, float(scale0), float(shift0), L.ptr(in1), w1, S,
               L.ptr(sdf), L.stream())
    else:
        L.call("rsdf_sdf_mlp_fwd", ctypes.byref(net), L.ptr(in0), w0, float(scale0), float(shift0), L.ptr(in1), w1, S,
               L.ptr(out), L.ptr(sdf), L.ptr(g0a), L.ptr(g0b), L.stream())


def _absmax(tensors, dev):
    """Device scalar (int32 bits of a float) = max |x| over the given tensors (None entries skipped)."""
    amax = torch.empty(1, device=dev, dtype=torch.int32)
    ts = [t for t in tensors if t is not None]
    for i in range(0, max(len(ts), 1), 2):
        a = ts[i] if i < len(ts) else None
        b = ts[i + 1] if i + 1 < len(ts) else None
        L.call("rsdf_absmax2", L.ptr(a), 0 if a is None else a.numel(), L.ptr(b), 0 if b is None else b.numel(),
               L.ptr(amax), 1 if i else 0, L.stream())
    return amax


class _FusedSDF(torch.autograd.Function):
    """(in0, in1, W1..b3) -> (out [S,n_out], sdf [S] = out[:,0], g0a [S,w0], g0b [S,w1]).  sdf and the two
    halves of g0 are separate outputs so that no slice/select backward (zero-fill + copy + add over
    [S,48] / [S,35]) appears in the graph: the backward kernel takes the four cotangents directly."""

    @staticmethod
    def forward(ctx, in0, in1, W1, b1, W2, b2, W3, b3, scale0, shift0, want_g0, sdf_only=False):
        L.require_cuda(in0, in1, W1)
        in0 = in0.contiguous().float()
        in1 = None if in1 is None else in1.contiguous().float()
        S, w0 = in0.shape
        w1 = 0 if in1 is None else in1.shape[1]
        dev = in0.device
        net, keep = _net_struct(W1, b1, W2, b2, W3, b3)
        # sdf_only (the six finite-difference neighbours of the split-sum config, models/geometry.py:229-240): only
        # out[:, 0] is wanted -- the 48-wide output is neither written here nor read back as a (zero) cotangent
        sdf_only = bool(sdf_only) and not want_g0
        out = None if sdf_only else torch.empty(S, W3.shape[0], device=dev, dtype=torch.float32)
        sdf = torch.empty(S, device=dev, dtype=torch.float32)
        g0a = torch.empty(S, w0, device=dev, dtype=torch.float32) if want_g0 else None
        g0b = torch.empty(S, w1, device=dev, dtype=torch.float32) if (want_g0 and w1) else None
        if S:
            _forward(net, in0, scale0, shift0, in1, out, sdf, g0a, g0b)
        ctx.save_for_backward(in0, in1, W1, b1, W2, b2, W3, b3)
        ctx.net, ctx.keep, ctx.scale0, ctx.shift0, ctx.want_g0 = net, keep, float(scale0), float(shift0), bool(want_g0)
        empty = []
        if out is None:
            out = in0.new_zeros(0); empty.append(out)
        if g0a is None:
            g0a = in0.new_zeros(0); empty.append(g0a)
        if g0b is None:
            g0b = in0.new_zeros(0); empty.append(g0b)
        if empty:
            ctx.mark_non_differentiable(*empty)
        return out, sdf, g0a, g0b

    @staticmethod
    def _backward_twice_differentiable(ctx, g_out, g_sdf, g_g0a, g_g0b):
        """The backward under `create_graph=True`: the curvature probe of models/geometry.py:246-282 takes
        `autograd.grad(sdf_t, points_t, create_graph=True)` through this node and then differentiates that gradient
        again (w.r.t. the weights AND the probe position), which the one-kernel backward cannot offer.  The same
        quantities are rebuilt here from differentiable primitives -- tcgen05 streaming GEMMs that are closed under
        differentiation (tc_autograd) + torch elementwise ops -- so that autograd can recurse as it does through the
        reference's nn.Linear stack.  (`once_differentiable` would not do: it only raises when a COTANGENT requires
        grad, and silently returns constants for the `ones_like(sdf)` cotangent of the probe.)"""
        import torch.nn.functional as F

        from . import tc_autograd as tca
        in0, in1, W1, b1, W2, b2, W3, b3 = ctx.saved_tensors
        w0 = in0.shape[1]
        with torch.enable_grad():
            h0 = in0 * ctx.scale0 + ctx.shift0
            if in1 is not None:
                h0 = torch.cat([h0, in1], -1)
            z1 = tca.linear(h0, W1, b1)
            a1 = F.softplus(z1, beta=100)
            z2 = tca.linear(a1, W2, b2)
            a2 = F.softplus(z2, beta=100)
            out = tca.linear(a2, W3, b3)
            outs, cots = [], []
            if g_out is not None:
                outs.append(out); cots.append(g_out)
            if g_sdf is not None:
                outs.append(out[:, 0]); cots.append(g_sdf)
            has_a = g_g0a is not None and g_g0a.numel() > 0
            has_b = g_g0b is not None and g_g0b.numel() > 0
            if ctx.want_g0 and (has_a or has_b):
                # softplus' with torch's threshold rule (aten softplus_backward): sigmoid(beta z), 1 above beta z = 20
                sp1 = torch.where(z1 * 100.0 > 20.0, torch.ones_like(z1), torch.sigmoid(z1 * 100.0))
                sp2 = torch.where(z2 * 100.0 > 20.0, torch.ones_like(z2), torch.sigmoid(z2 * 100.0))
                u1 = sp1 * tca.mm_nn(sp2 * W3[0], W2)
                g0 = tca.mm_nn(u1, W1)
                if has_a:
                    outs.append(g0[:, :w0]); cots.append(g_g0a)
                if has_b:
                    outs.append(g0[:, w0:]); cots.append(g_g0b)
            tensors = (in0, in1, W1, b1, W2, b2, W3, b3)
            idx = [i for i, t in enumerate(tensors) if t is not None and ctx.needs_input_grad[i] and t.requires_grad]
            grads = [None] * 8
            if outs and idx:
                got = torch.autograd.grad(outs, [tensors[i] for i in idx], cots, create_graph=True, allow_unused=True)
                for i, g in zip(idx, got):
                    grads[i] = g
        return (*grads, None, None, None, None)

    @staticmethod
    def backward(ctx, g_out, g_sdf, g_g0a, g_g0b):
        if torch.is_grad_enabled():            # create_graph=True: the caller differentiates this backward again
            return _FusedSDF._backward_twice_differentiable(ctx, g_out, g_sdf, g_g0a, g_g0b)
        in0, in1, W1, b1, W2, b2, W3, b3 = ctx.saved_tensors
        S, w0 = in0.shape
        w1 = 0 if in1 is None else in1.shape[1]
        dev = in0.device
        prep = lambda g: None if (g is None or g.numel() == 0) else g.contiguous().float()
        g_out, g_sdf, g_g0a, g_g0b = prep(g_out), prep(g_sdf), prep(g_g0a), prep(g_g0b)
        if g_out is None and g_sdf is None:
            g_sdf = torch.zeros(S, device=dev, dtype=torch.float32)
        g_in0 = torch.empty(S, w0, device=dev, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        g_in1 = torch.empty(S, w1, device=dev, dtype=torch.float32) if (ctx.needs_input_grad[1] and w1) else None
        gW1, gb1, gW2, gb2 = torch.zeros_like(W1), torch.zeros_like(b1), torch.zeros_like(W2), torch.zeros_like(b2)
        gW3, gb3 = torch.zeros_like(W3), torch.zeros_like(b3)
        if S:
            amax = _absmax([g_out, g_sdf, g_g0a, g_g0b], dev)
            L.call("rsdf_sdf_mlp_bwd", ctypes.byref(ctx.net), L.ptr(in0), w0, ctx.scale0, ctx.shift0, L.ptr(in1), w1, S,
                   L.ptr(g_out), L.ptr(g_sdf), L.ptr(g_g0a), L.ptr(g_g0b), L.ptr(amax), L.ptr(g_in0), L.ptr(g_in1),
                   L.ptr(gW1), L.ptr(gb1), L.ptr(gW2), L.ptr(gb2), L.ptr(gW3), L.ptr(gb3), L.stream())
        return g_in0, g_in1, gW1, gb1, gW2, gb2, gW3, gb3, None, None, None, None


def fused_sdf_parts(mlp, in0, scale0=1.0, shift0=0.0, in1=None, want_g0=True, sdf_only=False):
    """-> (out [S, dim_out] | None with sdf_only, sdf [S], g0a [S, w0] | None, g0b [S, w1] | None)."""
    (W1, b1), (W2, b2), (W3, b3) = mlp.effective_weights()
    out, sdf, g0a, g0b = _FusedSDF.apply(in0, in1, W1.float(), b1.float(), W2.float(), b2.float(), W3.float(),
                                         b3.float(), scale0, shift0, want_g0, sdf_only)
    if not want_g0:
        return (None if sdf_only else out), sdf, None, None
    return out, sdf, g0a, (g0b if in1 is not None else None)


def fused_sdf(mlp, in0, scale0=1.0, shift0=0.0, in1=None, want_g0=True):
    """-> (out [S, dim_out], g0 [S, dim_in] or None).  `mlp`: a VanillaMLP for which supports() holds."""
    out, _, g0a, g0b = fused_sdf_parts(mlp, in0, scale0, shift0, in1, want_g0)
    if not want_g0:
        return out, None
    return out, (g0a if g0b is None else torch.cat([g0a, g0b], -1))


class PackedSDF:
    """Inference-side cache of the packed weight images of an SDF-shaped VanillaMLP (re-packed when a
    parameter changes); runs the forward kernel without autograd.  Used by the eval / relighting render,
    the occupancy update and the finite-difference evaluations (7 per sample in the split-sum config)."""

    def __init__(self, mlp):
        self.mlp, self._key, self._net, self._keep = mlp, None, None, None

    def _struct(self):
        key = tuple((p.data_ptr(), p._version) for p in self.mlp.parameters()) + (fp16_variant(),)
        if key != self._key:
            with torch.no_grad():
                (W1, b1), (W2, b2), (W3, b3) = self.mlp.effective_weights()
                self._net, self._keep = _net_struct(W1.float(), b1.float(), W2.float(), b2.float(), W3.float(), b3.float())
            self._key = key
        return self._net

    @torch.no_grad()
    def __call__(self, in0, scale0=1.0, shift0=0.0, in1=None, sdf_only=False):
        """out [S, dim_out] (or just sdf [S] = out[:, 0] with sdf_only) for h0 = cat(in0 * scale0 + shift0, in1)."""
        L.require_cuda(in0, in1)
        in0 = in0.contiguous().float()
        in1 = None if in1 is None else in1.contiguous().float()
        S = in0.shape[0]
        out = None if sdf_only else torch.empty(S, self.mlp.dim_out, device=in0.device, dtype=torch.float32)
        sdf = torch.empty(S, device=in0.device, dtype=torch.float32) if sdf_only else None
        if S:
            _forward(self._struct(), in0, scale0, shift0, in1, out, sdf)
        return sdf if sdf_only else out
