"""Host side of the per-layer ReLU-MLP training kernels (csrc/relu_mlp.cu): `VanillaMLP`s with ReLU
hidden layers of width 128 (models/network_utils.py:109-157; the radiance / albedo / roughness /
metallic / env / secondary networks of models/texture.py) as ONE autograd node.

    out = relu_mlp(mlp, [in0, in1, in2])        # input = cat(segments), out [S, dim_out <= 16], no output act.

Forward: one launch per layer; the activations between layers live in HBM as fp16 hi/lo operand-image
streams (kept for the backward).  Backward: rsdf_absmax2 + one launch per layer, top down.  The node is
once-differentiable (the reference never differentiates the texture networks twice).
"""
import ctypes

import torch

from . import _lib as L
from .fused_mlp import fp16_variant, pack_weight, pad16

NS = 64
HID = 128


def supports(mlp, n_in=None):
    return (not getattr(mlp, "sphere_init", False) and mlp.n_neurons == HID and mlp.n_hidden_layers >= 1
            and (n_in or mlp.dim_in) <= 128 and mlp.dim_out <= 16)


def _stream(n_tiles, rows, device, fp16=0):
    """operand-image stream: per 64-sample tile an fp16 hi|lo pair of [rows x 64] planes (one plane in the fp16 variant)"""
    return torch.empty(n_tiles, (1 if fp16 else 2) * rows * 128, dtype=torch.uint8, device=device)


class _ReluMLP(torch.autograd.Function):
    @staticmethod
    def forward(ctx, n_seg, scales, shifts, *args):
        segs = [a.contiguous().float() for a in args[:n_seg]]
        params = [a.float().contiguous() for a in args[n_seg:]]          # W1, b1, ..., W_{L+1}, b_{L+1}
        L.require_cuda(*segs)
        Ws, bs = params[0::2], params[1::2]
        S = segs[0].shape[0]
        dev = segs[0].device
        n_in = sum(s.shape[1] for s in segs)
        n_out = Ws[-1].shape[0]
        k0 = pad16(n_in)
        n_tiles = (S + NS - 1) // NS
        out = torch.empty(S, n_out, device=dev, dtype=torch.float32)
        blobs = [pack_weight(W, HID if i + 1 < len(Ws) else 16, k0 if i == 0 else HID) for i, W in enumerate(Ws)]
        acts = []                                                        # a_0 (input image stream), a_1, ..., a_L
        fp16 = ctx.fp16 = fp16_variant()
        if S:
            a0 = _stream(n_tiles, k0, dev, fp16)
            acts.append(a0)
            for i in range(len(Ws) - 1):
                p = L.ReluFwdC()
                p.w, p.bias = blobs[i].data_ptr(), bs[i].data_ptr()
                p.r_pad, p.r_real, p.k_pad, p.n_samples, p.fp16 = HID, HID, (k0 if i == 0 else HID), S, fp16
                a_out = _stream(n_tiles, HID, dev, fp16)
                if i == 0:
                    for g, sg in enumerate(segs):
                        p.inp[g], p.in_w[g] = sg.data_ptr(), sg.shape[1]
                        p.in_scale[g], p.in_shift[g] = float(scales[g]), float(shifts[g])
                    p.n_in, p.a0_save = n_in, a0.data_ptr()
                else:
                    p.a_in = acts[-1].data_ptr()
                p.a_out = a_out.data_ptr()
                L.call("rsdf_relu_layer_fwd", ctypes.byref(p), L.stream())
                acts.append(a_out)
            p = L.ReluFwdC()
            p.w, p.bias = blobs[-1].data_ptr(), bs[-1].data_ptr()
            p.r_pad, p.r_real, p.k_pad, p.n_samples, p.fp16 = 16, n_out, HID, S, fp16
            p.a_in, p.rows_out = acts[-1].data_ptr(), out.data_ptr()
            L.call("rsdf_relu_layer_fwd", ctypes.byref(p), L.stream())
        ctx.n_seg, ctx.scales, ctx.seg_w = n_seg, [float(s) for s in scales], [s.shape[1] for s in segs]
        ctx.blobs, ctx.acts, ctx.S, ctx.k0, ctx.n_in = blobs, acts, S, k0, n_in
        ctx.save_for_backward(*params)
        return out

    @staticmethod
    def backward(ctx, g_out):
        if torch.is_grad_enabled():
            # `once_differentiable` only raises when the cotangent requires grad and otherwise hands back constants:
            # a caller differentiating through this backward (create_graph=True) would silently lose terms.  Nothing
            # on the render path does (the texture nets are first order), so refuse loudly.
            raise NotImplementedError("relu_mlp is first-order only: build a network that must be differentiated "
                                      "twice from tc_autograd.linear, which is closed under differentiation")
        params = ctx.saved_tensors
        Ws, bs = params[0::2], params[1::2]
        S, dev = ctx.S, g_out.device
        n_out = Ws[-1].shape[0]
        gWs = [torch.zeros_like(W) for W in Ws]
        gbs = [torch.zeros_like(b) for b in bs]
        g_segs = [torch.empty(S, w, device=dev, dtype=torch.float32) if ctx.needs_input_grad[3 + g] else None
                  for g, w in enumerate(ctx.seg_w)]
        if S:
            g_out = g_out.contiguous().float()
            n_tiles = (S + NS - 1) // NS
            amax = torch.empty(1, device=dev, dtype=torch.int32)
            L.call("rsdf_absmax2", L.ptr(g_out), g_out.numel(), None, 0, L.ptr(amax), 0, L.stream())
            zb = None
            for i in range(len(Ws) - 1, -1, -1):
                p = L.ReluBwdC()
                head, first = i == len(Ws) - 1, i == 0
                p.w = ctx.blobs[i].data_ptr()
                p.r_pad, p.r_real = (16, n_out) if head else (HID, HID)
                p.k_pad, p.k_real = (ctx.k0, ctx.n_in) if first else (HID, HID)
                p.n_samples, p.amax, p.a_in, p.fp16 = S, amax.data_ptr(), ctx.acts[i].data_ptr(), ctx.fp16
                if head:
                    p.g_rows, p.gb_self = g_out.data_ptr(), gbs[i].data_ptr()
                else:
                    p.zb_in = zb.data_ptr()
                if first:
                    p.first_layer = 1
                    for g, w in enumerate(ctx.seg_w):
                        p.seg_w[g], p.seg_scale[g] = w, ctx.scales[g]
                        p.rows_out[g] = None if g_segs[g] is None else g_segs[g].data_ptr()
                else:
                    zb_next = _stream(n_tiles, HID, dev, ctx.fp16)
                    p.zb_out, p.gb_prev = zb_next.data_ptr(), gbs[i - 1].data_ptr()
                p.gW = gWs[i].data_ptr()
                L.call("rsdf_relu_layer_bwd", ctypes.byref(p), L.stream())
                if not first:
                    zb = zb_next
        ctx.acts = None
        g_params = []
        for gW, gb in zip(gWs, gbs):
            g_params += [gW, gb]
        return (None, None, None, *g_segs, *g_params)


def relu_mlp(mlp, segments, scales=None, shifts=None):
    """mlp: VanillaMLP for which supports() holds; segments: list of <= 3 [S, w_i] CUDA tensors."""
    if isinstance(segments, torch.Tensor):
        segments = [segments]
    n = len(segments)
    scales = list(scales) if scales is not None else [1.0] * n
    shifts = list(shifts) if shifts is not None else [0.0] * n
    flat = []
    for W, b in mlp.effective_weights():
        flat += [W, b]
    return _ReluMLP.apply(n, scales, shifts, *segments, *flat)
