"""Host side of K3: run a `VanillaMLP` (models/network_utils.py:109-157) through the fused
tcgen05 forward kernel (`rsdf_mlp_fwd`).  Weight-norm is folded on the host (tiny tensors), the
effective weights are split into bf16 hi/lo "tile image" blobs by `rsdf_mlp_pack_weight`, and the
blobs are cached until a parameter changes.  Inference only (no autograd): used by the eval /
relighting render, occupancy-grid updates and secondary-ray shading.
"""
import ctypes

import torch

from . import _lib as L

ACT = {"none": 0, "relu": 1, "softplus100": 2, "sigmoid": 3}
MAX_LAYERS = 8


class _Layer(ctypes.Structure):
    _fields_ = [("blob", ctypes.c_void_p), ("bias", ctypes.c_void_p), ("n", ctypes.c_int32),
                ("n_pad", ctypes.c_int32), ("k_pad", ctypes.c_int32), ("act", ctypes.c_int32)]


class _Params(ctypes.Structure):
    _fields_ = [("n_layers", ctypes.c_int32), ("n_in", ctypes.c_int32), ("n_samples", ctypes.c_int32),
                ("out_w", ctypes.c_int32), ("layer", _Layer * MAX_LAYERS), ("inp", ctypes.c_void_p * 3),
                ("in_w", ctypes.c_int32 * 3), ("in_scale", ctypes.c_float * 3), ("in_shift", ctypes.c_float * 3),
                ("out", ctypes.c_void_p)]


def pad16(n):
    return (n + 15) // 16 * 16


def fp16_variant():
    """1 when VanillaMLP.mlp_precision selects the reduced-precision variant of the sdf_field and relu_mlp kernels
    (single fp16 plane, one product per GEMM), else 0."""
    from .network_utils import VanillaMLP
    return 1 if VanillaMLP.mlp_precision == "fp16" else 0


def pack_weight(W, n_pad=None, k_pad=None):
    """fp32 [N,K] (CUDA) -> uint8 blob of 4*N_pad*K_pad bytes (pads default to the next multiple of 16)."""
    W = W.detach().contiguous().float()
    N, K = W.shape
    n_pad, k_pad = n_pad or pad16(N), k_pad or pad16(K)
    assert n_pad >= N and k_pad >= K and n_pad % 16 == 0 and k_pad % 16 == 0
    blob = torch.empty(4 * n_pad * k_pad, dtype=torch.uint8, device=W.device)
    L.call("rsdf_mlp_pack_weight", L.ptr(W), N, K, n_pad, k_pad, L.ptr(blob), L.stream())
    return blob


class PackedMLP:
    """Blob cache + launcher for one VanillaMLP."""

    def __init__(self, mlp, out_act="none"):
        self.mlp = mlp
        self.out_act = out_act
        self._key = None
        self._layers = None

    def _version_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.mlp.parameters())

    def layers(self):
        key = self._version_key()
        if key != self._key:
            with torch.no_grad():
                ws = self.mlp.effective_weights()
                hidden = self.mlp.activation_name
                self._layers = []
                for i, (W, b) in enumerate(ws):
                    last = i == len(ws) - 1
                    self._layers.append((pack_weight(W), b.detach().contiguous().float(), W.shape[0], W.shape[1],
                                         ACT[self.out_act] if last else ACT[hidden]))
            self._key = key
        return self._layers

    @torch.no_grad()
    def __call__(self, inputs, scales=None, shifts=None):
        """inputs: list of up to 3 fp32 CUDA tensors [S, w_i]; returns [S, dim_out]."""
        if isinstance(inputs, torch.Tensor):
            inputs = [inputs]
        L.require_cuda(*inputs)
        inputs = [t.contiguous().float() for t in inputs]
        S = inputs[0].shape[0]
        layers = self.layers()
        if len(layers) > MAX_LAYERS or len(inputs) > 3:
            raise ValueError("fused MLP supports <= 8 layers and <= 3 input segments")
        out_w = layers[-1][2]
        out = torch.empty(S, out_w, device=inputs[0].device, dtype=torch.float32)
        if S == 0:
            return out
        p = _Params()
        p.n_layers, p.n_in, p.n_samples, p.out_w = len(layers), len(inputs), S, out_w
        p.out = out.data_ptr()
        for i, (blob, bias, n, k, act) in enumerate(layers):
            p.layer[i] = _Layer(blob.data_ptr(), bias.data_ptr(), n, pad16(n), pad16(k), act)
        for g, t in enumerate(inputs):
            p.inp[g] = t.data_ptr()
            p.in_w[g] = t.shape[1]
            p.in_scale[g] = 1.0 if scales is None else float(scales[g])
            p.in_shift[g] = 0.0 if shifts is None else float(shifts[g])
        if sum(t.shape[1] for t in inputs) != layers[0][3]:
            raise ValueError("input widths do not match the first layer")
        L.call("rsdf_mlp_fwd", ctypes.byref(p), L.stream())
        return out
