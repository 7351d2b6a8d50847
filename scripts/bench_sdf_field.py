"""Fused SDF-field MLP kernels: time per call at a training-step sample count."""
import sys, ctypes
import torch
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests')
from rise_sdf_b200 import _lib as L, sdf_field
from test_gpu_sdf_field import make_mlp

S = int(sys.argv[1]) if len(sys.argv) > 1 else 3340000
m = make_mlp()
x01 = torch.rand(S, 3, device='cuda'); enc = torch.randn(S, 32, device='cuda') * 0.1
(W1, b1), (W2, b2), (W3, b3) = [(w.detach(), b.detach()) for w, b in m.effective_weights()]
net, keep = sdf_field._net_struct(W1, b1, W2, b2, W3, b3)
out = torch.empty(S, 48, device='cuda'); g0a = torch.empty(S, 3, device='cuda'); g0b = torch.empty(S, 32, device='cuda')
go = torch.randn(S, 48, device='cuda'); gg = torch.randn(S, 35, device='cuda'); gga = gg[:, :3].contiguous(); ggb = gg[:, 3:].contiguous(); gin0 = torch.empty(S, 3, device='cuda'); gin1 = torch.empty(S, 32, device='cuda')
gW1, gb1, gW2, gb2, gW3, gb3 = [torch.zeros_like(t) for t in (W1, b1, W2, b2, W3, b3)]
st = L.stream()
amax = torch.empty(1, device='cuda', dtype=torch.int32)
L.call("rsdf_absmax2", L.ptr(go), go.numel(), L.ptr(gg), gg.numel(), L.ptr(amax), 0, st)
def t(name, fn, flops_per_sample, reps=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    print(f"{name:20s} {ms:8.3f} ms  {S / ms / 1e3:8.1f} Msamples/s  {flops_per_sample * S / ms / 1e9:7.1f} TFLOP/s fp32-equivalent")
f_fwd = 2 * (35 * 128 + 128 * 128 + 128 * 48)
f_chain = 2 * (128 * 128 + 128 * 35)
t("fwd (out only)", lambda: L.call("rsdf_sdf_mlp_fwd", ctypes.byref(net), L.ptr(x01), 3, 2.0, -1.0, L.ptr(enc), 32, S, L.ptr(out), None, None, None, st), f_fwd)
sdf1 = torch.empty(S, device='cuda')
t("eval TS (sdf only)", lambda: L.call("rsdf_sdf_mlp_eval", ctypes.byref(net), L.ptr(x01), 3, 2.0, -1.0, L.ptr(enc), 32, S, L.ptr(sdf1), st), f_fwd)
t("fwd (out + g0)", lambda: L.call("rsdf_sdf_mlp_fwd", ctypes.byref(net), L.ptr(x01), 3, 2.0, -1.0, L.ptr(enc), 32, S, L.ptr(out), None, L.ptr(g0a), L.ptr(g0b), st), f_fwd + f_chain)
f_bwd = 2 * (35 * 128 + 128 * 128) + f_chain + 2 * (35 * 128 + 128 * 128 + 48 * 128 + 128 * 128 + 128 * 35) + 2 * (2 * 35 * 128 + 2 * 128 * 128 + 48 * 128)
t("absmax2", lambda: L.call("rsdf_absmax2", L.ptr(go), go.numel(), L.ptr(gg), gg.numel(), L.ptr(amax), 0, st), 0)
t("bwd (2nd order)", lambda: L.call("rsdf_sdf_mlp_bwd", ctypes.byref(net), L.ptr(x01), 3, 2.0, -1.0, L.ptr(enc), 32, S, L.ptr(go), None, L.ptr(gga), L.ptr(ggb), L.ptr(amax), L.ptr(gin0), L.ptr(gin1),
                                    L.ptr(gW1), L.ptr(gb1), L.ptr(gW2), L.ptr(gb2), L.ptr(gW3), L.ptr(gb3), st), f_bwd)
