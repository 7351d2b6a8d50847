"""Fused SDF-field MLP kernels (csrc/sdf_train.cu) against an fp64 torch restatement of
models/geometry.py:206-228 + models/network_utils.py:109-157: out, the analytic gradient g0 = d sdf/d h0,
and the full backward (incl. second-order terms) of an arbitrary loss on both."""
import pytest
import torch
import torch.nn.functional as F

from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import sdf_field
from rise_sdf_b200.network_utils import VanillaMLP

pytestmark = pytest.mark.gpu


def make_mlp(dim_in=35, dim_out=48, seed=0):
    torch.manual_seed(seed)
    m = VanillaMLP(dim_in, dim_out, {"n_neurons": 128, "n_hidden_layers": 2, "sphere_init": True,
                                     "weight_norm": True, "output_activation": "none"}).cuda()
    with torch.no_grad():
        m.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
        m.layers[4].weight_v.normal_(0.0, 0.1)         # make every output row matter
        for i in (0, 2, 4):
            m.layers[i].bias.normal_(0.0, 0.02)
    return m


def ref64(m, x01, enc, want_g0=True):
    """fp64: h0 = cat(2 x01 - 1, enc); out = MLP(h0); g0 = d out[:,0] / d h0 (create_graph)."""
    ws = [(W.double(), b.double()) for W, b in m.effective_weights()]
    h0 = torch.cat([x01 * 2 - 1, enc], -1) if enc is not None else x01
    if not h0.requires_grad:
        h0.requires_grad_(True)
    h = h0
    for i, (W, b) in enumerate(ws):
        h = F.linear(h, W, b)
        if i + 1 < len(ws):
            h = F.softplus(h, beta=100)
    g0 = None
    if want_g0:
        (g0,) = torch.autograd.grad(h[:, 0].sum(), h0, create_graph=True)
    return h, g0


def rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max() / max(float(b.abs().max()), 1e-30))


@pytest.mark.parametrize("S", [1, 63, 64, 1000, 148 * 64 * 2 + 17])
def test_forward_and_gradient_chain(S):
    m = make_mlp()
    g = torch.Generator().manual_seed(S)
    x01 = torch.rand(S, 3, generator=g).cuda()
    enc = (torch.randn(S, 32, generator=g) * 0.1).cuda()
    with torch.no_grad():
        out, g0 = sdf_field.fused_sdf(m, x01, 2.0, -1.0, enc)
        out_plain, none = sdf_field.fused_sdf(m, x01, 2.0, -1.0, enc, want_g0=False)
    torch.cuda.synchronize()
    ro, rg = ref64(m, x01.double(), enc.double())
    assert out.shape == (S, 48) and g0.shape == (S, 35) and none is None
    assert rel(out, ro.detach()) <= 2e-6
    assert rel(g0, rg.detach()) <= 5e-6
    assert torch.equal(out, out_plain)


@pytest.mark.parametrize("S,with_g0", [(1000, True), (64 * 148 + 3, True), (5000, False), (77, True)])
def test_backward_first_and_second_order(S, with_g0):
    m = make_mlp(seed=1)
    g = torch.Generator().manual_seed(S)
    x01 = torch.rand(S, 3, generator=g).cuda().requires_grad_(True)
    enc = (torch.randn(S, 32, generator=g) * 0.1).cuda().requires_grad_(True)
    c_out = torch.randn(S, 48, generator=g).cuda() / S
    c_g0 = torch.randn(S, 35, generator=g).cuda() / S

    def loss_of(out, g0):
        l = (out * c_out.to(out)).sum() + (out[:, 0] ** 2).sum() / S
        if with_g0:
            l = l + (g0 * c_g0.to(g0)).sum() + ((g0[:, :3].norm(dim=-1) - 1.0) ** 2).sum() / S
        return l

    params = list(m.parameters())
    out, g0 = sdf_field.fused_sdf(m, x01, 2.0, -1.0, enc, want_g0=with_g0)
    got = torch.autograd.grad(loss_of(out, g0), [x01, enc] + params)
    torch.cuda.synchronize()

    x64 = x01.detach().double().requires_grad_(True)
    e64 = enc.detach().double().requires_grad_(True)
    ro, rg = ref64(m, x64, e64, want_g0=with_g0)
    want = torch.autograd.grad(loss_of(ro, rg), [x64, e64] + params)
    names = ["x01", "enc"] + [n for n, _ in m.named_parameters()]
    for n, a, b in zip(names, got, want):
        assert rel(a, b) <= 2e-5, (n, rel(a, b))


def test_plain_input_segment():
    """One input segment, no affine (the finite-difference evaluations of the split-sum config)."""
    m = make_mlp(seed=2)
    g = torch.Generator().manual_seed(5)
    h0 = (torch.randn(3000, 35, generator=g) * 0.3).cuda().requires_grad_(True)
    c = torch.randn(3000, 48, generator=g).cuda()
    out, _ = sdf_field.fused_sdf(m, h0, want_g0=False)
    got = torch.autograd.grad((out * c).sum(), [h0] + list(m.parameters()))
    h64 = h0.detach().double().requires_grad_(True)
    ro, _ = ref64(m, h64, None, want_g0=False)
    want = torch.autograd.grad((ro * c.double()).sum(), [h64] + list(m.parameters()))
    assert rel(out, ro.detach()) <= 2e-6
    for a, b in zip(got, want):
        assert rel(a, b) <= 2e-5


@pytest.mark.parametrize("S", [1, 63, 64, 65, 127, 128, 129, 257, 148 * 128 + 1, 2 * 148 * 128 + 77])
def test_inference_kernel_out_and_sdf_only(S):
    """PackedSDF: the full output (two-group shared-memory-operand kernel, two segments and one) and the sdf-only
    output (TMEM-operand kernel, output layer replaced by an fp32 dot product) against fp64."""
    m = make_mlp(seed=3)
    g = torch.Generator().manual_seed(S)
    x01 = torch.rand(S, 3, generator=g).cuda()
    enc = (torch.randn(S, 32, generator=g) * 0.1).cuda()
    packed = sdf_field.PackedSDF(m)
    out = packed(x01, 2.0, -1.0, enc)
    sdf = packed(x01, 2.0, -1.0, enc, sdf_only=True)
    h0 = torch.cat([x01 * 2 - 1, enc], -1)
    out1 = packed(h0)                                     # single input segment
    ro, _ = ref64(m, x01.double(), enc.double(), want_g0=False)
    assert out.shape == (S, 48) and sdf.shape == (S,)
    assert rel(out, ro.detach()) <= 2e-6 and rel(out1, ro.detach()) <= 2e-6
    assert float((sdf.double().cpu() - ro[:, 0].detach().cpu()).abs().max()) <= 2e-6 * max(float(ro[:, 0].abs().max()), 1.0)


@pytest.mark.parametrize("want_g0", [False, True])
def test_double_backward_through_the_fused_node(want_g0):
    """The curvature probe of models/geometry.py:246-282: `autograd.grad(sdf, h0, create_graph=True)` THROUGH the fused
    node, then a backward through that gradient to the inputs and every weight (the node's create_graph path:
    sdf_field._FusedSDF._backward_twice_differentiable).  Before round 2 the node was `once_differentiable`, which
    hands back constants for a cotangent that does not require grad: the second-order terms were silently lost."""
    m = make_mlp(seed=4)
    S = 700
    g = torch.Generator().manual_seed(9)
    h0 = (torch.randn(S, 35, generator=g) * 0.3).cuda().requires_grad_(True)
    c = torch.randn(S, 35, generator=g).cuda()
    params = list(m.parameters())

    def probe(out, h):
        (gh,) = torch.autograd.grad(out[:, 0], h, torch.ones_like(out[:, 0]), create_graph=True)
        return (gh * c.to(gh)).sum() + ((gh[:, :3].norm(dim=-1) - 1.0) ** 2).mean() + (out ** 2).mean()

    if want_g0:          # the analytic-normal node, double-differentiated on top of its own g0 output
        out, g0 = sdf_field.fused_sdf(m, h0, want_g0=True)
        l = probe(out, h0) + (g0 ** 2).mean()
    else:
        out, _ = sdf_field.fused_sdf(m, h0, want_g0=False)
        l = probe(out, h0)
    got = torch.autograd.grad(l, [h0] + params)
    h64 = h0.detach().double().requires_grad_(True)
    ro, rg = ref64(m, h64, None, want_g0=want_g0)
    lr = probe(ro, h64) + ((rg ** 2).mean() if want_g0 else 0.0)
    want = torch.autograd.grad(lr, [h64] + params)
    assert abs(float(l) - float(lr)) <= 1e-5 * abs(float(lr))
    for n, a, b in zip(["h0"] + [n for n, _ in m.named_parameters()], got, want):
        assert rel(a, b) <= 5e-5, (n, rel(a, b))


@pytest.mark.parametrize("S", [77, 64 * 148 + 3])
def test_sdf_only_training_node(S):
    """The finite-difference neighbours of the split-sum config only need out[:, 0] (models/geometry.py:229-240): the
    sdf-only node writes no 48-wide output, takes no 48-wide cotangent, and must give the gradients of the full node
    driven through its sdf output (same backward kernel; here also against fp64)."""
    m = make_mlp()
    g = torch.Generator().manual_seed(S)
    x01 = torch.rand(S, 3, generator=g).cuda()
    enc = (torch.randn(S, 32, generator=g) * 0.1).cuda().requires_grad_(True)
    cot = (torch.randn(S, generator=g) / S).cuda()
    res = []
    for sdf_only in (True, False):
        m.zero_grad(set_to_none=True)
        enc.grad = None
        out, sdf, _, _ = sdf_field.fused_sdf_parts(m, x01, 2.0, -1.0, enc, want_g0=False, sdf_only=sdf_only)
        assert (out is None) == sdf_only
        (sdf * cot).sum().backward()
        res.append((sdf.detach(), enc.grad.clone(), [p.grad.clone() for p in m.parameters() if p.grad is not None]))
    (sa, ea, pa), (sb, eb, pb) = res
    ro, _ = ref64(m, x01.double(), enc.detach().double(), want_g0=False)
    assert rel(sa, ro[:, 0].detach()) <= 2e-6 and rel(sb, ro[:, 0].detach()) <= 2e-6
    assert rel(ea, eb) <= 1e-6
    assert len(pa) == len(pb) > 0
    for x, y in zip(pa, pb):
        assert rel(x, y) <= 1e-5


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_forward_kernel_selection(precision, monkeypatch):
    """Which entry point each forward runs: the SDF field's sdf-only output in fp32 on the TMEM-operand kernel, every
    other SDF-field forward on rsdf_sdf_mlp_fwd; VanillaMLP under grad by net shape (fused SDF node, per-layer ReLU
    kernels, tc_autograd GEMMs for any other shape) and under no_grad on the fused inference kernels."""
    monkeypatch.setattr(VanillaMLP, "mlp_precision", precision)
    calls = []
    real = L.call
    monkeypatch.setattr(L, "call", lambda name, *a: (calls.append(name), real(name, *a))[1])

    def run(fn, *a, **k):
        calls.clear()
        fn(*a, **k)
        return [c for c in calls if c not in ("rsdf_mlp_pack_weight", "rsdf_absmax2")]

    sdf_only_kernel = "rsdf_sdf_mlp_eval" if precision == "fp32" else "rsdf_sdf_mlp_fwd"
    m = make_mlp(seed=5)
    g = torch.Generator().manual_seed(5)
    x01 = torch.rand(300, 3, generator=g).cuda()
    enc = (torch.randn(300, 32, generator=g) * 0.1).cuda()
    packed = sdf_field.PackedSDF(m)
    assert run(packed, x01, 2.0, -1.0, enc) == ["rsdf_sdf_mlp_fwd"]
    assert run(packed, x01, 2.0, -1.0, enc, sdf_only=True) == [sdf_only_kernel]
    assert run(sdf_field.fused_sdf_parts, m, x01, 2.0, -1.0, enc, want_g0=False, sdf_only=True) == [sdf_only_kernel]
    assert run(sdf_field.fused_sdf_parts, m, x01, 2.0, -1.0, enc, want_g0=False) == ["rsdf_sdf_mlp_fwd"]

    h0 = torch.cat([x01 * 2 - 1, enc], -1)
    relu = VanillaMLP(67, 3, {"n_neurons": 128, "n_hidden_layers": 4, "output_activation": "none"}).cuda()
    narrow = VanillaMLP(35, 48, {"n_neurons": 64, "n_hidden_layers": 2, "sphere_init": True, "weight_norm": True,
                                 "output_activation": "none"}).cuda()
    segs = [torch.randn(300, 48, device="cuda"), torch.randn(300, 16, device="cuda"), torch.randn(300, 3, device="cuda")]
    assert run(m, h0) == ["rsdf_sdf_mlp_fwd"]
    assert run(relu, torch.cat(segs, -1)) == ["rsdf_relu_layer_fwd"] * 5
    assert run(relu.forward_segments, segs) == ["rsdf_relu_layer_fwd"] * 5
    assert run(narrow, h0) == ["rsdf_mm_stream"] * 3
    with torch.no_grad():
        assert run(m, h0) == ["rsdf_sdf_mlp_fwd"]
        assert run(relu.forward_segments, segs) == ["rsdf_mlp_fwd"]
        assert run(narrow, h0) == ["rsdf_mlp_fwd"]
