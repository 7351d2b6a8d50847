"""K4 parity: scan / accumulate / fused NeuS render vs the C oracle (serial order), the torch
oracle (autograd) and the reference's compiled kernels (through the golden vectors they produced)."""
import glob
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import fields as of
from oracle import march as omarch
from rise_sdf_b200 import nerfacc as rn
from rise_sdf_b200.neus import _NeusRender

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def ragged(n_rays=300, max_len=1024, seed=0, special=True):
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, 70, size=n_rays)
    if special:
        counts[0] = 0; counts[1] = 1; counts[2] = max_len; counts[3] = 32; counts[4] = 33; counts[-1] = 0
    ri = np.repeat(np.arange(n_rays), counts)
    a = rng.uniform(0, 0.6, size=len(ri)).astype(np.float32)
    a[rng.integers(0, len(a), 50)] = 0.0
    a[rng.integers(0, len(a), 5)] = 1.0
    return ri, a, n_rays


def test_docstring_vectors():
    a = torch.tensor([0.4, 0.8, 0.1, 0.8, 0.1, 0.0, 0.9], device="cuda")
    ri = torch.tensor([0, 0, 0, 1, 1, 2, 2], device="cuda")
    w, T = rn.render_weight_from_alpha(a, ray_indices=ri, n_rays=3)
    np.testing.assert_allclose(w.cpu(), [0.4, 0.48, 0.012, 0.8, 0.02, 0.0, 0.9], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(T.cpu(), [1.0, 0.6, 0.12, 1.0, 0.2, 1.0, 1.0], rtol=1e-6)
    vis = rn.render_visibility(a[:, None], ray_indices=ri, n_rays=3, early_stop_eps=0.3, alpha_thre=0.2)
    assert vis.cpu().tolist() == [True, True, False, True, False, False, True]


def test_scan_forward_vs_serial_oracle():
    ri, a, n = ragged()
    pk = omarch.pack_info(ri, n)
    w0, T0 = omarch.weight_from_alpha(pk, a)
    w, T = rn.render_weight_from_alpha(torch.tensor(a).cuda(), ray_indices=torch.tensor(ri).cuda(), n_rays=n)
    # tree-ordered product vs the reference's serial product over up to 1024 factors: the two
    # roundings differ by O(sqrt(n)) ulp -> stated tolerance 1e-5 relative, exact zeros preserved
    np.testing.assert_allclose(T.cpu().numpy(), T0, rtol=1e-5, atol=1e-30)
    np.testing.assert_allclose(w.cpu().numpy(), w0, rtol=1e-5, atol=1e-30)
    assert np.array_equal(T.cpu().numpy() == 0, T0 == 0)


def test_scan_backward_vs_oracles():
    ri, a, n = ragged(special=False)
    a = np.clip(a, 0, 0.95)
    rng = np.random.default_rng(1)
    gw = rng.normal(size=len(a)).astype(np.float32)
    gT = rng.normal(size=len(a)).astype(np.float32)
    at = torch.tensor(a, device="cuda", requires_grad=True)
    w, T = rn.render_weight_from_alpha(at, ray_indices=torch.tensor(ri).cuda(), n_rays=n)
    (w * torch.tensor(gw).cuda()).sum().backward()
    g_w_only = at.grad.clone().cpu().numpy()
    at.grad = None
    w, T = rn.render_weight_from_alpha(at, ray_indices=torch.tensor(ri).cuda(), n_rays=n)
    ((w * torch.tensor(gw).cuda()).sum() + (T * torch.tensor(gT).cuda()).sum()).backward()
    g_both = at.grad.cpu().numpy()
    # float64 autograd oracle
    a64 = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    w64, T64 = of.render_weight_from_alpha(a64, torch.tensor(ri), n)
    (w64 * torch.tensor(gw, dtype=torch.float64)).sum().backward()
    ref_w = a64.grad.clone().numpy(); a64.grad = None
    w64, T64 = of.render_weight_from_alpha(a64, torch.tensor(ri), n)
    ((w64 * torch.tensor(gw, dtype=torch.float64)).sum() + (T64 * torch.tensor(gT, dtype=torch.float64)).sum()).backward()
    ref_both = a64.grad.numpy()
    scale = np.abs(ref_both).max()
    assert np.abs(g_w_only - ref_w).max() <= 1e-5 * max(np.abs(ref_w).max(), 1)
    assert np.abs(g_both - ref_both).max() <= 1e-5 * max(scale, 1)
    # reference kernel formula (serial C oracle)
    pk = omarch.pack_info(ri, n)
    w0, T0 = omarch.weight_from_alpha(pk, a)
    ga0 = omarch.weight_from_alpha_backward(pk, a, w0, gw)
    assert np.abs(g_w_only - ga0).max() <= 2e-4 * max(np.abs(ga0).max(), 1)


@pytest.mark.parametrize("gold", sorted(glob.glob(os.path.join(GOLD, "march_*.npz"))), ids=os.path.basename)
def test_scan_vs_reference_kernels(gold):
    """Against the reference's compiled weight_from_alpha_{forward,backward}_naive and
    transmittance_from_alpha_forward_naive (render_weight.cu:86-154), whose outputs on the marched samples
    are stored in tests/golden/march_*.npz (tests/golden/make_golden.py)."""
    z = np.load(gold)
    pk = torch.from_numpy(z["packed_info"]).cuda()
    at = torch.from_numpy(z["alphas"]).cuda().requires_grad_(True)
    w, T = rn.render_weight_from_alpha(at, packed_info=pk)
    np.testing.assert_allclose(w.detach().cpu().numpy(), z["weights"], rtol=1e-5, atol=1e-30)
    np.testing.assert_allclose(T.detach().cpu().numpy(), z["trans"], rtol=1e-5, atol=1e-30)
    (w * torch.from_numpy(z["grad_weights"]).cuda()).sum().backward()
    ga = z["grad_alphas"]
    assert np.abs(at.grad.cpu().numpy() - ga).max() <= 2e-4 * max(np.abs(ga).max(), 1)


@pytest.mark.parametrize("D", [1, 3, 8, 24])
def test_accumulate_vs_fp64(D):
    ri, a, n = ragged()
    rng = np.random.default_rng(D)
    w = rng.uniform(0, 1, len(ri)).astype(np.float32)
    v = rng.normal(size=(len(ri), D)).astype(np.float32)
    wt = torch.tensor(w, device="cuda", requires_grad=True)
    vt = torch.tensor(v, device="cuda", requires_grad=True)
    out = rn.accumulate_along_rays(wt, vt, ray_indices=torch.tensor(ri).cuda(), n_rays=n)
    assert out.shape == (n, D)
    ref = np.zeros((n, D)); np.add.at(ref, ri, w[:, None].astype(np.float64) * v)
    assert np.abs(out.detach().cpu().numpy() - ref).max() <= 1e-6 * max(np.abs(ref).max(), 1) * 8
    go = rng.normal(size=(n, D)).astype(np.float32)
    (out * torch.tensor(go).cuda()).sum().backward()
    np.testing.assert_allclose(wt.grad.cpu().numpy(), (go[ri] * v).sum(1), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(vt.grad.cpu().numpy(), go[ri] * w[:, None], rtol=1e-6, atol=1e-7)
    o1 = rn.accumulate_along_rays(wt.detach(), None, ray_indices=torch.tensor(ri).cuda(), n_rays=n)
    assert o1.shape == (n, 1)
    np.testing.assert_allclose(o1.cpu().numpy()[:, 0], np.bincount(ri, weights=w.astype(np.float64), minlength=n), rtol=1e-5, atol=1e-6)
    z = rn.accumulate_along_rays(torch.zeros(0, device="cuda"), None, ray_indices=torch.zeros(0, dtype=torch.long, device="cuda"), n_rays=5)
    assert z.shape == (5, 1) and float(z.abs().sum()) == 0


@pytest.mark.parametrize("ratio", [0.0, 0.37, 1.0])
def test_fused_neus_render_fwd_bwd(ratio):
    """Fused alpha+scan+accumulate == the op-by-op torch restatement (models/neus.py:258-277)."""
    rng = np.random.default_rng(3)
    n = 200
    counts = rng.integers(0, 90, size=n); counts[0] = 0; counts[5] = 300
    ri = np.repeat(np.arange(n), counts)
    S = len(ri)
    d = F.normalize(torch.tensor(rng.normal(size=(n, 3)), dtype=torch.float32), dim=-1)
    t0 = torch.tensor(rng.uniform(2, 5, S), dtype=torch.float32)
    t1 = t0 + 0.005
    sdf = torch.tensor(rng.normal(size=S) * 0.05, dtype=torch.float32)
    grad = torch.tensor(rng.normal(size=(S, 3)), dtype=torch.float32)
    rgb = torch.tensor(rng.uniform(size=(S, 3)), dtype=torch.float32)
    inv_s = torch.tensor(20.0855)
    go = torch.tensor(rng.normal(size=(n, 8)), dtype=torch.float32)
    gwx = torch.tensor(rng.normal(size=S), dtype=torch.float32)

    def ref(dtype):
        ins = [x.to(dtype).clone().requires_grad_(True) for x in (sdf, grad, rgb, inv_s)]
        s_, g_, c_, i_ = ins
        rit = torch.tensor(ri)
        normal = F.normalize(g_, p=2, dim=-1)
        alpha = of.get_alpha(s_, normal, d.to(dtype)[rit], (t1 - t0).to(dtype), i_.view(1, 1), ratio)
        w, _ = of.render_weight_from_alpha(alpha, rit, n)
        mid = ((t0 + t1)[:, None] / 2.0).to(dtype)
        out = torch.cat([of.accumulate_along_rays(w, c_, rit, n), of.accumulate_along_rays(w, normal, rit, n),
                         of.accumulate_along_rays(w, None, rit, n), of.accumulate_along_rays(w, mid, rit, n)], -1)
        ((out * go.to(dtype)).sum() + (w * gwx.to(dtype)).sum()).backward()
        return out.detach(), w.detach(), [x.grad for x in ins]

    out_r, w_r, g_r = ref(torch.float64)
    ins = [x.cuda().clone().requires_grad_(True) for x in (sdf, grad, rgb, inv_s)]
    pk = torch.tensor(omarch.pack_info(ri, n)).cuda()
    out, w, alpha = _NeusRender.apply(pk, d.cuda().contiguous(), t0.cuda(), t1.cuda(), ins[0], ins[1], ins[2], ins[3], ratio)
    ((out * go.cuda()).sum() + (w * gwx.cuda()).sum()).backward()
    assert np.abs(out.detach().cpu().numpy() - out_r.numpy()).max() <= 2e-5 * max(float(out_r.abs().max()), 1)
    assert np.abs(w.detach().cpu().numpy() - w_r.numpy()).max() <= 2e-6
    for got, want, name in zip([x.grad for x in ins], g_r, ["sdf", "grad", "rgb", "inv_s"]):
        want = want.numpy()
        err = np.abs(got.cpu().numpy() - want).max()
        assert err <= 2e-4 * max(np.abs(want).max(), 1e-3), (name, err, np.abs(want).max())


def test_sample_setup_normalize_and_sdf_regularisers_match_torch():
    """The single-launch glue ops against the torch expressions they replace (models/neus.py:247-256,
    systems/neus.py:117-131): sample set-up bit-exact, normalisation / regularisers to fp32 rounding,
    including their gradients."""
    import torch.nn.functional as F
    from rise_sdf_b200.neus import normalize3, sample_setup
    from rise_sdf_b200.train import sdf_regularisers
    g = torch.Generator().manual_seed(3)
    R, S = 300, 20000
    rays_o = torch.randn(R, 3, generator=g).cuda(); rays_d = F.normalize(torch.randn(R, 3, generator=g), dim=-1).cuda()
    ri = torch.sort(torch.randint(0, R, (S,), generator=g)).values.cuda()
    t0 = (torch.rand(S, generator=g) * 4).cuda(); t1 = t0 + 0.005
    pos, dirs, mid, dists = sample_setup(rays_o, rays_d, ri, t0, t1)
    mid_ref = (t0 + t1)[..., None] / 2.0
    assert torch.equal(mid, mid_ref) and torch.equal(dirs, rays_d[ri]) and torch.equal(dists, t1 - t0)
    assert torch.equal(pos, rays_o[ri] + rays_d[ri] * mid_ref)

    v = (torch.randn(S, 3, generator=g) * 0.7).cuda(); v[:3] = 0.0
    sdf = torch.randn(S, generator=g).cuda(); sdf[5] = 0.0
    c = torch.randn(S, 3, generator=g).cuda()
    va = v.clone().requires_grad_(True); vb = v.clone().double().requires_grad_(True)
    (ga,) = torch.autograd.grad((normalize3(va) * c).sum(), va)
    (gb,) = torch.autograd.grad((F.normalize(vb, p=2, dim=-1) * c.double()).sum(), vb)
    assert float((normalize3(v).double() - F.normalize(v.double(), dim=-1)).abs().max()) <= 1e-6
    assert float((ga.double() - gb)[3:].abs().max()) <= 1e-5 * float(gb[3:].abs().max())

    va = v.clone().requires_grad_(True); sa = sdf.clone().requires_grad_(True)
    e, s = sdf_regularisers(va, sa, 1.3)
    ga, gs = torch.autograd.grad(0.1 * e + 0.01 * s, [va, sa])
    vb = v.clone().double().requires_grad_(True); sb = sdf.clone().double().requires_grad_(True)
    e_ref = ((torch.linalg.norm(vb, ord=2, dim=-1) - 1.0) ** 2).mean(); s_ref = torch.exp(-1.3 * sb.abs()).mean()
    gb, gsb = torch.autograd.grad(0.1 * e_ref + 0.01 * s_ref, [vb, sb])
    assert abs(float(e) - float(e_ref)) <= 1e-5 * float(e_ref) and abs(float(s) - float(s_ref)) <= 1e-5 * float(s_ref)
    assert float((ga.double() - gb)[3:].abs().max()) <= 1e-5 * float(gb.abs().max())
    assert float((gs.double() - gsb).abs().max()) <= 1e-5 * float(gsb.abs().max())
