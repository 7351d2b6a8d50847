"""Test-stage metrics on the B200 (csrc/metrics.cu, rise_sdf_b200/metrics.py, relight.evaluate_frame): every metric
against the float64 oracle (oracle/metrics.py) within 1e-10, the median ratio bit-identical to torch.median, repeated
calls bit-identical, argument checks, no host synchronisation, and the evaluation driver end to end on the small
split-sum model."""
import numpy as np
import pytest
import torch

from oracle import metrics as om
from rise_sdf_b200 import metrics

pytestmark = pytest.mark.gpu

TOL = 1e-10
# 11x11: one valid pixel; 11x800: one valid row; odd sizes and sizes that are no multiple of the 16 x 32 SSIM tile
SHAPES = [(11, 11, 1), (11, 11, 3), (11, 800, 3), (800, 11, 1), (37, 53, 1), (45, 97, 3), (130, 67, 4), (800, 800, 3)]


def _pair(shape, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g)
    y = (x + 0.1 * torch.randn(shape, generator=g)).clamp(0, 1)
    return x, y


def _masks(H, W, seed):
    g = torch.Generator().manual_seed(seed)
    single = torch.zeros(H, W, dtype=torch.bool)
    single[H // 2, W // 3] = True
    return {"full": torch.ones(H, W, dtype=torch.bool), "sparse": torch.rand(H, W, generator=g) < 0.05,
            "single": single, "empty": torch.zeros(H, W, dtype=torch.bool)}


def _close(got, want):
    got = float(got)
    if np.isnan(want):
        return np.isnan(got)
    if np.isinf(want):
        return got == want
    return abs(got - want) <= TOL


@pytest.mark.parametrize("shape", SHAPES)
def test_psnr_and_ssim_match_oracle(shape):
    x, y = _pair(shape, sum(shape))
    xc, yc = x.cuda(), y.cuda()
    xn, yn = x.numpy(), y.numpy()
    assert _close(metrics.psnr(xc, yc), om.psnr(xn, yn))
    for name, m in _masks(*shape[:2], 7).items():
        got, want = metrics.psnr(xc, yc, m.cuda()), om.psnr(xn, yn, m.numpy())
        assert got.dim() == 0 and got.is_cuda
        assert _close(got, want), (name, float(got), want)
    got, want = metrics.ssim(xc, yc), om.ssim(xn, yn)
    assert got.dim() == 0 and _close(got, want), (float(got), want)
    assert float(metrics.psnr(xc, xc)) == float("inf")
    assert abs(float(metrics.ssim(xc, xc)) - 1.0) <= 1e-12


@pytest.mark.parametrize("shape", [(11, 11), (37, 53), (130, 67), (800, 800)])
def test_normal_mae_matches_oracle(shape):
    H, W = shape
    g = torch.Generator().manual_seed(H * W)
    a = torch.randn(H, W, 3, generator=g)
    b = a * (0.5 + torch.rand(H, W, 1, generator=g)) + torch.randn(H, W, 3, generator=g) * 10.0 ** torch.randint(
        -6, 0, (H, W, 1), generator=g)                       # angles from ~1e-4 degrees up to tens of degrees
    a[0, 0] = 0.0                                            # a zero vector (90 degrees whatever the other is)
    a[1, 0], b[1, 0] = 0.0, torch.tensor([-1.0, -2.0, 0.5])   # a . b = -0 there: atan2 alone would give 180
    b[-1, -1] = -a[-1, -1]                                   # antiparallel
    for name, m in _masks(H, W, 3).items():
        got, want = metrics.normal_mae(a.cuda(), b.cuda(), m.cuda()), om.normal_mae(a.numpy(), b.numpy(), m.numpy())
        assert got.dim() == 0 and _close(got, want), (name, float(got), want)


def _torch_median(pred, gt, mask, eps=1e-6):
    r = gt[mask] / pred[mask].clamp(min=eps)
    return torch.stack([torch.median(r[:, c]) for c in range(r.shape[1])]) if r.shape[0] else \
        torch.full((pred.shape[-1],), float("nan"), device=pred.device)


def _same_bits(got, want):
    got, want = got.cpu(), want.cpu()
    nan = torch.isnan(want)
    return torch.equal(torch.isnan(got), nan) and torch.equal(got[~nan].view(torch.int32), want[~nan].view(torch.int32))


def _median_cases():
    g = torch.Generator().manual_seed(11)
    H, W = 45, 77
    pred = torch.rand(H, W, 3, generator=g) * 0.9 + 0.05
    gt = torch.rand(H, W, 3, generator=g)
    yield "random", pred, gt, torch.rand(H, W, generator=g) < 0.5
    full = torch.ones(H, W, dtype=torch.bool)
    yield "odd count", pred, gt, full                                  # 3465 pixels
    even = full.clone()
    even[0, 0] = False
    yield "even count", pred, gt, even
    q = torch.randint(0, 4, (H, W, 3), generator=g).float() * 0.25    # many equal ratios
    yield "duplicates", torch.ones(H, W, 3), q, even
    p0 = pred.clone()
    p0[::3] = 0.0
    yield "pred = 0 (clamped)", p0, gt, full
    yield "negative targets", pred, gt - 0.5, even
    nan = gt.clone()
    nan[3, 4, 1] = float("nan")
    yield "one NaN target", pred, nan, full
    pn = pred.clone()
    pn[5, 6, 2] = float("nan")
    yield "one NaN prediction", pn, gt, full
    single = torch.zeros(H, W, dtype=torch.bool)
    single[7, 8] = True
    yield "single pixel", pred, gt, single
    yield "two pixels", pred, gt, single | (torch.arange(W) == 9)[None] & (torch.arange(H) == 7)[:, None]
    yield "empty", pred, gt, torch.zeros(H, W, dtype=torch.bool)
    yield "C = 1", pred[..., :1].contiguous(), gt[..., :1].contiguous(), full
    yield "C = 4", torch.rand(H, W, 4, generator=g), torch.rand(H, W, 4, generator=g) * 3, even
    g8 = torch.Generator().manual_seed(8)
    yield "800x800", torch.rand(800, 800, 3, generator=g8), torch.rand(800, 800, 3, generator=g8), \
        torch.rand(800, 800, generator=g8) < 0.4


@pytest.mark.parametrize("case", [c[0] for c in _median_cases()])
def test_albedo_scale_is_bit_identical_to_torch_median(case):
    _, pred, gt, mask = next(c for c in _median_cases() if c[0] == case)
    p, t, m = pred.cuda(), gt.cuda(), mask.cuda()
    got = metrics.albedo_scale(p, t, m)
    assert got.dtype == torch.float32 and got.shape == (pred.shape[-1],)
    assert _same_bits(got, _torch_median(p, t, m)), (got, _torch_median(p, t, m))
    assert _same_bits(got, torch.from_numpy(om.albedo_scale(pred.numpy(), gt.numpy(), mask.numpy())))


def test_two_runs_give_identical_bits():
    x, y = _pair((800, 800, 3), 1)
    x, y = x.cuda(), y.cuda()
    m = _masks(800, 800, 2)["sparse"].cuda()
    for fn in (lambda: metrics.psnr(x, y, m), lambda: metrics.psnr(x, y), lambda: metrics.ssim(x, y),
               lambda: metrics.normal_mae(x, y, m), lambda: metrics.albedo_scale(x, y, m)):
        a, b = fn(), fn()
        assert torch.equal(a.view(torch.int64 if a.dtype == torch.float64 else torch.int32),
                           b.view(torch.int64 if b.dtype == torch.float64 else torch.int32))


def test_bad_arguments():
    x = torch.rand(16, 16, 3, device="cuda")
    m = torch.ones(16, 16, dtype=torch.bool, device="cuda")
    bad = [lambda: metrics.psnr(x.double(), x), lambda: metrics.psnr(x, x[..., :2]), lambda: metrics.psnr(x[0], x[0]),
           lambda: metrics.psnr(torch.rand(4, 4, 5, device="cuda"), torch.rand(4, 4, 5, device="cuda")),
           lambda: metrics.psnr(x, x, m.to(torch.uint8)), lambda: metrics.psnr(x, x, m[:8]),
           lambda: metrics.ssim(x[:10], x[:10]), lambda: metrics.ssim(x[:, :10], x[:, :10]),
           lambda: metrics.normal_mae(x[..., :1], x[..., :1], m), lambda: metrics.normal_mae(x, x, None),
           lambda: metrics.albedo_scale(x, x, None), lambda: metrics.albedo_scale(x.half(), x.half(), m)]
    for call in bad:
        with pytest.raises(ValueError):
            call()
    with pytest.raises(NotImplementedError, match="Only support cuda inputs."):
        metrics.psnr(x, x, m.cpu())


def test_metrics_do_not_synchronise():
    x, y = _pair((64, 80, 3), 4)
    x, y = x.cuda(), y.cuda()
    m = _masks(64, 80, 5)["sparse"].cuda()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        outs = [metrics.psnr(x, y), metrics.psnr(x, y, m), metrics.ssim(x, y), metrics.normal_mae(x, y, m),
                metrics.albedo_scale(x, y, m)]
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert all(o.is_cuda for o in outs)


# ------------------------------------------------------------------ evaluate_frame on the small split-sum model
HW = (100, 100)


def _split_model():
    """the seeded split-sum test model of tests/test_gpu_splitsum.py, stage 1, ball occupancy grid"""
    from rise_sdf_b200 import synthetic as syn
    from rise_sdf_b200.split_mixed_occ import SplitMixedOCCModel, split_mixed_occ_config
    torch.manual_seed(0)
    cfg = split_mixed_occ_config()
    cfg["light"]["envlight_config"]["base_res"] = 64
    m = SplitMixedOCCModel(cfg).cuda()
    with torch.no_grad():
        m.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
        m.variance.variance.fill_(0.5)
        m.geometry.encoding.encoding.encoding.params.uniform_(-0.02, 0.02)
    m.eval()
    m.update_step(0, 20000)
    assert m.stage == 1
    m.background_color = torch.ones(3, device="cuda")
    m.occupancy_grid.binaries = syn.analytic_grid("ball")[None].cuda()
    m.render_step_size = 1.732 * 2 * 1.5 / 256
    return m


@pytest.fixture(scope="module")
def scene():
    from rise_sdf_b200 import synthetic as syn
    from rise_sdf_b200.relight import EVAL_KEYS, EnvSet, render_frame_shard
    m = _split_model()
    g = torch.Generator().manual_seed(5)
    envs = EnvSet(m, [torch.rand(32, 64, 3, generator=g) * 2.0, torch.rand(32, 64, 3, generator=g) ** 4 * 20.0])
    rays = syn.frame_rays(3, w=HW[1], h=HW[0]).cuda()
    out, _ = render_frame_shard(m, rays, envs, keys=EVAL_KEYS + ("opacity",))
    img = {e: {k: v.view(*HW, -1) for k, v in o.items()} for e, o in out.items()}
    mask = img[0]["opacity"][..., 0] > 0.5
    assert 500 < int(mask.sum()) < HW[0] * HW[1] - 500, "the frame must show the object and the background"
    return m, envs, rays, img, mask


def test_evaluate_frame_of_the_models_own_renders(scene):
    from rise_sdf_b200.relight import evaluate_frame
    m, envs, rays, img, mask = scene
    targets = {"mask": mask, "albedo": img[0]["comp_albedo"], "normal": img[0]["comp_normal"],
               "relit": [img[e]["comp_rgb_phys_full"] for e in range(2)]}
    r = evaluate_frame(m, rays, HW, envs, targets)
    assert r["albedo_scale"] == [1.0, 1.0, 1.0]
    assert r["albedo_psnr"] == float("inf") and abs(r["albedo_ssim"] - 1.0) <= 1e-12
    assert r["normal_mae"] == 0.0
    assert r["relit_psnr"] == [float("inf")] * 2 and all(abs(s - 1.0) <= 1e-12 for s in r["relit_ssim"])
    # twice the predicted albedo: the scale is exactly 2 and the aligned prediction equals the target
    r2 = evaluate_frame(m, rays, HW, envs, {"mask": mask, "albedo": img[0]["comp_albedo"] * 2.0})
    assert r2["albedo_scale"] == [2.0, 2.0, 2.0] and r2["albedo_psnr"] == float("inf")
    assert set(r2) == {"albedo_scale", "albedo_psnr", "albedo_ssim"}
    assert evaluate_frame(m, rays, HW, envs, {}) == {}


def test_evaluate_frame_matches_oracle_on_perturbed_targets(scene):
    from rise_sdf_b200.relight import evaluate_frame
    m, envs, rays, img, mask = scene
    g = torch.Generator().manual_seed(21)
    noise = lambda s: torch.randn(*HW, 3, generator=g).cuda() * s
    alb = img[0]["comp_albedo"] * torch.tensor([1.3, 0.8, 1.1], device="cuda") + noise(0.02)
    nrm = img[0]["comp_normal"] + noise(0.05)
    relit = [(img[e]["comp_rgb_phys_full"] + noise(0.03)).clamp(0, 1) for e in range(2)]
    r = evaluate_frame(m, rays, HW, envs, {"mask": mask, "albedo": alb, "normal": nrm, "relit": relit})
    mk, pa = mask.cpu().numpy(), img[0]["comp_albedo"].cpu().numpy()
    scale = om.albedo_scale(pa, alb.cpu().numpy(), mk)
    assert np.array_equal(np.array(r["albedo_scale"], np.float32), scale)
    aligned = pa * scale                                              # float32, as the product multiplies
    assert abs(r["albedo_psnr"] - om.psnr(aligned, alb.cpu().numpy(), mk)) <= TOL
    z = lambda a: np.where(mk[..., None], a, np.float32(0))
    assert abs(r["albedo_ssim"] - om.ssim(z(aligned), z(alb.cpu().numpy()))) <= TOL
    assert abs(r["normal_mae"] - om.normal_mae(img[0]["comp_normal"].cpu().numpy(), nrm.cpu().numpy(), mk)) <= TOL
    for e in range(2):
        p, t = img[e]["comp_rgb_phys_full"].cpu().numpy(), relit[e].cpu().numpy()
        assert abs(r["relit_psnr"][e] - om.psnr(p, t)) <= TOL
        assert abs(r["relit_ssim"][e] - om.ssim(p, t)) <= TOL
    assert 0.0 < r["normal_mae"] < 90.0 and 0.0 < r["albedo_ssim"] < 1.0


def test_evaluate_frame_reads_back_once(scene):
    from rise_sdf_b200.relight import EVAL_KEYS, evaluate_frame, render_frame_shard
    m, envs, rays, img, mask = scene
    targets = {"mask": mask, "albedo": img[0]["comp_albedo"] + 0.01, "normal": img[0]["comp_normal"],
               "relit": [img[e]["comp_rgb_phys_full"] for e in range(2)]}

    def d2h(fn):
        fn()                                                          # warm-up outside the trace
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if "DtoH" in e.name or "Device -> Host" in e.name
                or "Device -> Pageable" in e.name]

    render = d2h(lambda: render_frame_shard(m, rays, envs, keys=EVAL_KEYS))
    scored = d2h(lambda: evaluate_frame(m, rays, HW, envs, targets))
    assert len(scored) == len(render) + 1, (render, scored)
