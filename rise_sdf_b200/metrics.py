"""Test-stage scores on the device: PSNR, SSIM, normal angular error and median-ratio albedo alignment, the numbers
SplitOccSystem.test_step reports for every test view (systems/split_occ.py:417-424, criteria of systems/criterions.py).
Kernels in csrc/metrics.cu; every function returns a device tensor and never synchronises with the host, so a caller
can stack a frame's scores and read them back once (`relight.evaluate_frame`).

Images are [H, W, C] fp32 (C in 1..4; the rows of a render after `.view(H, W, C)`), masks [H, W] torch.bool.  The
kernels compute and accumulate in float64, and every reduction runs in a fixed order, so two calls give the same bits.

Definitions.  They follow the standard definitions the reference's criteria point to; they were NOT checked against the
reference's own `systems/criterions.py` and `systems/split_occ.py:417-424`, which were not available.  Choices made
where the reference may differ:
* psnr: instant-nsr-pl's criterion, -10 log10(mean squared error) over the selected elements (every channel of every
  selected pixel), with the data range fixed at 1.  +inf for identical inputs, NaN for an empty mask.
* ssim: torchmetrics' Gaussian defaults (Wang et al. 2004): an 11-tap Gaussian window with sigma 1.5 applied
  separably, C1 = 0.01^2 and C2 = 0.03^2, population moments sigma^2 = G*x^2 - mu^2 clamped at 0 as torchmetrics
  clamps them, and the mean of the SSIM map over the (H - 10) x (W - 10) valid pixels of every channel (torchmetrics'
  reflect-pad-then-crop and skimage's crop give the same region).  The data range is fixed at 1, where torchmetrics with
  `data_range=None` would infer it from the images.
* normal_mae: the mean angle in degrees between the two vectors of each selected pixel, atan2(|a x b|, a . b) after
  `light.safe_normalize` (squared norm clamped at 1e-20); atan2 rather than acos of a clamped dot product, which is off
  by up to 0.02 degrees for the near-parallel normals of a good reconstruction.  A zero vector (a pixel the render
  missed) scores 90 degrees, the value acos of the clamped dot product gives, where atan2(0, +-0) would follow the sign
  of a zero.
* albedo_scale: per channel the median of gt / pred.clamp(min=eps) over the selected pixels, with torch.median's lower
  median for an even count: bit-identical to `torch.median((gt[mask] / pred[mask].clamp(min=eps))[:, c])`, NaN if a
  selected ratio is NaN or the mask is empty.
LPIPS, the remaining image score of such evaluations, is not provided: it needs pretrained AlexNet / VGG weights.
"""
import ctypes
import math

import torch

from . import _lib as L

SSIM_KERNEL = 11
SSIM_SIGMA = 1.5


def _gaussian_window():
    d = [k - (SSIM_KERNEL - 1) / 2 for k in range(SSIM_KERNEL)]
    g = [math.exp(-0.5 * (x / SSIM_SIGMA) ** 2) for x in d]
    s = sum(g)
    return (ctypes.c_double * SSIM_KERNEL)(*[v / s for v in g])


_WINDOW = _gaussian_window()


def _check_images(pred, gt, channels=None):
    L.require_cuda(pred, gt)
    for name, t in (("pred", pred), ("gt", gt)):
        if t.dtype != torch.float32:
            raise ValueError(f"{name} must be float32, got {t.dtype}")
        if t.dim() != 3 or not 1 <= t.shape[2] <= 4:
            raise ValueError(f"{name} must be [H, W, C] with C in 1..4, got {tuple(t.shape)}")
    if pred.shape != gt.shape:
        raise ValueError(f"pred {tuple(pred.shape)} and gt {tuple(gt.shape)} differ in shape")
    if channels is not None and pred.shape[2] != channels:
        raise ValueError(f"expected {channels} channels, got {pred.shape[2]}")
    if pred.numel() >= 2 ** 31:
        raise ValueError(f"images of {pred.numel()} elements exceed the int32 element count")
    return pred.contiguous(), gt.contiguous()


def _check_mask(mask, pred, required=True):
    if mask is None:
        if required:
            raise ValueError("a [H, W] bool mask is required")
        return None
    L.require_cuda(mask)
    if mask.dtype != torch.bool or tuple(mask.shape) != tuple(pred.shape[:2]):
        raise ValueError(f"mask must be bool [{pred.shape[0]}, {pred.shape[1]}], got {mask.dtype} {tuple(mask.shape)}")
    return mask.contiguous()


def _partials(dev):
    return torch.empty(2 * L.METRIC_BLOCKS, dtype=torch.float64, device=dev)


def psnr(pred, gt, mask=None):
    """-10 log10(MSE) over the selected pixels' elements (all pixels without a mask), data range 1: 0-dim float64."""
    pred, gt = _check_images(pred, gt)
    mask = _check_mask(mask, pred, required=False)
    H, W, C = pred.shape
    out2 = torch.empty(2, dtype=torch.float64, device=pred.device)
    L.call("rsdf_sq_err_sum", L.ptr(pred), L.ptr(gt), L.ptr(mask), H, W, C, L.ptr(out2), L.ptr(_partials(pred.device)),
           L.stream())
    return -10.0 * torch.log10(out2[0] / out2[1])


def ssim(pred, gt):
    """Mean SSIM over the valid region of every channel (11-tap Gaussian, sigma 1.5, data range 1): 0-dim float64."""
    pred, gt = _check_images(pred, gt)
    H, W, C = pred.shape
    if H < SSIM_KERNEL or W < SSIM_KERNEL:
        raise ValueError(f"ssim needs images of at least {SSIM_KERNEL} x {SSIM_KERNEL}, got {H} x {W}")
    out = torch.empty((), dtype=torch.float64, device=pred.device)
    L.call("rsdf_ssim", L.ptr(pred), L.ptr(gt), H, W, C, _WINDOW, L.ptr(out), L.ptr(_partials(pred.device)), L.stream())
    return out


def normal_mae(pred, gt, mask):
    """Mean angle in degrees between pred and gt [H, W, 3] over the selected pixels: 0-dim float64 (NaN if none)."""
    pred, gt = _check_images(pred, gt, channels=3)
    mask = _check_mask(mask, pred)
    H, W, _ = pred.shape
    out2 = torch.empty(2, dtype=torch.float64, device=pred.device)
    L.call("rsdf_normal_angle_sum", L.ptr(pred), L.ptr(gt), L.ptr(mask), H, W, L.ptr(out2),
           L.ptr(_partials(pred.device)), L.stream())
    return out2[0] / out2[1]


def albedo_scale(pred, gt, mask, eps=1e-6):
    """Per-channel lower median of gt / pred.clamp(min=eps) over the selected pixels: float32 [C].  Multiply the
    predicted albedo by it to align it with the ground truth (the albedo's scale is ambiguous under unknown lighting)."""
    pred, gt = _check_images(pred, gt)
    mask = _check_mask(mask, pred)
    H, W, C = pred.shape
    out = torch.empty(C, dtype=torch.float32, device=pred.device)
    scratch = torch.empty(L.MEDIAN_SCRATCH_WORDS, dtype=torch.int32, device=pred.device)
    L.call("rsdf_ratio_median", L.ptr(pred), L.ptr(gt), L.ptr(mask), H, W, C, eps, L.ptr(out), L.ptr(scratch), L.stream())
    return out
