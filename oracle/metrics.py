"""Float64 CPU oracle of the test-stage metrics (rise_sdf_b200/metrics.py, csrc/metrics.cu).  Test infrastructure only.

Images are [H, W, C] arrays, masks [H, W] bool; everything is evaluated in float64 with numpy / scipy.
* psnr: -10 log10(mean of (pred - gt)^2 over the selected pixels' elements), data range 1.
* ssim: Gaussian window (11 taps, sigma 1.5), C1 = 0.01^2, C2 = 0.03^2, population moments with the variances clamped
  at 0, mean over the (H - 10) x (W - 10) valid pixels of every channel.  `ssim` filters separably
  (scipy.ndimage.correlate1d, then a valid crop); `ssim_bruteforce` sums every 11 x 11 window directly and exists only
  to pin the separable one on tiny images.
* angle_deg: atan2(|a x b|, a . b) in degrees after dividing each vector by sqrt(max(|v|^2, 1e-20)); 90 degrees when
  a vector is zero (atan2(0, +-0) would depend on the sign of a zero).
* lower_median: np.sort, element (n - 1) // 2 (torch.median's convention for an even count); NaN if any value is NaN or
  there is none.
"""
import numpy as np
from scipy import ndimage

K, R, SIGMA = 11, 5, 1.5
C1, C2 = 0.01 ** 2, 0.03 ** 2


def gaussian():
    d = np.arange(K, dtype=np.float64) - R
    g = np.exp(-0.5 * (d / SIGMA) ** 2)
    return g / g.sum()


def psnr(pred, gt, mask=None):
    d = np.asarray(pred, np.float64) - np.asarray(gt, np.float64)
    if mask is not None:
        d = d[np.asarray(mask, bool)]
    if not d.size:
        return np.nan
    with np.errstate(divide="ignore"):
        return -10.0 * np.log10(np.mean(d * d))


def _ssim_map(mx, my, xx, yy, xy):
    vx = np.maximum(xx - mx * mx, 0.0)
    vy = np.maximum(yy - my * my, 0.0)
    cxy = xy - mx * my
    return ((2 * mx * my + C1) * (2 * cxy + C2)) / ((mx * mx + my * my + C1) * (vx + vy + C2))


def ssim(pred, gt):
    x, y = np.asarray(pred, np.float64), np.asarray(gt, np.float64)
    H, W = x.shape[:2]
    g = gaussian()

    def blur(a):
        a = ndimage.correlate1d(a, g, axis=0, mode="constant")
        a = ndimage.correlate1d(a, g, axis=1, mode="constant")
        return a[R:H - R, R:W - R]

    return float(np.mean(_ssim_map(blur(x), blur(y), blur(x * x), blur(y * y), blur(x * y))))


def ssim_bruteforce(pred, gt):
    x, y = np.asarray(pred, np.float64), np.asarray(gt, np.float64)
    H, W, C = x.shape
    g = gaussian()
    w2 = np.outer(g, g)
    vals = []
    for c in range(C):
        for i in range(H - 2 * R):
            for j in range(W - 2 * R):
                a, b = x[i:i + K, j:j + K, c], y[i:i + K, j:j + K, c]
                m = [np.sum(w2 * t) for t in (a, b, a * a, b * b, a * b)]
                vals.append(_ssim_map(*m))
    return float(np.mean(vals))


def angle_deg(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    a = a / np.sqrt(np.maximum(np.sum(a * a, -1, keepdims=True), 1e-20))
    b = b / np.sqrt(np.maximum(np.sum(b * b, -1, keepdims=True), 1e-20))
    cn, dot = np.linalg.norm(np.cross(a, b), axis=-1), np.sum(a * b, -1)
    return np.where((cn == 0) & (dot == 0), 90.0, np.degrees(np.arctan2(cn, dot)))


def normal_mae(pred, gt, mask):
    m = np.asarray(mask, bool)
    return float(np.mean(angle_deg(np.asarray(pred)[m], np.asarray(gt)[m]))) if m.any() else np.nan


def lower_median(v):
    v = np.asarray(v).reshape(-1)
    if v.size == 0 or np.isnan(v).any():
        return np.nan
    return np.sort(v)[(v.size - 1) // 2]


def albedo_scale(pred, gt, mask, eps=1e-6):
    """per channel lower median of the float32 ratio gt / max(pred, eps) (computed in float32, as the product does)"""
    m = np.asarray(mask, bool)
    p, g = np.asarray(pred, np.float32)[m], np.asarray(gt, np.float32)[m]
    r = g / np.maximum(p, np.float32(eps))                        # np.maximum keeps NaN, like torch.clamp
    return np.array([lower_median(r[:, c]) for c in range(p.shape[-1])], np.float32)
