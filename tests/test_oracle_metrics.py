"""The float64 metric oracle (oracle/metrics.py) against closed forms and an independent brute-force SSIM.  CPU only."""
import numpy as np
import pytest

from oracle import metrics as om


def test_ssim_of_an_image_with_itself_is_one():
    x = np.random.default_rng(0).random((23, 17, 3))
    assert abs(om.ssim(x, x) - 1.0) <= 1e-15


@pytest.mark.parametrize("a,b", [(0.3, 0.7), (0.0, 0.5), (1.0, 1.0), (0.9, 0.1)])
def test_ssim_of_two_constant_images_is_the_luminance_term(a, b):
    x, y = np.full((14, 12, 1), a), np.full((14, 12, 1), b)
    want = (2 * a * b + om.C1) / (a * a + b * b + om.C1)
    assert abs(om.ssim(x, y) - want) <= 1e-12          # G*x^2 - mu^2 rounds to ~1e-17, against C2 = 9e-4


@pytest.mark.parametrize("shape", [(11, 11, 1), (13, 16, 3), (12, 11, 2)])
def test_separable_ssim_equals_brute_force(shape):
    rng = np.random.default_rng(sum(shape))
    x = rng.random(shape)
    y = np.clip(x + rng.normal(0, 0.2, shape), 0, 1)
    assert abs(om.ssim(x, y) - om.ssim_bruteforce(x, y)) <= 1e-13


def test_window_is_the_normalised_gaussian():
    g = om.gaussian()
    assert g.shape == (11,) and abs(g.sum() - 1) <= 1e-15 and np.allclose(g, g[::-1])
    assert abs(g[6] / g[5] - np.exp(-0.5 / 1.5 ** 2)) <= 1e-15


def test_psnr_of_a_known_mse():
    x = np.zeros((4, 5, 3))
    y = x + 0.1                                             # mse 0.01 -> 20 dB
    assert abs(om.psnr(x, y) - 20.0) <= 1e-12
    mask = np.zeros((4, 5), bool)
    mask[1, 2] = True
    y[1, 2] = 0.01                                          # the one selected pixel: mse 1e-4 -> 40 dB
    assert abs(om.psnr(x, y, mask) - 40.0) <= 1e-12
    assert om.psnr(x, x) == np.inf
    assert np.isnan(om.psnr(x, y, np.zeros((4, 5), bool)))


def test_atan2_angle_equals_arccos_away_from_parallel():
    rng = np.random.default_rng(1)
    a, b = rng.normal(size=(1000, 3)), rng.normal(size=(1000, 3)) * 3
    cos = np.sum(a * b, -1) / np.linalg.norm(a, axis=-1) / np.linalg.norm(b, axis=-1)
    keep = np.abs(cos) < 0.99
    assert keep.sum() > 900
    assert np.abs(om.angle_deg(a, b)[keep] - np.degrees(np.arccos(cos[keep]))).max() <= 1e-9
    assert om.angle_deg(np.array([0.0, 0, 1]), np.array([0.0, 0, 2])) == 0.0
    assert abs(om.angle_deg(np.array([1.0, 0, 0]), np.array([-1.0, 0, 0])) - 180.0) <= 1e-12
    assert om.angle_deg(np.zeros(3), np.array([-1.0, 0, 0])) == 90.0    # a zero vector: 90, not atan2(0, -0) = 180


def test_lower_median():
    assert om.lower_median([3.0, 1.0, 2.0]) == 2.0
    assert om.lower_median([4.0, 1.0, 3.0, 2.0]) == 2.0                 # even count: the lower of the two middle values
    assert om.lower_median([5.0, 5.0, 1.0, 5.0]) == 5.0                 # ties
    assert om.lower_median([2.0, 2.0, 7.0, 7.0]) == 2.0
    assert om.lower_median([-1.0]) == -1.0
    assert np.isnan(om.lower_median([1.0, np.nan, 2.0]))
    assert np.isnan(om.lower_median([]))
