"""What the test-stage metrics refuse before anything reaches the device: CPU tensors in the Python interface, and bad
shapes at the C ABI (-1 before any launch).  Also pins the SSIM window the product passes to the oracle's.  CPU only."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import metrics as om
from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import metrics


def test_ssim_window_is_the_oracle_gaussian():
    assert np.abs(np.array(metrics._WINDOW[:]) - om.gaussian()).max() <= 1e-17


def test_cpu_tensors_are_refused():
    x, m = torch.rand(16, 16, 3), torch.ones(16, 16, dtype=torch.bool)
    for call in (lambda: metrics.psnr(x, x), lambda: metrics.psnr(x, x, m), lambda: metrics.ssim(x, x),
                 lambda: metrics.normal_mae(x, x, m), lambda: metrics.albedo_scale(x, x, m)):
        with pytest.raises(NotImplementedError, match="Only support cuda inputs."):
            call()


def test_c_abi_rejects_bad_sizes():
    from rise_sdf_b200.build import build
    build(verbose=False)
    lib = L.lib()
    p = ctypes.c_void_p(16)                       # never dereferenced: every call below is refused before a launch
    win = (ctypes.c_double * 11)()
    for H, W, C in ((4, 4, 0), (4, 4, 5), (1 << 16, 1 << 15, 1), (-1, 4, 3)):
        assert lib.rsdf_sq_err_sum(p, p, None, H, W, C, p, p, None) == -1, (H, W, C)
        assert lib.rsdf_ratio_median(p, p, p, H, W, C, 1e-6, p, p, None) == -1, (H, W, C)
    for H, W in ((10, 64), (64, 10), (1 << 15, 1 << 15)):
        assert lib.rsdf_ssim(p, p, H, W, 3, win, p, p, None) == -1, (H, W)
    assert lib.rsdf_normal_angle_sum(p, p, p, 27000, 27000, p, p, None) == -1         # 3 H W >= 2^31 > H W
    assert lib.rsdf_normal_angle_sum(p, p, None, 8, 8, p, p, None) == -1              # the mask is required
    assert lib.rsdf_ratio_median(p, p, None, 8, 8, 3, 1e-6, p, p, None) == -1
