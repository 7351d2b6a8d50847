"""Test-stage metric timing (rise_sdf_b200.metrics, relight.evaluate_frame); prints one JSON line.

    python scripts/bench_metrics.py [--launches 200] [--frames 3]

* `kernel_ms`: each metric on one 800x800x3 fp32 frame pair (mask: ~half the pixels), CUDA events around `--launches`
  back-to-back calls after a warm-up, divided by the count.  A frame pair is 15 MB, so the inputs are read from L2.
* `frame_ms`: the configs[3] scene of bench.py's relighting leg (seed 42, variance 0.5, the occupancy grid refreshed
  once, two synthetic env maps, an 800x800 frame), host clock around calls that end in a device synchronise, the three
  alternated over `--frames` rounds after one warm-up round: `render` = render_frame_shard as bench.py calls it,
  `render_eval_keys` = the same with the albedo and normal keys that evaluate_frame renders, `evaluate` =
  evaluate_frame with every target (mask, albedo, normal, one relit frame per env map), read-back included.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rise_sdf_b200 import metrics  # noqa: E402
from rise_sdf_b200 import synthetic as syn  # noqa: E402
from rise_sdf_b200.relight import EVAL_KEYS, EnvSet, evaluate_frame, render_frame_shard, synthetic_envs  # noqa: E402
from rise_sdf_b200.split_mixed_occ import SplitMixedOCCModel, split_mixed_occ_config  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def kernel_times(n):
    g = torch.Generator().manual_seed(0)
    x = torch.rand(800, 800, 3, generator=g).cuda()
    y = (x.cpu() + 0.05 * torch.randn(800, 800, 3, generator=g)).cuda()
    m = (torch.rand(800, 800, generator=g) < 0.5).cuda()
    calls = {"psnr_masked": lambda: metrics.psnr(x, y, m), "psnr": lambda: metrics.psnr(x, y),
             "ssim": lambda: metrics.ssim(x, y), "normal_mae": lambda: metrics.normal_mae(x, y, m),
             "albedo_scale": lambda: metrics.albedo_scale(x, y, m)}
    out = {}
    for k, fn in calls.items():
        for _ in range(10):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        out[k] = round(a.elapsed_time(b) / n, 4)
    return out


def relight_scene():
    """bench.run_relight's model, occupancy grid and env maps (variance 0.5)"""
    torch.manual_seed(42)
    model = SplitMixedOCCModel(split_mixed_occ_config()).cuda()
    with torch.no_grad():
        model.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
        model.variance.variance.fill_(0.5)
    model.train()
    model.update_step(0, 80000)
    gj = torch.Generator().manual_seed(7)
    model.occupancy_grid._update(0, model.occ_eval_fn, occ_thre=0.001, jitter=torch.rand(128 ** 3, 3, generator=gj))
    model.eval()
    model.background_color = torch.ones(3, device="cuda")
    return model, EnvSet(model, synthetic_envs())


def frame_times(rounds):
    model, envs = relight_scene()
    rays = syn.frame_rays(3, syn.camera_poses(), syn.ray_directions()).cuda()
    hw = (800, 800)
    out, _ = render_frame_shard(model, rays, envs, keys=EVAL_KEYS + ("opacity",))
    g = torch.Generator().manual_seed(1)
    noise = lambda: torch.randn(800, 800, 3, generator=g).cuda() * 0.02
    img = lambda e, k: out[e][k].view(800, 800, -1)
    targets = {"mask": img(0, "opacity")[..., 0] > 0.5, "albedo": img(0, "comp_albedo") * 1.2 + noise(),
               "normal": img(0, "comp_normal") + noise(),
               "relit": [(img(e, "comp_rgb_phys_full") + noise()).clamp(0, 1) for e in range(len(envs.maps))]}
    calls = {"render": lambda: render_frame_shard(model, rays, envs),
             "render_eval_keys": lambda: render_frame_shard(model, rays, envs, keys=EVAL_KEYS),
             "evaluate": lambda: evaluate_frame(model, rays, hw, envs, targets)}
    ms = {k: [] for k in calls}
    scores = None
    for r in range(rounds + 1):
        for k, fn in calls.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize()
            if r:                                                   # round 0 is the warm-up
                ms[k].append((time.perf_counter() - t0) * 1e3)
            if k == "evaluate":
                scores = res
    mean = {k: round(sum(v) / len(v), 2) for k, v in ms.items()}
    return {"ms": mean, "ms_each": {k: [round(x, 2) for x in v] for k, v in ms.items()},
            "mask_pixels": int(targets["mask"].sum()), "env_maps": len(envs.maps),
            "scores": {k: ([round(x, 4) for x in v] if isinstance(v, list) else round(v, 4)) for k, v in scores.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--frames", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_metrics.py measures the GPU path and needs a CUDA device"
    name, power = card()
    out = {"gpu": name, "power_limit": power, "launches": args.launches, "frame": [800, 800, 3],
           "kernel_ms": kernel_times(args.launches), "frame_ms": frame_times(args.frames)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
