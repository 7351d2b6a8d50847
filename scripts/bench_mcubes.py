"""Marching-cubes kernel timing (rise_sdf_b200.mcubes.marching_cubes, csrc/mcubes.cu); prints one JSON line.

    python scripts/bench_mcubes.py [--reps 20]

Volumes: an analytic sphere sdf (radius 0.6 of the [-1, 1]^3 box) and the level grid of the seeded neus test model
(`tests/test_gpu_neus.py::build(table_scale=0.002)`, `VolumeSDF.isosurface_level`), each at 256^3 and 512^3, meshed as
`MarchingCubeHelper` does (-level, threshold 0).  Each entry is the mean of `--reps` warm calls between CUDA events,
host read-back of (V, F) and output allocation included.  Algorithmic bytes = the grid read twice (count and emit
pass) + the mesh written (12 B per vertex, 24 B per face).  A 256^3 grid (64 MB) fits in the 126 MB L2, so its
second read is served from there; the 512^3 grid (512 MB) does not.  The card's name and power limit are read in the
same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rise_sdf_b200.mcubes import marching_cubes, scratch_bytes  # noqa: E402
from rise_sdf_b200.neus import NeuSModel, neus_blender_config  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def sphere(n):
    g = torch.linspace(-1.0, 1.0, n, device="cuda")
    x, y, z = torch.meshgrid(g, g, g, indexing="ij")
    return (x * x + y * y + z * z).sqrt_() - 0.6


def model_level(n):
    torch.manual_seed(0)
    m = NeuSModel(neus_blender_config()).cuda().eval()
    with torch.no_grad():
        m.geometry.encoding.encoding.params.uniform_(-0.002, 0.002)
        m.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
    return m.geometry.isosurface_level(n)


def time_one(level, reps):
    for _ in range(3):
        v, f = marching_cubes(level, 0.0, negate=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        marching_cubes(level, 0.0, negate=True)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    nbytes = 2 * level.numel() * 4 + v.shape[0] * 12 + f.shape[0] * 24
    return {"ms": round(ms, 4), "V": v.shape[0], "F": f.shape[0], "scratch_bytes": scratch_bytes(level.shape),
            "algorithmic_bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_mcubes.py measures the GPU kernels and needs a CUDA device"
    name, power = card()
    out = {"gpu": name, "power_limit": power, "reps": args.reps, "results": {}}
    for n in (256, 512):
        for kind, make in (("sphere", sphere), ("neus_level", model_level)):
            level = make(n)
            out["results"][f"{kind}_{n}"] = time_one(level, args.reps)
            del level
            torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
