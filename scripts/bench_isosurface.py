"""Streamed isosurface extraction timing (`VolumeSDF.isosurface`, `mcubes.marching_cubes_slabs`); prints one JSON line.

    python scripts/bench_isosurface.py [--reps 3] [--sizes 512,1024,2048]

* `isosurface_<n>`: `VolumeSDF.isosurface(n)` on bench.py's neus model (seed 42, hash-feature columns of the first
  layer drawn as bench.py draws them), eval mode: coarse level grid + mesh, padded bounds, fine level grid + mesh, all
  streamed in x-slabs of `mcubes.SLAB_BYTES` level values.
* `sphere_<n>`: `marching_cubes_slabs` alone on an analytic sphere sdf (radius 0.6 of the [-1, 1]^3 box) computed
  slab by slab into one buffer, so the time includes generating the field.
* `parent_path_512`: what `isosurface(512)` ran before it streamed -- the whole level grid (`isosurface_level`) meshed
  by `MarchingCubeHelper`, twice -- timed alternately with `isosurface_512` in the same run; `same_mesh` says whether
  the two meshes are identical.
Each time is the mean over `--reps` warm calls, from a host clock around work that ends in a device synchronise.
`peak_MiB` is the peak allocated device memory during one call above what was allocated before it (output included).
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

from rise_sdf_b200.geometry import MarchingCubeHelper  # noqa: E402
from rise_sdf_b200.mcubes import marching_cubes_slabs, plan_slabs  # noqa: E402
from rise_sdf_b200.neus import NeuSModel, neus_blender_config  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def bench_model():
    torch.manual_seed(42)
    m = NeuSModel(neus_blender_config()).cuda().eval()
    with torch.no_grad():
        m.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
    return m


def parent_isosurface(geo, resolution, threshold=0.0):
    """The non-streamed isosurface: one resolution^3 level buffer, dense marching cubes, coarse mesh kept whole."""
    helper = MarchingCubeHelper(resolution)
    dev = next(geo.parameters()).device
    buf = torch.empty(resolution ** 3, device=dev, dtype=torch.float32)
    r = geo.radius
    vmin = torch.full((3,), -r, dtype=torch.float32, device=dev)
    vmax = torch.full((3,), r, dtype=torch.float32, device=dev)
    for fine in (False, True):
        mesh = helper(geo.isosurface_level(resolution, vmin, vmax, out=buf), threshold)
        mesh["v_pos"] = mesh["v_pos"] * (vmax - vmin) + vmin
        if fine or mesh["v_pos"].shape[0] == 0:
            return mesh
        lo, hi = mesh["v_pos"].amin(dim=0), mesh["v_pos"].amax(dim=0)
        vmin = (lo - (hi - lo) * 0.1).clamp(-r, r)
        vmax = (hi + (hi - lo) * 0.1).clamp(-r, r)


def sphere_layers(n):
    shape = (n, n, n)
    buf = torch.empty(max(p for _, _, p in plan_slabs(shape)) * n * n, device="cuda")
    g = torch.linspace(-1.0, 1.0, n, device="cuda")

    def layers(x0, k):
        out = buf[:k * n * n].view(k, n, n)
        x, y, z = g[x0:x0 + k].view(k, 1, 1), g.view(1, n, 1), g.view(1, 1, n)
        torch.add(x * x + y * y, z * z, out=out)
        return out.sqrt_().sub_(0.6)
    return layers


def timed(fn):
    """(result, seconds, peak bytes above the memory allocated before the call)"""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, torch.cuda.max_memory_allocated() - base


def entry(times, peak, v, f, n):
    ms = [round(1e3 * t, 2) for t in times]
    return {"ms": round(sum(ms) / len(ms), 2), "ms_each": ms, "V": int(v.shape[0]), "F": int(f.shape[0]),
            "slabs": len(plan_slabs((n, n, n))), "peak_MiB": round(peak / 2 ** 20, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", default="512,1024,2048")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_isosurface.py measures the GPU path and needs a CUDA device"
    sizes = [int(s) for s in args.sizes.split(",")]
    name, power = card()
    out = {"gpu": name, "power_limit": power, "reps": args.reps, "results": {}}
    geo = bench_model().geometry
    for n in sizes:
        runs = {"isosurface": lambda: geo.isosurface(n)}
        if n == 512:
            runs["parent_path"] = lambda: parent_isosurface(geo, n)
        layers = sphere_layers(n)
        runs["sphere"] = lambda: dict(zip(("v_pos", "t_pos_idx"), marching_cubes_slabs(layers, (n, n, n), 0.0,
                                                                                        negate=True)))
        for fn in runs.values():                                     # warm-up
            timed(fn)
        times, peaks, meshes = {k: [] for k in runs}, {}, {}
        for _ in range(args.reps):                                   # the paths alternate
            for k, fn in runs.items():
                meshes[k] = None
                meshes[k], t, peaks[k] = timed(fn)
                times[k].append(t)
        for k, mesh in meshes.items():
            out["results"][f"{k}_{n}"] = entry(times[k], peaks[k], mesh["v_pos"], mesh["t_pos_idx"], n)
        if "parent_path" in meshes:
            a, b = meshes["isosurface"], meshes["parent_path"]
            out["results"][f"parent_path_{n}"]["same_mesh"] = (torch.equal(a["v_pos"], b["v_pos"])
                                                              and torch.equal(a["t_pos_idx"], b["t_pos_idx"]))
        del runs, meshes, layers
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
