"""Textured export timing (`SplitMixedOCCModel.export` and its phases); prints one JSON line.

    python scripts/bench_bake.py [--reps 3] [--resolution 512] [--texture-size 8192] [--chunk-size 1048576]
                                 [--normal-map]

The model is the seeded split-sum test model (tests/test_gpu_splitsum.py `_split_model`: seed 0, hash-feature columns
of the first layer ~ N(0, 0.05), table ~ U(-0.02, 0.02)) in eval mode at stage 1.  Phases, each timed with CUDA events
on the current stream after one warm-up pass of all of them, mean over `--reps`:
* `isosurface`: `geometry.isosurface(resolution)`;
* `vertex_materials`: normals (`geometry(v, with_grad=True)`) and `bake.material_at` at the vertices;
* `texel_bands`: `bake.bake_material_atlas` (texels/s counts the texel rows that hold cells, the ones evaluated);
* `glb_write`: `formats.save_mesh_glb` of the export to a temporary directory (host work: atlas copy, PNG encoding).
With `--normal-map` (what `export(normal_map=True)` runs instead of `texel_bands`):
* `normal_bands`: `bake.atlas_tangents` and `bake.bake_atlases`, the material and normal atlases from one geometry
  evaluation (with the finite-difference gradient) per band; `normal_texels_per_s` counts the same texels as
  `texels_per_s`, and `glb_write` then writes the normal map too.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rise_sdf_b200 import bake, formats  # noqa: E402
from rise_sdf_b200.neus import chunk_batch  # noqa: E402
from rise_sdf_b200.split_mixed_occ import SplitMixedOCCModel, split_mixed_occ_config  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def split_model():
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
    return m


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--resolution", type=int, default=512)
    ap.add_argument("--texture-size", type=int, default=8192)
    ap.add_argument("--chunk-size", type=int, default=1 << 20)
    ap.add_argument("--normal-map", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_bake.py measures the GPU path and needs a CUDA device"
    name, power = card()
    m = split_model()
    res, T, chunk = args.resolution, args.texture_size, args.chunk_size
    tmp = tempfile.mkdtemp()
    state = {}

    @torch.no_grad()
    def vertex_materials():
        v = state["mesh"]["v_pos"]
        _, g = chunk_batch(m.geometry, chunk, False, v, with_grad=True, with_feature=False)
        return F.normalize(g, p=2, dim=-1), bake.material_at(m, v, chunk)

    def glb():
        mesh = state["mesh"]
        nrm, mats = state["vertex"]
        extra = {"t_tangent": state["normals"][0], "normal_atlas": state["normals"][1]} if args.normal_map else {}
        return formats.save_mesh_glb(os.path.join(tmp, "export.glb"), {
            **mesh, "v_nrm": nrm, "t_uv": bake.atlas_uv(mesh["t_pos_idx"].shape[0], T, "cuda"),
            "material_atlas": state["atlas"], **extra})

    def normal_bands():
        v, f = state["mesh"]["v_pos"], state["mesh"]["t_pos_idx"]
        t_tangent = bake.atlas_tangents(v, f, state["vertex"][0], T)
        _, normal_atlas = bake.bake_atlases(m, v, f, state["vertex"][0], t_tangent, T, chunk)
        state["normals"] = (t_tangent, normal_atlas)

    phases = {
        "isosurface": lambda: state.__setitem__("mesh", m.geometry.isosurface(res)),
        "vertex_materials": lambda: state.__setitem__("vertex", vertex_materials()),
        "texel_bands": lambda: state.__setitem__("atlas", bake.bake_material_atlas(
            m, state["mesh"]["v_pos"], state["mesh"]["t_pos_idx"], T, chunk)),
        "glb_write": glb,
    }
    if args.normal_map:
        phases = {**{k: v for k, v in phases.items() if k != "glb_write"}, "normal_bands": normal_bands,
                  "glb_write": glb}
    for fn in phases.values():                                   # warm-up
        fn()
    ms = {k: [] for k in phases}
    for _ in range(args.reps):
        for k, fn in phases.items():
            ms[k].append(timed(fn)[1])
    V, Fn = state["mesh"]["v_pos"].shape[0], state["mesh"]["t_pos_idx"].shape[0]
    C, cols = bake.atlas_layout(Fn, T)
    texels = -(-((Fn + 1) // 2) // cols) * C * T
    mean = {k: sum(v) / len(v) for k, v in ms.items()}
    out = {"gpu": name, "power_limit": power, "reps": args.reps, "resolution": res, "texture_size": T,
           "chunk_size": chunk, "V": V, "F": Fn, "cell": C, "texels_evaluated": texels,
           "glb_MiB": round(os.path.getsize(os.path.join(tmp, "export.glb")) / 2 ** 20, 1),
           "ms": {k: round(v, 2) for k, v in mean.items()},
           "ms_each": {k: [round(x, 2) for x in v] for k, v in ms.items()},
           "texels_per_s": round(texels / (mean["texel_bands"] * 1e-3)),
           "export_ms": round(mean["isosurface"] + mean["vertex_materials"] + mean["texel_bands"], 2)}
    if args.normal_map:
        out["normal_texels_per_s"] = round(texels / (mean["normal_bands"] * 1e-3))
        out["export_normal_map_ms"] = round(mean["isosurface"] + mean["vertex_materials"] + mean["normal_bands"], 2)
    os.remove(os.path.join(tmp, "export.glb"))
    os.rmdir(tmp)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
