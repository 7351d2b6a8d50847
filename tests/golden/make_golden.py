"""Generates tests/golden/*.npz by running the REFERENCE's own compiled kernels
(oracle/_ref/nerfacc_cuda.so, built by oracle/build_ref.py from lib/nerfacc/cuda/csrc) on the
GPU box.  Run there:   python tests/golden/make_golden.py gpurun_out/golden
then copy the files into tests/golden/ and commit them.  Inputs are seeded synthetic rays."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref as oref  # noqa: E402
from rise_sdf_b200 import synthetic as syn  # noqa: E402

ROI = [-1.5] * 3 + [1.5] * 3
# rays stored per file: the five special rays and every k-th ray after them, so that each file stays under 1 MB
KEEP_EVERY = {"ball": 5, "random": 3}
PER_RAY = ("rays_o", "rays_d", "t_min", "t_max")
PER_SAMPLE = ("t_starts", "t_ends", "alphas", "weights", "trans", "grad_weights", "grad_alphas")


def keep_rays(rec, every):
    """`rec` restricted to rays 0-4 and every `every`-th ray.  A ray's samples are one contiguous run of the packed
    arrays and every kernel here works ray by ray, so the kept runs are exactly what the kernels give for the kept rays;
    only packed_info and ray_indices are renumbered."""
    pk = rec["packed_info"]
    keep = np.array([r for r in range(len(pk)) if r < 5 or r % every == 0])
    sel = np.concatenate([np.arange(pk[r, 0], pk[r, 0] + pk[r, 1]) for r in keep]).astype(np.int64)
    n = pk[keep, 1]
    out = dict(rec)
    out.update({k: rec[k][keep] for k in PER_RAY})
    out.update({k: rec[k][sel] for k in PER_SAMPLE})
    out["packed_info"] = np.stack([np.cumsum(n) - n, n], 1).astype(pk.dtype)
    out["ray_indices"] = np.repeat(np.arange(len(keep)), n).astype(rec["ray_indices"].dtype)
    return out


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    C = oref.nerfacc_cuda()
    assert C is not None, "build oracle/_ref first"
    only = os.environ.get("RSDF_GOLDEN_ONLY")            # e.g. "ball_cone": regenerate one file
    for kind, res, R, step, cone in [("ball", 128, 1024, 1.732 * 3 / 1024, 0.0), ("shell", 128, 1024, 1.732 * 3 / 1024, 0.0),
                                     ("random", 32, 768, 0.01, 0.0), ("ones", 16, 512, 1.732 * 3 / 128, 0.0),
                                     ("ball", 128, 512, 1.732 * 3 / 512, 0.004)]:
        tag = kind + ("_cone" if cone else "")
        if only and tag != only:
            continue
        rays, _, _, _ = syn.training_rays(R, seed=21)
        sp_o = torch.tensor([[0, 0, -4], [0, 0, 0], [5, 5, 5], [0.3, -0.2, 0.1], [1.5, 0, -4]], dtype=torch.float32)
        sp_d = torch.tensor([[0, 0, 1], [0.6, 0.8, 0], [0, 0, 1], [0, 1, 0], [0, 0, 1]], dtype=torch.float32)
        rays[:5] = torch.cat([sp_o, sp_d], -1)
        grid = syn.analytic_grid(kind, res=res)
        o, d = rays[:, :3].contiguous().cuda(), rays[:, 3:].contiguous().cuda()
        roi = torch.tensor(ROI, device="cuda")
        tmin, tmax = C.ray_aabb_intersect(o, d, roi)
        pk, ri, ts, te = C.ray_marching(o, d, tmin, tmax, roi, grid.cuda(), C.ContractionType.AABB, float(np.float32(step)), float(cone))
        a = torch.rand(ri.shape[0], 1, device="cuda", generator=torch.Generator("cuda").manual_seed(1)) * 0.2
        w = C.weight_from_alpha_forward_naive(pk, a)
        T = C.transmittance_from_alpha_forward_naive(pk, a)
        gw = torch.randn_like(w)
        ga = C.weight_from_alpha_backward_naive(w, gw, pk, a)
        rec = dict(
            cone=np.float32(cone), rays_o=o.cpu().numpy(), rays_d=d.cpu().numpy(),
            roi=np.array(ROI, np.float32), grid=grid.numpy(), step=np.float32(step), t_min=tmin.cpu().numpy(),
            t_max=tmax.cpu().numpy(), packed_info=pk.cpu().numpy(), ray_indices=ri.cpu().numpy(),
            t_starts=ts[:, 0].cpu().numpy(), t_ends=te[:, 0].cpu().numpy(), alphas=a[:, 0].cpu().numpy(),
            weights=w[:, 0].cpu().numpy(), trans=T[:, 0].cpu().numpy(), grad_weights=gw[:, 0].cpu().numpy(),
            grad_alphas=ga[:, 0].cpu().numpy())
        if tag in KEEP_EVERY:
            rec = keep_rays(rec, KEEP_EVERY[tag])
        np.savez_compressed(os.path.join(out_dir, f"march_{tag}.npz"), **rec)
        print(tag, "rays", R, "samples", ri.shape[0])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/golden")


def cubemap_golden(out_dir):
    """tests/golden/cubemap_*.npz from the reference's renderutils plugin (lib/renderutils/c_src/cubemap.cu)."""
    P = oref.renderutils_plugin()
    assert P is not None
    from oracle import textures as ot
    g = torch.Generator().manual_seed(11)
    cube = torch.rand(6, 16, 16, 3, generator=g) * 0.5 + 0.25
    go = torch.randn(6, 16, 16, 3, generator=g)
    d_out = P.diffuse_cubemap_fwd(cube.cuda())
    d_g = P.diffuse_cubemap_bwd(cube.cuda(), go.cuda().contiguous())
    rec = dict(cube16=cube.numpy(), go16=go.numpy(), diffuse_fwd=d_out.cpu().numpy(), diffuse_bwd=d_g.cpu().numpy())
    for N, rough in [(16, 1.0), (32, 0.08)]:
        c = torch.rand(6, N, N, 3, generator=g) * 0.5 + 0.25
        cut = ot.ndf_cutoff(rough, 0.99)
        b = P.specular_bounds(N, cut)
        raw = P.specular_cubemap_fwd(c.cuda(), b, rough, cut)
        rec.update({f"spec{N}_cube": c.numpy(), f"spec{N}_rough": np.float32(rough), f"spec{N}_cut": np.float64(cut),
                    f"spec{N}_bounds": b.cpu().numpy().astype(np.int16), f"spec{N}_raw": raw.cpu().numpy()})
    np.savez_compressed(os.path.join(out_dir, "cubemap_prefilter.npz"), **rec)
    print("cubemap golden written")


if __name__ == "__main__":
    cubemap_golden(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/golden")
