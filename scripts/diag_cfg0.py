"""cfg0 forward: error of the product and of the fp32 CPU oracle against the fp64 oracle."""
import sys
import numpy as np
import torch
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests')
from oracle import neus as oneus
from rise_sdf_b200 import synthetic as syn
from rise_sdf_b200.neus import NeuSModel, neus_blender_config
from helpers import oracle_params_from_model

torch.manual_seed(0)
m = NeuSModel(neus_blender_config(), fused_render=True).cuda().eval()
m.render_step_size = 1.732 * 2 * 1.5 / 128
m.occupancy_grid.binaries = torch.ones_like(m.occupancy_grid.binaries)
rays, _, _, bg = syn.training_rays(384, seed=1)
m.background_color = bg.cuda()
P = oracle_params_from_model(m)
grid = np.ones((128,) * 3, bool)
ref64 = oneus.forward(P.to(torch.float64), rays, grid, m.render_step_size, 1.0, background=bg, dtype=torch.float64)
ref32 = oneus.forward(P, rays, grid, m.render_step_size, 1.0, background=bg)
keys = ("comp_rgb", "comp_normal", "opacity", "depth")
def err(o):
    return {k: float(np.abs(o[k].detach().cpu().double().numpy() - ref64[k].detach().numpy()).max()) for k in keys}
print("cpu fp32 oracle vs fp64:", err(ref32))
with torch.no_grad():
    out = m(rays.cuda())
print("product vs fp64:", err(out))
e = np.abs(out["comp_normal"].detach().cpu().numpy() - ref64["comp_normal"].detach().numpy()).max(1)
i = int(e.argmax())
print("  worst ray", i, "opacity", float(ref64["opacity"][i]), "err", e[i])
