import sys, time, numpy as np, torch
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests')
from rise_sdf_b200 import synthetic as syn
from rise_sdf_b200.split_mixed_occ import SplitMixedOCCModel, split_mixed_occ_config
from oracle import split as osplit
from helpers import split_oracle_params
torch.manual_seed(0)
cfg = split_mixed_occ_config(); cfg["light"]["envlight_config"]["base_res"] = 64
m = SplitMixedOCCModel(cfg).cuda()
with torch.no_grad():
    m.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05); m.variance.variance.fill_(0.5)
    m.geometry.encoding.encoding.encoding.params.uniform_(-0.02, 0.02)
m.eval(); m.update_step(0, 20000)
with torch.no_grad(): m.emitter.build_mips()
R = 192
rays, rgb, fg, bg = syn.training_rays(R, seed=3); m.background_color = bg.cuda()
grid = syn.analytic_grid('ball'); m.occupancy_grid.binaries = grid[None].cuda()
m.render_step_size = 1.732*2*1.5/256
P = split_oracle_params(m)
# use the product's own prefiltered maps in the oracle so that only the render path is compared
P.specular = [t.detach().cpu() for t in m.emitter.specular]; P.diffuse = m.emitter.diffuse.detach().cpu()
ref = osplit.forward(P, rays, grid.numpy(), m.render_step_size, stage=1, relighting=False, background=bg)
with torch.no_grad(): out = m(rays.cuda(), relighting=False)
print('samples', ref['num_samples'], int(out['num_samples'].sum()))
for k in ('comp_rgb', 'comp_rgb_phys', 'comp_normal', 'opacity', 'depth', 'comp_albedo', 'comp_spec_rgb'):
    a, b = out[k].cpu().numpy(), ref[k].numpy(); e = np.abs(a - b).max(-1)
    print(f'  {k:18s} max {e.max():.2e} mean {e.mean():.2e} p99 {np.quantile(e, .99):.2e} argmax {e.argmax()} n>1e-3 {(e>1e-3).sum()}')
bad = np.abs(out['comp_rgb'].cpu().numpy() - ref['comp_rgb'].numpy()).max(-1).argmax()
print('  worst ray', bad, 'opacity', float(out['opacity'][bad]), float(ref['opacity'][bad]), 'in valid(ref)', bad in ref['valid_indices'].tolist())
