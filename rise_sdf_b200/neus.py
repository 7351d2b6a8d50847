"""Host-side mirror of models/neus.py (`NeuSModel`, `VarianceNetwork`): same call signatures
and output dict (models/neus.py:227-327), with the callee ops routed to librsdf_b200.so:

    occupancy_grid.sampling ........ K1 march + compaction       (nerfacc.py)
    geometry (hash grid + MLP) ..... K2 hash grid + K3 MLP       (tinycudann.py, geometry.py)
    get_alpha + render_weight_from_alpha + 4x accumulate_along_rays
                                     K4 fused NeuS render        (`fused_render=True`, default)
The un-fused, op-by-op path of the reference is kept (`fused_render=False`) because it is the
drop-in surface other callers use; both are parity-tested.  The learned-background branch
(models/neus.py:152-225) is out of scope (`learned_background: false` in both configs).
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib as L
from .geometry import VolumeSDF
from .nerfacc import OccGridEstimator, accumulate_along_rays, render_weight_from_alpha
from .network_utils import Config, update_module_step
from .texture import VolumeRadiance


def neus_blender_config(n_neurons=128, base_resolution=16, grad_type="analytic"):
    """configs/neus-blender.yaml:21-78 as a plain dict."""
    return Config({
        "name": "neus", "radius": 1.5, "num_samples_per_ray": 1024, "train_num_rays": 4096,
        "max_train_num_rays": 4096, "grid_prune": True, "grid_prune_occ_thre": 0.001,
        "dynamic_ray_sampling": False, "batch_image_sampling": True, "randomized": True,
        "ray_chunk": 4096, "cos_anneal_end": 20000, "learned_background": False,
        "background_color": "random",
        "variance": {"init_val": 0.3, "modulate": False},
        "geometry": {
            "name": "volume-sdf", "radius": 1.5, "feature_dim": 48, "grad_type": grad_type,
            "xyz_encoding_config": {"otype": "HashGrid", "n_levels": 16, "n_features_per_level": 2,
                                    "log2_hashmap_size": 19, "base_resolution": base_resolution,
                                    "per_level_scale": 1.447269237440378, "include_xyz": True},
            "mlp_network_config": {"otype": "VanillaMLP", "activation": "ReLU", "output_activation": "none",
                                   "n_neurons": n_neurons, "n_hidden_layers": 2, "sphere_init": True,
                                   "sphere_init_radius": 0.5, "weight_norm": True},
        },
        "texture": {
            "name": "volume-radiance", "input_feature_dim": 48 + 3,
            "dir_encoding_config": {"otype": "SphericalHarmonics", "degree": 4},
            "mlp_network_config": {"otype": "VanillaMLP", "activation": "ReLU", "output_activation": "none",
                                   "n_neurons": n_neurons, "n_hidden_layers": 4},
            "color_activation": "sigmoid",
        },
    })


class VarianceNetwork(nn.Module):
    """models/neus.py:21-50."""

    def __init__(self, config):
        super().__init__()
        self.config = config = Config(config)
        self.init_val = config.init_val
        self.register_parameter("variance", nn.Parameter(torch.tensor(float(config.init_val))))
        self.modulate = config.get("modulate", False)
        if self.modulate:
            self.mod_start_steps = config.mod_start_steps
            self.reach_max_steps = config.reach_max_steps
            self.max_inv_s = config.max_inv_s
            self.do_mod = False

    @property
    def inv_s(self):
        val = torch.exp(self.variance * 10.0)
        if self.modulate and self.do_mod:
            val = val.clamp_max(self.mod_val)
        return val

    def forward(self, x):
        return torch.ones([len(x), 1], device=self.variance.device) * self.inv_s

    def update_step(self, epoch, global_step):
        if self.modulate:
            self.do_mod = global_step > self.mod_start_steps
            if not self.do_mod:
                self.prev_inv_s = self.inv_s.item()
            else:
                self.mod_val = min((global_step / self.reach_max_steps) * (self.max_inv_s - self.prev_inv_s)
                                   + self.prev_inv_s, self.max_inv_s)


class _NeusRender(torch.autograd.Function):
    """K4: alpha + scan + accumulate in one pass; out[R,8] = (rgb3, normal3, opacity, depth)."""

    @staticmethod
    def forward(ctx, packed, rays_d, t_starts, t_ends, sdf, sdf_grad, rgb, inv_s, ratio):
        R = packed.shape[0]
        S = sdf.shape[0]
        dev = sdf.device
        sdf, sdf_grad, rgb = sdf.contiguous(), sdf_grad.contiguous(), rgb.contiguous()
        ctx.inv_shape = inv_s.shape
        inv_s = inv_s.reshape(1).contiguous().float()
        alpha = torch.empty(S, device=dev)
        w = torch.empty(S, device=dev)
        T = torch.empty(S, device=dev)
        out = torch.empty(R, 8, device=dev)
        L.call("rsdf_neus_render_fwd", L.ptr(packed), L.ptr(rays_d), L.ptr(t_starts), L.ptr(t_ends),
               L.ptr(sdf), L.ptr(sdf_grad), L.ptr(rgb), L.ptr(inv_s), float(ratio), R, L.ptr(alpha),
               L.ptr(w), L.ptr(T), L.ptr(out), L.stream())
        ctx.save_for_backward(packed, rays_d, t_starts, t_ends, sdf, sdf_grad, rgb, inv_s, alpha, w, T)
        ctx.ratio = float(ratio)
        ctx.mark_non_differentiable(alpha)
        return out, w, alpha

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_out, g_w, _g_alpha):
        packed, rays_d, t_starts, t_ends, sdf, sdf_grad, rgb, inv_s, alpha, w, T = ctx.saved_tensors
        R, S = packed.shape[0], sdf.shape[0]
        dev = sdf.device
        g_out = g_out.contiguous() if g_out is not None else torch.zeros(R, 8, device=dev)
        g_w = g_w.contiguous() if g_w is not None else None
        g_sdf = torch.empty(S, device=dev)
        g_grad = torch.empty(S, 3, device=dev)
        g_rgb = torch.empty(S, 3, device=dev)
        g_inv = torch.zeros(R, device=dev)
        L.call("rsdf_neus_render_bwd", L.ptr(packed), L.ptr(rays_d), L.ptr(t_starts), L.ptr(t_ends),
               L.ptr(sdf), L.ptr(sdf_grad), L.ptr(rgb), L.ptr(alpha), L.ptr(w), L.ptr(T), L.ptr(g_out),
               L.ptr(g_w), L.ptr(inv_s), ctx.ratio, R, L.ptr(g_sdf), L.ptr(g_grad), L.ptr(g_rgb),
               L.ptr(g_inv), L.stream())
        return None, None, None, None, g_sdf, g_grad, g_rgb, g_inv.sum().reshape(ctx.inv_shape), None


@torch.no_grad()
def neus_alpha(sdf, normal, dirs, dists, inv_s, cos_anneal_ratio):
    """get_alpha (models/neus.py:128-150 == models/split_mixed_occ.py:151-177) without autograd, one launch; same op
    order as the torch chain (tests/test_gpu_glue.py compares them)."""
    n = sdf.shape[0]
    alpha = torch.empty(n, device=sdf.device, dtype=torch.float32)
    L.call("rsdf_neus_alpha", L.ptr(sdf.reshape(-1).contiguous().float()), L.ptr(normal.contiguous().float()),
           L.ptr(dirs.contiguous().float()), L.ptr(dists.reshape(-1).contiguous().float()),
           L.ptr(inv_s.detach().reshape(1).contiguous().float()), float(cos_anneal_ratio), n, L.ptr(alpha), L.stream())
    return alpha


@torch.no_grad()
def sample_setup(rays_o, rays_d, ray_indices, t_starts, t_ends):
    """models/neus.py:247-252 in one launch -> (positions [S,3], t_dirs [S,3], midpoints [S,1], dists [S])."""
    S = ray_indices.shape[0]
    dev = rays_o.device
    positions = torch.empty(S, 3, device=dev, dtype=torch.float32)
    t_dirs = torch.empty(S, 3, device=dev, dtype=torch.float32)
    midpoints = torch.empty(S, 1, device=dev, dtype=torch.float32)
    dists = torch.empty(S, device=dev, dtype=torch.float32)
    L.call("rsdf_sample_setup", L.ptr(rays_o.contiguous()), L.ptr(rays_d.contiguous()), L.ptr(ray_indices.contiguous()),
           L.ptr(t_starts.contiguous()), L.ptr(t_ends.contiguous()), S, L.ptr(positions), L.ptr(t_dirs),
           L.ptr(midpoints), L.ptr(dists), L.stream())
    return positions, t_dirs, midpoints, dists


class _Normalize3(torch.autograd.Function):
    """F.normalize(g, p=2, dim=-1) for [S,3] CUDA tensors: one kernel forward, one backward."""

    @staticmethod
    def forward(ctx, g, eps):
        g = g.contiguous().float()
        out = torch.empty_like(g)
        L.call("rsdf_normalize3_fwd", L.ptr(g), g.shape[0], float(eps), L.ptr(out), L.stream())
        ctx.save_for_backward(g)
        ctx.eps = float(eps)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gn):
        (g,) = ctx.saved_tensors
        gg = torch.empty_like(g)
        L.call("rsdf_normalize3_bwd", L.ptr(g), L.ptr(gn.contiguous().float()), g.shape[0], ctx.eps, L.ptr(gg), L.stream())
        return gg, None


def normalize3(g, eps=1e-12):
    if g.is_cuda and g.dim() == 2 and g.shape[1] == 3 and g.shape[0] > 0:
        return _Normalize3.apply(g, eps)
    return F.normalize(g, p=2, dim=-1, eps=eps)


class NeuSModel(nn.Module):
    def __init__(self, config, fused_render=True):
        super().__init__()
        self.config = config = Config(config)
        self.fused_render = fused_render
        self.geometry = VolumeSDF(config.geometry)
        self.texture = VolumeRadiance(config.texture)
        if config.learned_background:
            raise NotImplementedError("learned background is out of scope (SURVEY.md §8b)")
        self.variance = VarianceNetwork(config.variance)
        r = config.radius
        self.register_buffer("scene_aabb", torch.as_tensor([-r, -r, -r, r, r, r], dtype=torch.float32))
        if config.grid_prune:
            self.occupancy_grid = OccGridEstimator(roi_aabb=self.scene_aabb, resolution=128)
        self.randomized = config.randomized
        self.background_color = None
        self.render_step_size = 1.732 * 2 * config.radius / config.num_samples_per_ray
        self.cos_anneal_ratio = 1.0

    # ------------------------------------------------------------------ schedule / grid update
    def occ_eval_fn(self, x):
        """models/neus.py:101-112."""
        sdf = self.geometry(x, with_grad=False, with_feature=False)
        inv_s = self.variance(torch.zeros([1, 3]))[:, :1].clip(1e-6, 1e6)
        inv_s = inv_s.expand(sdf.shape[0], 1)
        estimated_next_sdf = sdf[..., None] - self.render_step_size * 0.5
        estimated_prev_sdf = sdf[..., None] + self.render_step_size * 0.5
        prev_cdf = torch.sigmoid(estimated_prev_sdf * inv_s)
        next_cdf = torch.sigmoid(estimated_next_sdf * inv_s)
        p = prev_cdf - next_cdf
        c = prev_cdf
        return ((p + 1e-5) / (c + 1e-5)).view(-1, 1).clip(0.0, 1.0)

    def update_step(self, epoch, global_step):
        update_module_step(self.geometry, epoch, global_step)
        update_module_step(self.texture, epoch, global_step)
        update_module_step(self.variance, epoch, global_step)
        cos_anneal_end = self.config.get("cos_anneal_end", 0)
        self.cos_anneal_ratio = 1.0 if cos_anneal_end == 0 else min(1.0, global_step / cos_anneal_end)
        if self.training and self.config.grid_prune:
            self.occupancy_grid.update_every_n_steps(
                step=global_step, occ_eval_fn=self.occ_eval_fn,
                occ_thre=self.config.get("grid_prune_occ_thre", 0.01))

    # ------------------------------------------------------------------ alpha (un-fused path)
    def get_alpha(self, sdf, normal, dirs, dists):
        """models/neus.py:128-150."""
        if sdf.is_cuda and not torch.is_grad_enabled() and sdf.shape[0] > 0:
            return neus_alpha(sdf, normal, dirs, dists, self.variance.inv_s, self.cos_anneal_ratio)
        inv_s = self.variance(torch.zeros([1, 3]))[:, :1].clip(1e-6, 1e6)
        inv_s = inv_s.expand(sdf.shape[0], 1)
        true_cos = (dirs * normal).sum(-1, keepdim=True)
        iter_cos = -(F.relu(-true_cos * 0.5 + 0.5) * (1.0 - self.cos_anneal_ratio)
                     + F.relu(-true_cos) * self.cos_anneal_ratio)
        estimated_next_sdf = sdf[..., None] + iter_cos * dists.reshape(-1, 1) * 0.5
        estimated_prev_sdf = sdf[..., None] - iter_cos * dists.reshape(-1, 1) * 0.5
        prev_cdf = torch.sigmoid(estimated_prev_sdf * inv_s)
        next_cdf = torch.sigmoid(estimated_next_sdf * inv_s)
        p = prev_cdf - next_cdf
        c = prev_cdf
        return ((p + 1e-5) / (c + 1e-5)).view(-1).clip(0.0, 1.0)

    # ------------------------------------------------------------------ render
    def forward_(self, rays):
        n_rays = rays.shape[0]
        rays_o, rays_d = rays[:, 0:3].contiguous(), rays[:, 3:6].contiguous()
        with torch.no_grad():
            ray_indices, t_starts, t_ends, packed = self.occupancy_grid.sampling(
                rays_o, rays_d, render_step_size=self.render_step_size, stratified=self.randomized,
                cone_angle=0.0, alpha_thre=0.0, _return_packed=True)
        dev = rays.device
        if t_starts.shape[0] == 0:
            z = lambda *s: torch.zeros(*s, device=dev)
            comp_rgb, comp_normal, opacity, depth = z(n_rays, 3), z(n_rays, 3), z(n_rays, 1), z(n_rays, 1)
            sdf, sdf_grad, weights, midpoints, dists = z(0), z(0, 3), z(0), z(0, 1), z(0)
        else:
            if rays.is_cuda and not (rays_o.requires_grad or rays_d.requires_grad):
                positions, t_dirs, midpoints, dists = sample_setup(rays_o, rays_d, ray_indices, t_starts, t_ends)
            else:
                t_origins = rays_o[ray_indices]
                t_dirs = rays_d[ray_indices]
                midpoints = (t_starts + t_ends)[..., None] / 2.0
                positions = t_origins + t_dirs * midpoints
                dists = t_ends - t_starts
            sdf, sdf_grad, feature = self.geometry(positions, with_grad=True, with_feature=True)
            normal = normalize3(sdf_grad)
            rgb = self.texture(feature, t_dirs, normal)
            if self.fused_render:
                out8, weights, _ = _NeusRender.apply(packed, rays_d, t_starts, t_ends, sdf, sdf_grad, rgb,
                                                     self.variance.inv_s, self.cos_anneal_ratio)
                comp_rgb, comp_normal = out8[:, 0:3], out8[:, 3:6]
                opacity, depth = out8[:, 6:7], out8[:, 7:8]
            else:
                alpha = self.get_alpha(sdf, normal, t_dirs, dists)
                weights, _ = render_weight_from_alpha(alpha, ray_indices=ray_indices, n_rays=n_rays)
                kw = dict(ray_indices=ray_indices, n_rays=n_rays, packed_info=packed)
                opacity = accumulate_along_rays(weights, values=None, **kw)
                depth = accumulate_along_rays(weights, values=midpoints, **kw)
                comp_rgb = accumulate_along_rays(weights, values=rgb, **kw)
                comp_normal = accumulate_along_rays(weights, values=normal, **kw)
            comp_normal = F.normalize(comp_normal, p=2, dim=-1)
        out = {
            "comp_rgb": comp_rgb, "comp_normal": comp_normal, "opacity": opacity, "depth": depth,
            "rays_valid": opacity > 0,
            "num_samples": torch.as_tensor([len(t_starts)], dtype=torch.int32, device=dev),
        }
        if self.training:
            out.update({"sdf_samples": sdf, "sdf_grad_samples": sdf_grad, "weights": weights.view(-1),
                        "points": midpoints.view(-1), "intervals": dists.view(-1),
                        "ray_indices": ray_indices.view(-1)})
        out_bg = {
            "comp_rgb": self.background_color[None, :].expand(*comp_rgb.shape),
            "num_samples": torch.zeros_like(out["num_samples"]),
            "rays_valid": torch.zeros_like(out["rays_valid"]),
        }
        from .glue import composite
        out_full = {
            "comp_rgb": composite(out["comp_rgb"], out["opacity"], self.background_color),
            "num_samples": out["num_samples"] + out_bg["num_samples"],
            "rays_valid": out["rays_valid"] | out_bg["rays_valid"],
        }
        return {**out, **{k + "_bg": v for k, v in out_bg.items()},
                **{k + "_full": v for k, v in out_full.items()}}

    def forward(self, rays):
        if self.training:
            out = self.forward_(rays)
        else:
            out = chunk_batch(self.forward_, self.config.ray_chunk, True, rays)
        return {**out, "inv_s": self.variance.inv_s}

    def train(self, mode=True):
        self.randomized = mode and self.config.randomized
        return super().train(mode=mode)

    def eval(self):
        self.randomized = False
        return super().eval()

    def regularizations(self, out):
        return {}

    @torch.no_grad()
    def export(self, chunk_size=1 << 20, resolution=512, threshold=0.0):
        """`NeuSModel.export` of models/neus.py (instant-nsr-pl), with vertex colours: the isosurface mesh, then the
        geometry at its vertices (chunked, analytic normals), normal = normalize(grad) and
        v_rgb = texture(feature, -normal, normal), i.e. the colour seen looking straight at the surface.  Returns
        {'v_pos', 't_pos_idx', 'v_rgb'} on the device (formats.save_mesh_obj writes it)."""
        mesh = self.geometry.isosurface(resolution, threshold)
        v_pos = mesh["v_pos"]
        if v_pos.shape[0] == 0:
            mesh["v_rgb"] = torch.zeros(0, 3, device=v_pos.device)
            return mesh
        _, sdf_grad, feature = chunk_batch(self.geometry, chunk_size, False, v_pos, with_grad=True, with_feature=True)
        normal = F.normalize(sdf_grad, p=2, dim=-1)
        mesh["v_rgb"] = self.texture(feature, -normal, normal)
        return mesh


def chunk_batch(func, chunk_size, move_to_cpu, *args, **kwargs):
    """models/utils.py:14-51: run `func` over the leading dim in chunks and merge dict/tuple/
    tensor outputs.  Unlike the reference, chunks are concatenated on the device and moved to
    the host ONCE at the end (157 per-chunk `.cpu()` syncs per 800x800 frame collapse to one)."""
    B = None
    for arg in args:
        if isinstance(arg, torch.Tensor):
            B = arg.shape[0]
            break
    out, out_type = {}, None
    for i in range(0, B, chunk_size):
        out_chunk = func(*[a[i:i + chunk_size] if isinstance(a, torch.Tensor) else a for a in args], **kwargs)
        if out_chunk is None:
            continue
        out_type = type(out_chunk)
        if isinstance(out_chunk, torch.Tensor):
            out_chunk = {0: out_chunk}
        elif isinstance(out_chunk, (tuple, list)):
            out_chunk = {k: c for k, c in enumerate(out_chunk)}
        elif not isinstance(out_chunk, dict):
            raise TypeError(f"Return value of func must be in type [torch.Tensor, list, tuple, dict], get {type(out_chunk)}.")
        for k, v in out_chunk.items():
            v = v if torch.is_grad_enabled() else v.detach()
            out.setdefault(k, []).append(v)
    if out_type is None:
        return None
    merged = {}
    for k, v in out.items():
        m = torch.cat(v, dim=0)
        merged[k] = m.cpu() if move_to_cpu else m
    if out_type is torch.Tensor:
        return merged[0]
    if out_type in (tuple, list):
        return out_type([merged[k] for k in sorted(merged)])
    return merged
