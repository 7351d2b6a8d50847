"""Host-side mirror of models/split_mixed_occ.py (`SplitMixedOCCModel`): split-sum PBR render of
the neural SDF -- primary march with the alpha_fn visibility filter, 7/24-channel shading
accumulate, reflection secondary rays, optional third bounce when relighting, normal-orientation
regulariser and the sRGB composite (models/split_mixed_occ.py:179-456).  Callee ops run on
librsdf_b200.so: K1 march (nerfacc.py), K2 hash grid (tinycudann.py), K3 fused MLPs in inference
(network_utils.VanillaMLP -> fused_mlp.py), K4 scan/accumulate (nerfacc.py), K5 texture lookups and
cube-map prefilter (nvdiffrast.py, renderutils.py, light.py).
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .geometry import VolumeSDF
from .light import EnvironmentLightMipCube, rgb_to_srgb
from .nerfacc import ContractionType, OccGridEstimator, accumulate_along_rays, pack_info
from .network_utils import Config, update_module_step
from .neus import VarianceNetwork, chunk_batch, neus_alpha, normalize3, sample_setup
from .split_shade import split_render
from .texture import VolumeMixedMipSplitOcc
from .volrend import rendering_with_normals_sdf, secondary_rendering


def split_mixed_occ_config(n_neurons=128):
    """configs/split-mixed-occ-tensoir.yaml:29-136 as a plain dict."""
    mlp = lambda h: {"otype": "VanillaMLP", "activation": "ReLU", "output_activation": "none",
                     "n_neurons": n_neurons, "n_hidden_layers": h}
    return Config({
        "name": "split-mixed-occ", "indirect_pred": True, "relighting_threshold": 0.3, "radius": 1.5,
        "num_samples_per_ray": 1024, "num_samples_per_secondary_ray": 96, "train_num_rays": 256,
        "max_train_num_rays": 4096, "grid_prune": True, "grid_prune_occ_thre": 0.001,
        "dynamic_ray_sampling": True, "batch_image_sampling": True, "randomized": True, "ray_chunk": 4096,
        "cos_anneal_end": 10000, "learned_background": False, "split_sum_kick_in_step": 10000,
        "background_color": "random",
        "variance": {"init_val": 0.3, "modulate": False},
        "geometry": {
            "name": "volume-sdf", "radius": 1.5, "feature_dim": 48, "grad_type": "finite_difference",
            "finite_difference_eps": "progressive",
            "xyz_encoding_config": {"otype": "ProgressiveBandHashGrid", "n_levels": 16, "start_level": 6,
                                    "start_step": 6000, "update_steps": 500, "n_features_per_level": 2,
                                    "log2_hashmap_size": 19, "base_resolution": 32,
                                    "per_level_scale": 1.447269237440378, "include_xyz": True},
            "mlp_network_config": {"otype": "VanillaMLP", "activation": "ReLU", "output_activation": "none",
                                   "n_neurons": n_neurons, "n_hidden_layers": 2, "sphere_init": True,
                                   "sphere_init_radius": 0.5, "weight_norm": True},
        },
        "texture": {
            "name": "volume-mixed-mip-split-occ", "input_feature_dim": 48, "other_dim": 3, "sample_size": 8,
            "dir_encoding_config": {"otype": "SphericalHarmonics", "degree": 5, "reflected": True},
            "metallic_mlp_network_config": mlp(2), "albedo_mlp_network_config": mlp(4),
            "spec_mlp_network_config": mlp(4), "roughness_mlp_network_config": mlp(2),
            "secondary_mlp_network_config": mlp(4),
            "xyz_encoding_config": {"otype": "VanillaFrequency", "n_frequencies": 6},
            "color_activation": "sigmoid",
        },
        "light": {"name": "envlight-mip-cube",
                  "envlight_config": {"hdr_filepath": None, "clamp": True, "nmf_format": False, "scale": 0.5,
                                      "bias": 0.25, "base_res": 512}},
    })


class SplitMixedOCCModel(nn.Module):
    def __init__(self, config, latlong=None, fg_lut=None):
        super().__init__()
        self.config = config = Config(config)
        self.geometry = VolumeSDF(config.geometry)
        self.texture = VolumeMixedMipSplitOcc(config.texture, fg_lut=fg_lut)
        self.emitter = EnvironmentLightMipCube(config.light, latlong=latlong)
        self.geometry.contraction_type = ContractionType.AABB
        self.variance = VarianceNetwork(config.variance)
        r = config.radius
        self.register_buffer("scene_aabb", torch.as_tensor([-r, -r, -r, r, r, r], dtype=torch.float32))
        if config.grid_prune:
            self.occupancy_grid = OccGridEstimator(roi_aabb=self.scene_aabb, resolution=128)
        self.randomized = config.randomized
        self.background_color = None
        self.render_step_size = 1.732 * 2 * config.radius / config.num_samples_per_ray
        self.num_samples_per_secondary_ray = config.get("num_samples_per_secondary_ray", 96)
        self.secondary_near_plane = config.get("secondary_near_plane", 0.05)
        self.secondary_far_plane = config.get("secondary_far_plane", 1.5)
        self.secondary_shader_chunk = config.get("secondary_shader_chunk", 160000)
        self.cos_anneal_ratio = 1.0
        self.stage = 0

    # ------------------------------------------------------------------ schedule
    def occ_eval_fn(self, x):
        sdf = self.geometry(x, with_grad=False, with_feature=False)
        inv_s = self.variance(torch.zeros([1, 3]))[:, :1].clip(1e-6, 1e6)
        inv_s = inv_s.expand(sdf.shape[0], 1)
        prev_cdf = torch.sigmoid((sdf[..., None] + self.render_step_size * 0.5) * inv_s)
        next_cdf = torch.sigmoid((sdf[..., None] - self.render_step_size * 0.5) * inv_s)
        return ((prev_cdf - next_cdf + 1e-5) / (prev_cdf + 1e-5)).view(-1, 1).clip(0.0, 1.0)

    def update_step(self, epoch, global_step):
        update_module_step(self.geometry, epoch, global_step)
        update_module_step(self.texture, epoch, global_step)
        update_module_step(self.variance, epoch, global_step)
        cos_anneal_end = self.config.get("cos_anneal_end", 0)
        self.cos_anneal_ratio = 1.0 if cos_anneal_end == 0 else min(1.0, global_step / cos_anneal_end)
        if self.training and self.config.grid_prune:
            self.occupancy_grid.update_every_n_steps(step=global_step, occ_eval_fn=self.occ_eval_fn,
                                                     occ_thre=self.config.get("grid_prune_occ_thre", 0.01))
        self.stage = 1 if global_step >= self.config.split_sum_kick_in_step else 0

    def get_alpha(self, sdf, normal, dirs, dists):
        """models/split_mixed_occ.py:151-177 (identical to models/neus.py:128-150)."""
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

    fused_render = True              # csrc/render.cu sdf_render_*_kernel<CD, false, true>; False: op-by-op (parity yardstick)
    reuse_sampling_pass = True       # no-grad passes only; results are bit-identical either way (test)
    _skip_alpha = False
    _tile_cache = None               # relight.render_frame_shard: one dict per tile, shared by its env maps

    def _memo(self, key, fn):
        """Relighting renders the same rays under several environment maps (systems/split_occ.py:331-458 runs the
        whole test loop once per map).  Everything up to the emitter lookups -- sampling, field evaluations,
        material networks, the secondary bounce -- does not depend on the map, so with a tile cache installed it
        is computed for the first map and reused for the others (no-grad only; bit-identical, see the test)."""
        c = self._tile_cache
        if c is None or torch.is_grad_enabled():
            return fn()
        if key not in c:
            c[key] = fn()
        return c[key]


    def _alpha_fn(self, rays_o, rays_d, keep=None, with_feature=False):
        """`alpha_fn` of models/split_mixed_occ.py:197-208.  With `keep` (a list) the results of every call are
        appended to it: the reference evaluates the field a second time on the samples that survive `sampling`
        (:228-240 / compute_indirect_radiance :183-191), which for a no-grad pass recomputes exactly the same
        numbers -- the caller gathers them by the rows `sampling(..., _return_mask=True)` reports instead."""
        def alpha_fn(t_starts, t_ends, ray_indices):
            if ray_indices.shape[0] == 0:
                return torch.zeros((0,), device=rays_o.device)
            if rays_o.is_cuda and not torch.is_grad_enabled():
                # one launch: gathered directions, positions (same op order as below), interval lengths
                positions, t_dirs, _, dists = sample_setup(rays_o, rays_d, ray_indices, t_starts, t_ends)
            else:
                t_origins = rays_o[ray_indices]
                t_dirs = rays_d[ray_indices]
                positions = t_origins + t_dirs * (t_starts + t_ends)[..., None] / 2.0
                dists = (t_ends - t_starts)[..., None]
            feature = None
            if keep is not None and with_feature:
                sdf, sdf_grad, feature = self.geometry(positions, with_grad=True, with_feature=True)
            else:
                sdf, sdf_grad = self.geometry(positions, with_grad=True, with_feature=False)
            normal = normalize3(sdf_grad, eps=1e-6)
            alphas = self.get_alpha(sdf, normal, t_dirs, dists)
            if keep is not None:
                keep.append(dict(sdf=sdf, sdf_grad=sdf_grad, normal=normal, alphas=alphas, feature=feature))
            return alphas
        return alpha_fn

    @staticmethod
    def _kept(keep, key, rows):
        """rows of the concatenated per-call results of the visibility pass"""
        return (keep[0][key] if len(keep) == 1 else torch.cat([c[key] for c in keep]))[rows]

    def compute_indirect_radiance(self, rays_o, rays_d):
        n_rays = rays_o.shape[0]
        keep = [] if self.reuse_sampling_pass else None
        alpha_fn = self._alpha_fn(rays_o, rays_d, keep)
        with torch.no_grad():
            step = (self.secondary_far_plane - self.secondary_near_plane) / (self.num_samples_per_secondary_ray - 1)
            ray_indices, t_starts, t_ends, rows = self.occupancy_grid.sampling(
                rays_o, rays_d, alpha_fn=alpha_fn, near_plane=self.secondary_near_plane,
                far_plane=self.secondary_far_plane, render_step_size=step, stratified=False, _return_mask=True)
            if keep and rows is not None:
                cached = self._kept(keep, "alphas", rows)
                alpha_fn = lambda ts, te, ri: cached          # the survivors' alphas, as computed a moment ago
                chunk = None
            else:
                chunk = self.secondary_shader_chunk
            acc_map, depth_map, _ = secondary_rendering(t_starts, t_ends, ray_indices=ray_indices, n_rays=n_rays,
                                                        alpha_fn=alpha_fn, chunk_size=chunk)
        return 1.0 - acc_map, depth_map

    # ------------------------------------------------------------------ render
    def forward_(self, rays, relighting=False):
        n_rays = rays.shape[0]
        rays_o, rays_d = rays[:, 0:3].contiguous(), rays[:, 3:6].contiguous()
        fd_train = self.config.geometry.grad_type == "finite_difference" and self.training
        # no-grad render (eval / relighting): the shading pass reuses the visibility pass's field evaluation
        keep = [] if (self.reuse_sampling_pass and not torch.is_grad_enabled()) else None
        alpha_fn = self._alpha_fn(rays_o, rays_d, keep, with_feature=True)

        def rgb_normal_alpha_fn(t_starts, t_ends, ray_indices):
            t_origins = rays_o[ray_indices]
            t_dirs = rays_d[ray_indices]
            positions = t_origins + t_dirs * (t_starts + t_ends)[..., None] / 2.0
            if fd_train:
                sdf, sdf_grad, feature, sdf_laplace = self.geometry(positions, with_grad=True, with_feature=True,
                                                                    with_laplace=True)
                normal = normalize3(sdf_grad, eps=1e-6)
                alphas = None if self._skip_alpha else self.get_alpha(sdf, normal, t_dirs, (t_ends - t_starts)[..., None])
                colors = self.texture(feature, t_dirs, normal, positions, self.emitter, self.stage)
                return colors, normal, alphas, sdf, sdf_grad, sdf_laplace

            def fields():
                if survivors:                      # gathered from the visibility pass instead of re-evaluated
                    got = tuple(self._kept(keep, k, survivors[0])
                                for k in ("sdf", "sdf_grad", "feature", "normal", "alphas"))
                    keep.clear()
                    return got
                sdf, sdf_grad, feature = self.geometry(positions, with_grad=True, with_feature=True)
                normal = normalize3(sdf_grad, eps=1e-6)
                if self._skip_alpha:
                    return sdf, sdf_grad, feature, normal, None
                return sdf, sdf_grad, feature, normal, self.get_alpha(sdf, normal, t_dirs, (t_ends - t_starts)[..., None])

            sdf, sdf_grad, feature, normal, alphas = self._memo("fields", fields)
            mat = self._memo("material", lambda: self.texture.material(feature, t_dirs, normal, positions, self.stage))
            colors = self.texture.shade(mat, normal, self.emitter, self.stage)
            return colors, normal, alphas, sdf, sdf_grad

        def sample():
            r = self.occupancy_grid.sampling(
                rays_o, rays_d, alpha_fn=alpha_fn, render_step_size=self.render_step_size,
                stratified=self.randomized, cone_angle=0.0, alpha_thre=0.0, _return_mask=True)
            ok = bool(keep) and r[3] is not None
            return r[:3], ([r[3]] if ok else []), keep

        (ray_indices, t_starts, t_ends), survivors, keep = self._memo("sampling", sample)
        color_dim = 7 if self.stage == 0 else 24
        orientation_map = None
        if self.fused_render and rays.is_cuda and t_starts.shape[0] > 0:
            # get_alpha + weights + the five accumulations (colours, normals, opacity, depth, orientation) in one pass
            self._skip_alpha = True
            try:
                got = rgb_normal_alpha_fn(t_starts, t_ends, ray_indices)
            finally:
                self._skip_alpha = False
            colors, normals, sdf, sdf_grad = got[0], got[1], got[3], got[4]
            packed = self._memo("packed", lambda: pack_info(ray_indices, n_rays))
            acc, weights, _ = split_render(packed, rays_d, t_starts, t_ends, sdf, normals, colors, self.variance.inv_s,
                                           self.cos_anneal_ratio)
            rgb_map, normal_map = acc[:, :color_dim], acc[:, color_dim:color_dim + 3]
            acc_map, depth_map = acc[:, color_dim + 3:color_dim + 4], acc[:, color_dim + 4:color_dim + 5]
            orientation_map = acc[:, color_dim + 5:color_dim + 6]
            extras = {"weights": weights, "sdf": sdf, "sdf_grad": sdf_grad, "normals": normals}
            if fd_train:
                extras["sdf_laplace"] = got[5]
        else:
            rgb_map, normal_map, acc_map, depth_map, extras = rendering_with_normals_sdf(
                t_starts, t_ends, ray_indices=ray_indices, n_rays=n_rays, rgb_alpha_fn=rgb_normal_alpha_fn,
                render_bkgd=None, has_laplace=fd_train, color_dim=color_dim)

        valid_indices = torch.nonzero(acc_map > 0.5)[..., 0]
        rgb_map = rgb_map.clone()      # the reference writes through slices of rgb_map in place
        diff_rgb_map, spec_rgb_map, blend_map = rgb_map[..., :3], rgb_map[..., 3:6], rgb_map[..., 6:7]
        if self.stage != 0:
            diff_rgb_pbr_map, spec_rgb_pbr_map = rgb_map[..., 7:10], rgb_map[..., 10:13]
            spec_ref_map, spec_light_map = rgb_map[..., 13:16], rgb_map[..., 16:19]
            albedo_map, metallic_map, roughness_map = rgb_map[..., 19:22], rgb_map[..., 22:23], rgb_map[..., 23:]

        if valid_indices.numel() > 0 and self.config.indirect_pred:
            secondary_rays_o = rays_o[valid_indices] + depth_map[valid_indices] * rays_d[valid_indices]
            wo = -rays_d[valid_indices]
            nm = normal_map[valid_indices]
            secondary_rays_d = 2 * torch.sum(wo * nm, dim=-1, keepdim=True) * nm - wo
            tr, secondary_depth = self._memo("indirect", lambda: self.compute_indirect_radiance(
                secondary_rays_o.detach().contiguous(), secondary_rays_d.detach().contiguous()))
            tr = tr.clamp(0, 1).detach()
            secondary_depth = secondary_depth.detach()

            def secondary():
                _, secondary_feature = self.geometry(secondary_rays_o, with_grad=False, with_feature=True)
                return self.texture.secondary_shading(secondary_feature, secondary_rays_d, nm)
            secondary_rgb = self._memo("secondary_rgb", secondary)
            spec_rgb_map[valid_indices] = tr * spec_rgb_map[valid_indices] + (1 - tr) * secondary_rgb
            if self.stage != 0:
                if not relighting:
                    spec_rgb_pbr_map[valid_indices] = tr * spec_rgb_pbr_map[valid_indices] + (1 - tr) * secondary_rgb
                else:
                    # (integer rows computed once -- roughness does not depend on the env map -- instead of seven
                    # boolean-mask gathers, each of which is a nonzero + host read-back)
                    roughness_mask = self._memo("rough_rows", lambda: torch.nonzero(
                        (roughness_map[valid_indices] <= self.config.relighting_threshold)[..., 0])[:, 0])
                    third_rays_o = secondary_rays_o[roughness_mask] + secondary_depth[roughness_mask] * secondary_rays_d[roughness_mask]
                    third_dirs = secondary_rays_d[roughness_mask]

                    def third():
                        _, third_grad, third_feature = self.geometry(third_rays_o, with_grad=True, with_feature=True)
                        third_normal = normalize3(third_grad, eps=1e-6)
                        if third_dirs.shape[0] == 0:
                            return third_normal, None
                        return third_normal, self.texture.secondary_material_pbr(third_feature, third_dirs,
                                                                                 third_normal, third_rays_o)
                    third_normal, third_mat = self._memo("third", third)
                    third_rgb = (torch.zeros((0, 3), device=third_dirs.device) if third_mat is None else
                                 self.texture.secondary_shade_pbr(third_mat, third_dirs, third_normal, self.emitter))
                    slv = spec_light_map[valid_indices]
                    slv[roughness_mask] = tr[roughness_mask] * slv[roughness_mask] + (1 - tr[roughness_mask]) * third_rgb
                    spec_light_map[valid_indices] = slv
                    # models/split_mixed_occ.py:332 recombines EVERY ray of the batch -- and a batch without a single
                    # valid ray never gets here.  The reference's batches are `ray_chunk`-ray chunks (models/utils.py:
                    # 14-51), so for a larger batch the rule is applied per reference chunk: a ray is recombined iff
                    # ITS 4096-ray chunk holds a ray with opacity > 0.5 (batches start on a chunk boundary: relight.py).
                    recombined = spec_ref_map * spec_light_map
                    rc = int(self.config.get("ray_chunk", 0) or 0)
                    if rc and n_rays > rc and not self.training:
                        n_chunks = -(-n_rays // rc)
                        flags = torch.zeros(n_chunks * rc, dtype=torch.bool, device=rays.device)
                        flags[valid_indices] = True
                        in_live_chunk = flags.view(n_chunks, rc).any(1).repeat_interleave(rc)[:n_rays]
                        spec_rgb_pbr_map = torch.where(in_live_chunk[:, None], recombined, spec_rgb_pbr_map)
                    else:
                        spec_rgb_pbr_map = recombined

        rgb_full = diff_rgb_map + spec_rgb_map
        out = {
            "comp_rgb": rgb_full, "comp_diffuse_rgb": diff_rgb_map, "comp_spec_rgb": spec_rgb_map,
            "comp_blend": blend_map, "comp_normal": normal_map, "opacity": acc_map, "depth": depth_map,
            "rays_valid": acc_map > 0,
            "num_samples": torch.as_tensor([len(t_starts)], dtype=torch.int32, device=rays.device),
        }
        if self.stage != 0:
            rgb_pbr_map = diff_rgb_pbr_map + spec_rgb_pbr_map
            out.update({"comp_rgb_phys": rgb_pbr_map, "comp_diffuse_rgb_phys": diff_rgb_pbr_map,
                        "comp_spec_rgb_phys": spec_rgb_pbr_map, "comp_albedo": albedo_map,
                        "comp_metallic": metallic_map, "comp_roughness": roughness_map})
        if self.training:
            weights = extras["weights"]
            out.update({"sdf_samples": extras["sdf"], "sdf_grad_samples": extras["sdf_grad"],
                        "weights": weights.view(-1), "ray_indices": ray_indices.view(-1)})
            if self.config.geometry.grad_type == "finite_difference":
                out["sdf_laplace_samples"] = extras["sdf_laplace"]
            if orientation_map is not None:
                out["normals_orientation_loss_map"] = orientation_map
            elif ray_indices.numel() > 0:
                orient = torch.sum(rays_d[ray_indices] * extras["normals"], dim=-1, keepdim=True).clamp(min=0)
                out["normals_orientation_loss_map"] = accumulate_along_rays(
                    weights, values=orient, ray_indices=ray_indices, n_rays=n_rays)
            else:
                out["normals_orientation_loss_map"] = torch.zeros_like(rgb_full[..., :1])

        bg = self.background_color[None, :]
        out_bg = {"comp_rgb": bg.expand(*rgb_full.shape), "num_samples": torch.zeros_like(out["num_samples"]),
                  "rays_valid": torch.zeros_like(out["rays_valid"])}
        from .glue import composite
        out_full = {
            "comp_rgb": composite(out["comp_rgb"], out["opacity"], self.background_color, srgb=True),
            "num_samples": out["num_samples"] + out_bg["num_samples"],
            "rays_valid": out["rays_valid"] | out_bg["rays_valid"],
        }
        if self.stage != 0:
            out_bg["comp_rgb_phys"] = bg.expand(*rgb_pbr_map.shape)
            comp = lambda x: composite(x, out["opacity"], self.background_color, srgb=True)
            out_full.update({"comp_rgb_phys": comp(out["comp_rgb_phys"]), "comp_spec_rgb": comp(out["comp_spec_rgb"]),
                             "comp_spec_rgb_phys": comp(out["comp_spec_rgb_phys"])})
        return {**out, **{k + "_bg": v for k, v in out_bg.items()}, **{k + "_full": v for k, v in out_full.items()}}

    def forward(self, rays, relighting=False):
        if self.training:
            out = self.forward_(rays, relighting=relighting)
        else:
            out = chunk_batch(self.forward_, self.config.ray_chunk, True, rays, relighting)
        return {**out, "inv_s": self.variance.inv_s}

    def train(self, mode=True):
        self.randomized = mode and self.config.randomized
        return super().train(mode=mode)

    def eval(self):
        self.randomized = False
        return super().eval()

    @torch.no_grad()
    def export(self, chunk_size=1 << 20, resolution=512, threshold=0.0, texture_size=8192, normal_map=False):
        """The recovered geometry and PBR materials as a textured mesh (formats.save_mesh_glb writes it as glTF).
        Like `NeuSModel.export`: the isosurface mesh, then normal = normalize(grad) at its vertices (chunked).
        Materials (linear albedo, roughness, metallic; view-independent, so defined in every stage) are evaluated at
        the vertices and baked into a texture_size^2 atlas of one-triangle charts (rise_sdf_b200/bake.py).  Returns, on
        the device: v_pos [V,3], t_pos_idx [F,3], v_nrm [V,3], v_albedo [V,3], v_roughness [V,1], v_metallic [V,1],
        t_uv [F,3,2] and material_atlas [T,T,5] (albedo rgb, roughness, metallic; 0 where no face owns the texel).
        With `normal_map`, also t_tangent [F,3,4] (glTF TANGENTs per face corner) and normal_atlas [T,T,3]: the shading
        normal normalize(grad) at every texel's surface point in tangent space, so detail finer than the mesh survives
        the export (the same band pass evaluates both atlases; the other entries do not change).
        Raises ValueError when the mesh has too many faces for `texture_size` (the message names the smallest size
        that fits)."""
        from . import _lib as L
        from .bake import atlas_tangents, atlas_uv, bake_atlases, bake_material_atlas, material_at
        L.require_cuda(self.scene_aabb)
        mesh = self.geometry.isosurface(resolution, threshold)
        v_pos, t_pos_idx = mesh["v_pos"], mesh["t_pos_idx"]
        dev = v_pos.device
        t_uv = atlas_uv(t_pos_idx.shape[0], texture_size, dev)         # a too-small atlas raises before the materials
        if v_pos.shape[0] == 0:
            mats = torch.zeros(0, 5, device=dev)
            mesh["v_nrm"] = torch.zeros(0, 3, device=dev)
        else:
            _, sdf_grad = chunk_batch(self.geometry, chunk_size, False, v_pos, with_grad=True, with_feature=False)
            mesh["v_nrm"] = F.normalize(sdf_grad, p=2, dim=-1)
            mats = material_at(self, v_pos, chunk_size)
        if normal_map:
            t_tangent = atlas_tangents(v_pos, t_pos_idx, mesh["v_nrm"], texture_size)
            atlas, normal_atlas = bake_atlases(self, v_pos, t_pos_idx, mesh["v_nrm"], t_tangent, texture_size,
                                               chunk_size)
        else:
            atlas = bake_material_atlas(self, v_pos, t_pos_idx, texture_size, chunk_size)
        mesh.update(v_albedo=mats[:, :3].contiguous(), v_roughness=mats[:, 3:4].contiguous(),
                    v_metallic=mats[:, 4:5].contiguous(), t_uv=t_uv, material_atlas=atlas)
        if normal_map:
            mesh.update(t_tangent=t_tangent, normal_atlas=normal_atlas)
        return mesh
