"""Host-side mirror of models/texture.py for the render path.
    VolumeRadiance ............ models/texture.py:15-41 (`volume-radiance`, the neus config)
"""
import torch
import torch.nn as nn

from . import nvdiffrast as dr
from .network_utils import Config, get_activation, get_encoding, get_mlp, update_module_step


class VolumeRadiance(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config = Config(config)
        self.n_dir_dims = config.get("n_dir_dims", 3)
        self.n_output_dims = 3
        self.encoding = get_encoding(self.n_dir_dims, config.dir_encoding_config)
        self.n_input_dims = config.input_feature_dim + self.encoding.n_output_dims
        self.network = get_mlp(self.n_input_dims, self.n_output_dims, config.mlp_network_config)

    def forward(self, features, dirs, *args):
        dirs = (dirs + 1.0) / 2.0
        dirs_embd = self.encoding(dirs.view(-1, self.n_dir_dims))
        segs = [features.view(-1, features.shape[-1]), dirs_embd] + [arg.view(-1, arg.shape[-1]) for arg in args]
        if hasattr(self.network, "forward_segments"):
            color = self.network.forward_segments(segs)
        else:
            color = self.network(torch.cat(segs, dim=-1))
        color = color.view(*features.shape[:-1], self.n_output_dims).float()
        if "color_activation" in self.config:
            color = get_activation(self.config.color_activation)(color)
        return color

    def update_step(self, epoch, global_step):
        update_module_step(self.encoding, epoch, global_step)

    def regularizations(self, out):
        return {}


class VolumeMixedMipSplitOcc(nn.Module):
    """models/texture.py:234-434 (`volume-mixed-mip-split-occ`): five MLPs (albedo 6, roughness 1,
    metallic 2, env 3, secondary 3) on [feature48 | VanillaFrequency(pos) 36 | SH5(dir) 25], and the
    split-sum combine against the prefiltered env light + the 256x256 FG LUT.  Output channel order
    of forward() is the reference's (models/texture.py:345):
    [diff3, spec3, blend1, diff_pbr3, spec_pbr3, spec_ref3, spec_light3, albedo3, metallic1, roughness1]."""

    def __init__(self, config, fg_lut=None):
        super().__init__()
        self.config = config = Config(config)
        self.n_dir_dims = config.get("n_dir_dims", 3)
        self.n_pos_dims = config.get("n_pos_dims", 3)
        self.n_output_dims = 3
        self.dir_encoding = get_encoding(self.n_dir_dims, config.dir_encoding_config)
        self.xyz_encoding = get_encoding(self.n_pos_dims, config.xyz_encoding_config)
        fdim = config.input_feature_dim
        dn, xn = self.dir_encoding.n_output_dims, self.xyz_encoding.n_output_dims
        self.secondary_network = get_mlp(fdim + config.other_dim + dn, 3, config.secondary_mlp_network_config)
        self.albedo_network = get_mlp(fdim + xn, 6, config.albedo_mlp_network_config)
        self.roughness_network = get_mlp(fdim + xn, 1, config.roughness_mlp_network_config)
        self.env_network = get_mlp(fdim + dn, 3, config.spec_mlp_network_config)
        self.metallic_network = get_mlp(fdim + xn, 2, config.metallic_mlp_network_config)
        if fg_lut is None:
            # the reference loads load/bsdf/bsdf_256_256.bin (models/texture.py:285); offline we
            # integrate the same split-sum table synthetically (same [1,256,256,2] layout)
            from .synthetic import bsdf_lut
            fg_lut = bsdf_lut()
        self.register_buffer("FG_LUT", fg_lut.float().reshape(1, 256, 256, 2).contiguous())

    fused_shade = True          # csrc/split_shade.cu; False: the op-by-op path below (kept as the parity yardstick)

    def _fused(self, t):
        return self.fused_shade and t.is_cuda and self.config.get("color_activation", None) == "sigmoid"

    def _act(self, x):
        if "color_activation" in self.config:
            return get_activation(self.config.color_activation)(x)
        return x

    def _fg(self, NoV, roughness):
        fg_uv = torch.cat([torch.clamp(NoV, min=0.0, max=1.0), torch.clamp(roughness, min=0.0, max=1.0)], -1)
        pn = fg_uv.shape[0]
        return dr.texture(self.FG_LUT, fg_uv.reshape(1, pn, 1, 2).contiguous(), filter_mode="linear",
                          boundary_mode="clamp").reshape(pn, 2)

    def material_nets(self, features, positions):
        """Raw outputs of the three view-independent material networks on [feature, VanillaFrequency(position)]:
        albedo [..., 6] (diffuse rgb | albedo), roughness [..., 1], metallic [..., 2] (blend | metallic).  `material`
        and the atlas baker (`bake.material_at`) both start from these."""
        xyz_embd = self.xyz_encoding(positions.view(-1, self.n_pos_dims))
        network_inp = [features.view(-1, features.shape[-1]), xyz_embd]
        raw6 = self.albedo_network.forward_segments(network_inp).view(*features.shape[:-1], 6).float()
        roughness = self.roughness_network.forward_segments(network_inp).view(*features.shape[:-1], 1).float()
        raw2 = self.metallic_network.forward_segments(network_inp).view(*features.shape[:-1], 2).float()
        return raw6, roughness, raw2

    def material(self, features, dirs, normals, positions, stage=0):
        """The light-independent half of `forward` (models/texture.py:330-377 up to the emitter lookups): material
        networks, activations, reflection direction, FG lookup.  A relighting render under several environment
        maps evaluates it once per tile (`SplitMixedOCCModel._memo`)."""
        wi = -dirs
        wo = torch.sum(wi * normals, -1, keepdim=True) * normals * 2 - wi
        NoV = torch.sum(normals * wi, -1, keepdim=True)
        raw6, roughness, raw2 = self.material_nets(features, positions)
        diff_rgb, albedo = raw6[..., :3], raw6[..., 3:]
        blend, metallic = raw2[..., :1], raw2[..., 1:]
        wo_enc = self.dir_encoding(((wo + 1.0) / 2.0).view(-1, self.n_dir_dims))
        spec_rgb = self.env_network.forward_segments([features, wo_enc]).view(*features.shape[:-1], 3).float()
        if self._fused(features):
            # activations, mixes and lookups happen in ONE kernel in shade(); the networks' raw outputs are all it needs
            return {"raw_albedo": raw6, "raw_roughness": roughness, "raw_metallic": raw2, "raw_env": spec_rgb,
                    "dirs": dirs}
        albedo, diff_rgb, blend = self._act(albedo), self._act(diff_rgb), self._act(blend)
        metallic, roughness, spec_rgb = self._act(metallic), self._act(roughness), self._act(spec_rgb)
        spec_rgb = blend * spec_rgb
        diff_rgb = (1 - blend) * diff_rgb
        m = {"diff_rgb": diff_rgb, "spec_rgb": spec_rgb, "blend": blend}
        if stage != 0:
            diffuse_albedo = (1 - metallic) * albedo
            specular_albedo = 0.04 * (1 - metallic) + metallic * albedo
            fg_lookup = self._fg(NoV, roughness)
            m.update(wo=wo, albedo=albedo, metallic=metallic, roughness=roughness, diffuse_albedo=diffuse_albedo,
                     specular_ref=specular_albedo * fg_lookup[:, 0:1] + fg_lookup[:, 1:2])
        return m

    def shade(self, m, normals, emitter, stage=0):
        """The emitter-dependent half of `forward`: split-sum lighting lookups + channel packing."""
        if "raw_albedo" in m:
            from .split_shade import split_shade
            return split_shade(m["raw_albedo"], m["raw_roughness"], m["raw_metallic"], m["raw_env"], normals, m["dirs"],
                               emitter, self.FG_LUT, stage)
        if stage == 0:
            return torch.cat([m["diff_rgb"], m["spec_rgb"], m["blend"]], dim=-1)
        diffuse_light = emitter.eval_mip(normals)
        diff_rgb_pbr = m["diffuse_albedo"] * diffuse_light
        specular_light = emitter.eval_mip(m["wo"], specular=True, roughness=m["roughness"])
        spec_rgb_pbr = m["specular_ref"] * specular_light
        return torch.cat([m["diff_rgb"], m["spec_rgb"], m["blend"], diff_rgb_pbr, spec_rgb_pbr, m["specular_ref"],
                          specular_light, m["albedo"], m["metallic"], m["roughness"]], dim=-1)

    def forward(self, features, dirs, normals, positions, emitter, stage=0, *args):
        if dirs.shape[0] == 0:
            return torch.zeros((0, 3), device=dirs.device)
        return self.shade(self.material(features, dirs, normals, positions, stage), normals, emitter, stage)

    def secondary_shading(self, features, rays_d, *args):
        rays_d = (rays_d + 1.0) / 2.0
        dirs_embd = self.dir_encoding(rays_d.view(-1, self.n_dir_dims))
        network_inp = torch.cat([features.view(-1, features.shape[-1]), dirs_embd]
                                + [arg.view(-1, arg.shape[-1]) for arg in args], dim=-1)
        color = self.secondary_network(network_inp).view(*network_inp.shape[:-1], self.n_output_dims).float()
        return self._act(color)

    def secondary_material_pbr(self, features, dirs, normals, positions):
        """Light-independent half of `secondary_shading_pbr` (models/texture.py:404-434)."""
        wi = -dirs
        NoV = torch.sum(normals * wi, -1, keepdim=True)
        xyz_embd = self.xyz_encoding(positions.view(-1, self.n_pos_dims))
        network_inp = torch.cat([features.view(-1, features.shape[-1]), xyz_embd], dim=-1)
        albedo = self.albedo_network(network_inp).view(*features.shape[:-1], 6).float()[..., 3:]
        roughness = self.roughness_network(network_inp).view(*features.shape[:-1], 1).float()
        metallic = self.metallic_network(network_inp).view(*features.shape[:-1], 2).float()[..., 1:]
        albedo, metallic, roughness = self._act(albedo), self._act(metallic), self._act(roughness)
        diffuse_albedo = (1 - metallic) * albedo
        specular_albedo = 0.04 * (1 - metallic) + metallic * albedo
        fg_lookup = self._fg(NoV, roughness)
        return {"diffuse_albedo": diffuse_albedo, "roughness": roughness,
                "specular_ref": specular_albedo * fg_lookup[:, 0:1] + fg_lookup[:, 1:2]}

    def secondary_shade_pbr(self, m, dirs, normals, emitter):
        diff_rgb_pbr = m["diffuse_albedo"] * emitter.eval_mip(normals)
        specular_light = emitter.eval_mip(dirs, specular=True, roughness=m["roughness"])
        return diff_rgb_pbr + m["specular_ref"] * specular_light

    def secondary_shading_pbr(self, features, dirs, normals, positions, emitter):
        if dirs.shape[0] == 0:
            return torch.zeros((0, 3), device=dirs.device)
        return self.secondary_shade_pbr(self.secondary_material_pbr(features, dirs, normals, positions), dirs, normals,
                                        emitter)

    def update_step(self, epoch, global_step):
        update_module_step(self.dir_encoding, epoch, global_step)
        update_module_step(self.xyz_encoding, epoch, global_step)

    def regularizations(self, out):
        return {}
