"""Host-side mirror of models/geometry.py for the render path: `VolumeSDF` (the `volume-sdf`
geometry of both configs) with the reference's call signature
    forward(points, with_grad=True, with_feature=True, with_laplace=False)
(models/geometry.py:206-292).  Encoding and scan kernels come from librsdf_b200.so.
Isosurface extraction (models/geometry.py:31-112) runs on the device: the level grid on the sdf-only inference kernel,
marching cubes on csrc/mcubes.cu (`MarchingCubeHelper`, `VolumeSDF.isosurface`).
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .nerfacc import ContractionType
from .network_utils import Config, get_encoding, get_mlp, update_module_step


def scale_anything(dat, inp_scale, tgt_scale):
    """models/utils.py:109-114."""
    dat = (dat - inp_scale[0]) / (inp_scale[1] - inp_scale[0])
    if tgt_scale[0] == 0 and tgt_scale[1] == 1:
        return dat                     # `* 1 + 0` is the identity bit for bit (x01 >= 0: no -0.0)
    return dat * (tgt_scale[1] - tgt_scale[0]) + tgt_scale[0]


def contract_to_unisphere(x, radius, contraction_type):
    """models/geometry.py:17-29 (AABB branch)."""
    if contraction_type == ContractionType.AABB:
        return scale_anything(x, (-radius, radius), (0, 1))
    raise NotImplementedError("unbounded contraction belongs to the learned-background branch")


class MarchingCubeHelper(nn.Module):
    """models/geometry.py:31-68 (`isosurface.method: mc`): the surface `-level = threshold` of a [res, res, res] level
    grid, vertices scaled to [0, 1].  PyMCubes on `.cpu()` copies there, rise_sdf_b200.mcubes on the device here: the
    negation is folded into the kernel, and the outputs stay on the level's device."""

    def __init__(self, resolution):
        super().__init__()
        self.resolution = resolution

    def forward(self, level, threshold=0.0):
        from .mcubes import marching_cubes
        r = self.resolution
        level = level.float().view(r, r, r)
        verts, faces = marching_cubes(level, threshold, negate=True)
        return {"v_pos": verts / (r - 1.0), "t_pos_idx": faces}


class VolumeSDF(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config = Config(config)
        self.radius = config.radius
        self.contraction_type = ContractionType.AABB
        self.n_output_dims = config.feature_dim
        self.encoding = get_encoding(3, config.xyz_encoding_config)
        self.network = get_mlp(self.encoding.n_output_dims, self.n_output_dims, config.mlp_network_config)
        self.grad_type = config.grad_type
        self._finite_difference_eps = None
        self.finite_difference_eps = config.get("finite_difference_eps", 1e-3)
        # models/geometry.py:218-221 applies `sdf_activation(sdf + sdf_bias)` / `feature_activation(feature)` when the
        # keys are present.  Neither shipped config sets them; they are honoured on the op-by-op path and switch the
        # fused kernels (which return the raw network outputs) off.
        self._post_activations = "sdf_activation" in config or "feature_activation" in config

    def _fused_parts(self):
        """(hash-grid Encoding, level mask or None) when the analytic-normal path can run on the fused
        SDF-field kernels (csrc/sdf_train.cu): include_xyz composite over a HashGrid, SDF-shaped MLP."""
        from . import sdf_field, tinycudann as tcnn
        from .network_utils import CompositeEncoding, ProgressiveBandHashGrid, VanillaMLP
        comp = self.encoding
        if not (isinstance(comp, CompositeEncoding) and comp.include_xyz
                and isinstance(self.network, VanillaMLP) and sdf_field.supports(self.network, comp.n_output_dims)
                and self.network.config_output_activation_is_identity and not self._post_activations):
            return None
        inner, mask = comp.encoding, None
        if isinstance(inner, ProgressiveBandHashGrid):
            # all levels switched on (global_step >= start_step + (n_level - start_level) * update_steps): the mask is
            # exactly 1.0 everywhere and multiplying by it -- [S,32] forward and backward per field evaluation -- is
            # a bit-exact no-op, skipped
            inner, mask = inner.encoding, (None if inner.all_levels_on else inner.mask)
        if not (isinstance(inner, tcnn.Encoding) and inner.kind == "hashgrid"):
            return None
        return inner, mask

    def _forward_fused_analytic(self, points, parts):
        """sdf, d sdf/d points, feature with ONE fused MLP node (models/geometry.py:206-228 semantics:
        grad == autograd.grad(sdf, points, create_graph=True))."""
        from . import sdf_field, tinycudann as tcnn
        inner, mask = parts
        comp = self.encoding
        shape = points.shape[:-1]
        # (differentiable w.r.t. `points` as well: every node below returns its position leg when asked to -- the
        # curvature probe needs it, the render path proper does not)
        x01 = contract_to_unisphere(points.reshape(-1, 3), self.radius, self.contraction_type).contiguous().float()
        y, dy_dx, link = tcnn.hashgrid_with_jacobian(inner, x01)
        enc = y if mask is None else y * mask
        out, sdf, g0_xyz, g0_enc = sdf_field.fused_sdf_parts(self.network, x01, comp.xyz_scale, comp.xyz_offset, enc)
        g_enc = g0_enc if mask is None else g0_enc * mask
        grad_x01 = tcnn.hashgrid_input_grad(inner, g_enc, x01, dy_dx, link) + g0_xyz * comp.xyz_scale
        grad = grad_x01 / (2.0 * self.radius)          # d x01 / d points (scale_anything)
        return sdf.view(*shape), grad.view(*shape, 3), out.view(*shape, self.n_output_dims)

    def _field(self, x01, sdf_only=False):
        """network(encoding(x01)) for x01 [S,3] in the unit cube (sdf_only: just channel 0, [S]).  On the fused kernels the MLP reads the two
        segments (x01 with the xyz affine, hash features) directly: no [S,35] concatenation, and under
        no_grad (eval / relighting / occupancy update / the 7 finite-difference evaluations per sample of
        the split-sum config) no autograd bookkeeping either."""
        from . import sdf_field
        parts = self._fused_parts() if (x01.is_cuda and not x01.requires_grad and x01.shape[0] > 0) else None
        if parts is None:
            out = self.network(self.encoding(x01))
            return out[..., 0] if sdf_only else out
        inner, mask = parts
        comp = self.encoding
        y = inner(x01)
        if mask is not None:
            y = y * mask
        # (_fused_parts: the output activation is the identity; sdf_only writes just the sdf head, 4 B instead of 192 B
        # per point)
        if not torch.is_grad_enabled():
            return self.network.packed()(x01, comp.xyz_scale, comp.xyz_offset, y, sdf_only=sdf_only)
        out, sdf, _, _ = sdf_field.fused_sdf_parts(self.network, x01, comp.xyz_scale, comp.xyz_offset, y, want_g0=False,
                                                   sdf_only=sdf_only)
        return sdf if sdf_only else out

    def _fd6_sdf(self, points, eps):
        """sdf at the six finite-difference neighbours of `points` [..., 3] -> [..., 6], or None when the fused
        path does not apply.  One hash-grid launch builds the neighbours exactly as the reference does (add, clamp,
        scale: models/geometry.py:229-237) and re-gathers corners only when a neighbour leaves the previous one's
        cell; the MLP then writes just the sdf head.  Under autograd the hash-grid launch is differentiable w.r.t. the
        table and the MLP is the sdf-only fused node -- instead of building the 6S neighbour positions with torch ops
        and running the generic hash-grid forward over them."""
        from . import sdf_field, tinycudann as tcnn
        grad = torch.is_grad_enabled()
        if not points.is_cuda or points.numel() == 0 or (grad and points.requires_grad):
            return None
        parts = self._fused_parts()
        if parts is None:
            return None
        inner, mask = parts
        comp = self.encoding
        fd6 = tcnn.hashgrid_fd6_train if grad else tcnn.hashgrid_fd6
        x01, y = fd6(inner, points.reshape(-1, 3), eps, self.radius)
        if mask is not None:
            y = y * mask
        if grad:
            _, sdf, _, _ = sdf_field.fused_sdf_parts(self.network, x01, comp.xyz_scale, comp.xyz_offset, y,
                                                     want_g0=False, sdf_only=True)
        else:
            sdf = self.network.packed()(x01, comp.xyz_scale, comp.xyz_offset, y, sdf_only=True)
        return sdf.view(*points.shape[:-1], 6)

    def forward(self, points, with_grad=True, with_feature=True, with_laplace=False):
        analytic = with_grad and self.grad_type == "analytic"
        # (sample positions are data on the render path; a caller that differentiates w.r.t. the points
        # themselves takes the op-by-op autograd path below)
        parts = self._fused_parts() if (analytic and points.is_cuda and not with_laplace
                                        and not points.requires_grad) else None
        if parts is not None:
            with torch.set_grad_enabled(self.training and torch.is_grad_enabled()):
                sdf, grad, feature = self._forward_fused_analytic(points, parts)
            rv = [sdf, grad] + ([feature] if with_feature else [])
            return [v if self.training else v.detach() for v in rv]
        # The reference enables grad whenever self.training (models/geometry.py:208), even when the
        # caller sits under no_grad (occupancy update, sampling's alpha_fn) and the graph is thrown
        # away (SURVEY.md Appendix F).  Same numbers, no wasted graph: only build it if it can be used.
        with torch.set_grad_enabled((self.training and torch.is_grad_enabled()) or analytic):
            if analytic:
                if not self.training:
                    points = points.clone()
                points.requires_grad_(True)
            points_ = points
            points = contract_to_unisphere(points, self.radius, self.contraction_type)
            out = self._field(points.view(-1, 3)).view(*points.shape[:-1], self.n_output_dims).float()
            sdf, feature = out[..., 0], out
            if "sdf_activation" in self.config:
                from .network_utils import get_activation
                sdf = get_activation(self.config.sdf_activation)(sdf + float(self.config.sdf_bias))
            if "feature_activation" in self.config:
                from .network_utils import get_activation
                feature = get_activation(self.config.feature_activation)(feature)
            if with_grad:
                if self.grad_type == "analytic":
                    grad = torch.autograd.grad(sdf, points_, grad_outputs=torch.ones_like(sdf),
                                               create_graph=True, retain_graph=True, only_inputs=True)[0]
                elif self.grad_type == "finite_difference":
                    eps = self._finite_difference_eps
                    points_d_sdf = self._fd6_sdf(points_, eps)
                    if points_d_sdf is None:
                        offsets = torch.as_tensor([[eps, 0.0, 0.0], [-eps, 0.0, 0.0], [0.0, eps, 0.0],
                                                   [0.0, -eps, 0.0], [0.0, 0.0, eps], [0.0, 0.0, -eps]]).to(points_)
                        points_d_ = (points_[..., None, :] + offsets).clamp(-self.radius, self.radius)
                        points_d = scale_anything(points_d_, (-self.radius, self.radius), (0, 1))
                        points_d_sdf = self._field(points_d.view(-1, 3), sdf_only=True).view(*points.shape[:-1], 6).float()
                    grad = 0.5 * (points_d_sdf[..., 0::2] - points_d_sdf[..., 1::2]) / eps
                    if with_laplace:
                        # curvature probe (models/geometry.py:246-282)
                        eps_c = 1e-4
                        rand_directions = F.normalize(torch.rand_like(points_), dim=-1, eps=1e-6)
                        normal = F.normalize(grad, dim=-1, eps=1e-6)
                        tangent = torch.cross(normal, rand_directions, dim=-1)
                        points_t_ = points_ + eps_c * tangent
                        if not points_t_.requires_grad:
                            points_t_ = points_t_.requires_grad_(True)
                        probe = self._fused_parts() if points_t_.is_cuda else None
                        if probe is not None:
                            # d sdf / d points_t with its full second-order graph (weights, table AND the probe
                            # position, which depends on the parameters through `tangent`) on the fused kernels:
                            # hash grid + Jacobian -> one fused MLP node -> dy_dx^T g0, exactly the analytic-normal path
                            _, grad_t, _ = self._forward_fused_analytic(points_t_, probe)
                        else:
                            points_t = contract_to_unisphere(points_t_, self.radius, self.contraction_type)
                            sdf_t = self.network(self.encoding(points_t.view(-1, 3)))[..., 0].view(*points.shape[:-1]).float()
                            grad_t = torch.autograd.grad(sdf_t, points_t_, grad_outputs=torch.ones_like(sdf_t),
                                                         create_graph=True, retain_graph=True, only_inputs=True)[0]
                        dot = torch.sum(F.normalize(grad, dim=-1, eps=1e-6) * F.normalize(grad_t, dim=-1, eps=1e-6), dim=-1)
                        laplace = torch.acos(torch.clamp(dot, -1.0 + 1e-6, 1.0 - 1e-6)) / np.pi
        rv = [sdf]
        if with_grad:
            rv.append(grad)
        if with_feature:
            rv.append(feature)
        if with_laplace:
            assert self.grad_type == "finite_difference", \
                "Laplace computation is only supported with grad_type='finite_difference'"
            rv.append(laplace)
        rv = [v if self.training else v.detach() for v in rv]
        return rv[0] if len(rv) == 1 else rv

    # ------------------------------------------------------------------ isosurface query (models/geometry.py:76-112)
    @torch.no_grad()
    def forward_level(self, points):
        """models/geometry.py:294-299: sdf at world-space points, no gradients (sdf-only inference kernel)."""
        x01 = contract_to_unisphere(points.reshape(-1, 3), self.radius, self.contraction_type)
        sdf = self._field(x01.contiguous().float(), sdf_only=True).view(*points.shape[:-1])
        if "sdf_activation" in self.config:
            from .network_utils import get_activation
            sdf = get_activation(self.config.sdf_activation)(sdf + float(self.config.sdf_bias))
        return sdf

    @torch.no_grad()
    def isosurface_level(self, resolution=512, vmin=None, vmax=None, chunk=1 << 22, out=None):
        """The level grid `BaseImplicitGeometry.isosurface_` evaluates before marching cubes (models/geometry.py:76-91):
        sdf at the resolution^3 vertices of linspace(0, 1, resolution)^3 scaled into [vmin, vmax] (default: the whole
        [-radius, radius]^3 box), x-major like `MarchingCubeHelper.grid_vertices` (:43-49).  The reference moves 2 M-point
        chunks to the GPU and back (`.cpu()` per chunk); here the vertices are generated on the device chunk by chunk
        (nothing but the [resolution^3] result is ever materialised: 512 MB at 512^3) and each chunk is one hash-grid
        launch + one sdf-only tcgen05 inference launch.  Returns a float32 tensor [resolution, resolution, resolution]."""
        r = int(resolution)
        dev = next(self.parameters()).device
        lo = torch.as_tensor([-self.radius] * 3 if vmin is None else vmin, dtype=torch.float32, device=dev)
        hi = torch.as_tensor([self.radius] * 3 if vmax is None else vmax, dtype=torch.float32, device=dev)
        level = out if out is not None else torch.empty(r ** 3, device=dev, dtype=torch.float32)
        lin = torch.linspace(0.0, 1.0, r, device=dev)
        for s in range(0, r ** 3, chunk):
            idx = torch.arange(s, min(s + chunk, r ** 3), device=dev)
            v = torch.stack([lin[idx // (r * r)], lin[(idx // r) % r], lin[idx % r]], -1)
            level[s:s + idx.numel()] = self.forward_level(v * (hi - lo) + lo)       # scale_anything((0,1) -> (vmin, vmax))
        return level.view(r, r, r)

    @torch.no_grad()
    def isosurface_bounds(self, level, vmin=None, vmax=None, threshold=0.0):
        """World-space bounding box of the level set: the cells whose corner values straddle `threshold`.  The reference
        takes it from the coarse marching-cubes mesh (models/geometry.py:104-110) to place the fine grid; marching cubes
        itself (PyMCubes, a CPU third-party dependency) is not part of the path."""
        r = level.shape[0]
        dev = level.device
        lo = torch.as_tensor([-self.radius] * 3 if vmin is None else vmin, dtype=torch.float32, device=dev)
        hi = torch.as_tensor([self.radius] * 3 if vmax is None else vmax, dtype=torch.float32, device=dev)
        inside = level > threshold
        cross = torch.zeros(r, r, r, dtype=torch.bool, device=dev)
        for d in range(3):
            a, b = inside.narrow(d, 0, r - 1), inside.narrow(d, 1, r - 1)
            c = a != b
            cross.narrow(d, 0, r - 1).logical_or_(c)
            cross.narrow(d, 1, r - 1).logical_or_(c)
        nz = torch.nonzero(cross)
        if nz.numel() == 0:
            return None
        mn, mx = nz.min(0).values.float() / (r - 1), nz.max(0).values.float() / (r - 1)
        bmin, bmax = mn * (hi - lo) + lo, mx * (hi - lo) + lo
        pad = (bmax - bmin) * 0.1                                                  # :106-107
        return (bmin - pad).clamp(-self.radius, self.radius), (bmax + pad).clamp(-self.radius, self.radius)

    @torch.no_grad()
    def isosurface(self, resolution=512, threshold=0.0):
        """`BaseImplicitGeometry.isosurface` (models/geometry.py:76-112): a coarse mesh over the whole [-radius, radius]^3
        box places a fine grid on its bounding box padded by 10 % and clamped to the radius; returns the fine mesh
        {'v_pos' [V,3] world space, 't_pos_idx' [F,3] int64} on the device.  Both level grids share one buffer.  An
        empty coarse mesh (no surface in the box) gives an empty mesh."""
        helper = MarchingCubeHelper(resolution)
        dev = next(self.parameters()).device
        buf = torch.empty(resolution ** 3, device=dev, dtype=torch.float32)
        r = self.radius
        vmin = torch.full((3,), -r, dtype=torch.float32, device=dev)
        vmax = torch.full((3,), r, dtype=torch.float32, device=dev)
        for fine in (False, True):
            level = self.isosurface_level(resolution, vmin, vmax, out=buf)
            mesh = helper(level, threshold)
            mesh["v_pos"] = mesh["v_pos"] * (vmax - vmin) + vmin           # scale_anything((0, 1) -> (vmin, vmax))
            if fine or mesh["v_pos"].shape[0] == 0:
                return mesh
            lo, hi = mesh["v_pos"].amin(dim=0), mesh["v_pos"].amax(dim=0)
            vmin = (lo - (hi - lo) * 0.1).clamp(-r, r)
            vmax = (hi + (hi - lo) * 0.1).clamp(-r, r)

    def update_step(self, epoch, global_step):
        update_module_step(self.encoding, epoch, global_step)
        update_module_step(self.network, epoch, global_step)
        if self.grad_type == "finite_difference":
            if isinstance(self.finite_difference_eps, float):
                self._finite_difference_eps = self.finite_difference_eps
            elif self.finite_difference_eps == "progressive":
                hg = self.config.xyz_encoding_config
                assert hg.otype == "ProgressiveBandHashGrid"
                level = min(hg.start_level + max(global_step - hg.start_step, 0) // hg.update_steps, hg.n_levels)
                grid_res = hg.base_resolution * hg.per_level_scale ** (level - 1)
                self._finite_difference_eps = 2 * self.config.radius / grid_res
            else:
                raise ValueError(f"Unknown finite_difference_eps={self.finite_difference_eps}")

    def regularizations(self, out):
        if "normals_orientation_loss_map" in out:
            return {"normal_orientation": out["normals_orientation_loss_map"].mean()}
        return {}
