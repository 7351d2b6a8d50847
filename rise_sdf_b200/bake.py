"""Bake the split-sum model's materials into a texture atlas, for `SplitMixedOCCModel.export()`.

Albedo, roughness and metallic of `VolumeMixedMipSplitOcc` depend on the surface point alone (the material networks
read [feature, VanillaFrequency(position)], models/texture.py), so they can be stored in textures and used by any
renderer that reads glTF's `pbrMetallicRoughness` material.  Without a UV unwrapper, every face gets a chart of its
own: faces are paired into square cells of a T x T atlas (layout and texel rule: include/rsdf_b200.h,
`rsdf_bake_uv`), and every texel a face owns holds the materials at its surface point.  Bilinear sampling inside a
face's UV triangle reads only texels of that face, so the atlas needs no gutters.

The atlas is evaluated in bands of texel rows: csrc/bake.cu gives each texel of the band its face and surface point,
the geometry feature and the three material networks run on the existing no-grad kernels, and `rsdf_material_pack`
applies the sigmoid and writes the band's rows of the atlas.  Device memory beyond the atlas is bounded by the band.

The optional normal map carries the surface detail the mesh is too coarse for: every texel holds the model's own
shading normal, normalize(grad) of the SDF at its surface point (finite differences or analytic, as the model's
`grad_type` says), in the tangent frame a glTF viewer builds from the mesh's NORMAL and TANGENT (`atlas_tangents`,
`rsdf_bake_tangents`; `rsdf_normal_pack` writes the band's rows).  `bake_atlases` evaluates the field once per band for
both atlases: the geometry call that returns the gradient returns the feature the material networks read.
"""
import math

import torch

from . import _lib as L

MIN_TEXTURE, MAX_TEXTURE = 16, 16384
MIN_CELL = 4                   # a cell must hold triangle A's corners (0, 0), (C-3, 0), (0, C-3) with C - 3 >= 1


def atlas_layout(n_faces, texture_size):
    """(C, cols) of the atlas of `n_faces` faces in a texture of `texture_size`^2 texels: P = ceil(F / 2) cells of
    C x C texels, `cols` per row, C = T // cols.  Raises ValueError when T is outside [16, 16384] or C < 4."""
    F, T = int(n_faces), int(texture_size)
    if F < 0:
        raise ValueError(f"n_faces must be non-negative, got {F}")
    if not MIN_TEXTURE <= T <= MAX_TEXTURE:
        raise ValueError(f"texture_size must be in [{MIN_TEXTURE}, {MAX_TEXTURE}], got {T}")
    P = (F + 1) // 2
    cols = max(1, math.isqrt(P - 1) + 1 if P > 0 else 0)
    C = T // cols
    if C < MIN_CELL:
        raise ValueError(f"{F} faces need a texture of at least {MIN_CELL * cols} texels per side "
                         f"({cols} cells of {MIN_CELL} x {MIN_CELL} per row); texture_size is {T}")
    return C, cols


def atlas_uv(n_faces, texture_size, device):
    """Per-corner glTF UVs float32 [F, 3, 2] of the atlas layout (`rsdf_bake_uv`)."""
    atlas_layout(n_faces, texture_size)
    t_uv = torch.empty(int(n_faces), 3, 2, dtype=torch.float32, device=device)
    if n_faces:
        L.call("rsdf_bake_uv", int(n_faces), int(texture_size), L.ptr(t_uv), L.stream())
    return t_uv


def _check_model(model):
    if model.texture.config.get("color_activation", None) != "sigmoid":
        raise ValueError("material baking applies the sigmoid `color_activation` of the split-sum config; this "
                         f"texture has {model.texture.config.get('color_activation', None)!r}")


def _materials(model, points, face_id, out, feature=None):
    """materials of `points` [n, 3] into `out` [n, 5] (rows with face id -1 are 0); `feature`: the geometry feature at
    `points` when the caller has it"""
    if feature is None:
        _, feature = model.geometry(points, with_grad=False, with_feature=True)
    raw6, raw1, raw2 = model.texture.material_nets(feature, points)
    raw6, raw1, raw2 = raw6.contiguous(), raw1.contiguous(), raw2.contiguous()
    L.call("rsdf_material_pack", L.ptr(raw6), L.ptr(raw1), L.ptr(raw2), L.ptr(face_id), points.shape[0], L.ptr(out),
           L.stream())


def _chunk(chunk_size):
    chunk_size = int(chunk_size)
    if chunk_size < 1:
        raise ValueError(f"chunk_size must be positive, got {chunk_size}")
    return chunk_size


@torch.no_grad()
def material_at(model, points, chunk_size=1 << 20):
    """Materials of a `SplitMixedOCCModel` at world-space points [N, 3] (CUDA): float32 [N, 5] = (albedo rgb,
    roughness, metallic), linear, in [0, 1].  Evaluated `chunk_size` points at a time."""
    L.require_cuda(points)
    _check_model(model)
    chunk_size = _chunk(chunk_size)
    points = points.detach().reshape(-1, 3).float().contiguous()
    out = torch.empty(points.shape[0], 5, dtype=torch.float32, device=points.device)
    for s in range(0, points.shape[0], chunk_size):
        _materials(model, points[s:s + chunk_size], None, out[s:s + chunk_size])
    return out


@torch.no_grad()
def atlas_tangents(v_pos, t_pos_idx, v_nrm, texture_size):
    """glTF TANGENTs float32 [F, 3, 4] of the atlas layout, one per face corner (`rsdf_bake_tangents`): the atlas's +u
    direction made orthogonal to the corner's normal `v_nrm` [V, 3], and w = +-1 per face so that w cross(N, T) points
    image-up.  Raises ValueError like `atlas_layout`."""
    L.require_cuda(v_pos, t_pos_idx, v_nrm)
    F = t_pos_idx.shape[0]
    atlas_layout(F, texture_size)
    t_tangent = torch.empty(F, 3, 4, dtype=torch.float32, device=v_pos.device)
    if F:
        v_pos = v_pos.detach().float().contiguous()
        v_nrm = v_nrm.detach().float().contiguous()
        t_pos_idx = t_pos_idx.detach().to(torch.int64).contiguous()
        L.call("rsdf_bake_tangents", L.ptr(v_pos), L.ptr(t_pos_idx), L.ptr(v_nrm), F, int(texture_size),
               L.ptr(t_tangent), L.stream())
    return t_tangent


def _bake_bands(model, v_pos, t_pos_idx, texture_size, chunk_size, materials, normals):
    """(material atlas [T, T, 5] if `materials` else None, normal atlas [T, T, 3] if `normals` = (v_nrm, t_tangent)
    else None), one geometry call per band of texel rows"""
    L.require_cuda(v_pos, t_pos_idx)
    if materials:
        _check_model(model)
    T = int(texture_size)
    F = t_pos_idx.shape[0]
    C, cols = atlas_layout(F, T)
    dev = v_pos.device
    atlas = torch.zeros(T, T, 5, dtype=torch.float32, device=dev) if materials else None
    normal_atlas = None
    if normals is not None:
        v_nrm, t_tangent = normals
        L.require_cuda(v_nrm, t_tangent)
        if tuple(t_tangent.shape) != (F, 3, 4):
            raise ValueError(f"t_tangent must be [{F}, 3, 4] for {F} faces, got {list(t_tangent.shape)}")
        v_nrm = v_nrm.detach().float().contiguous()
        t_tangent = t_tangent.detach().float().contiguous()
        normal_atlas = torch.zeros(T, T, 3, dtype=torch.float32, device=dev)
        normal_atlas[..., 2] = 1.0                                   # unowned texels: flat
    if F == 0:
        return atlas, normal_atlas
    v_pos = v_pos.detach().float().contiguous()
    t_pos_idx = t_pos_idx.detach().to(torch.int64).contiguous()
    rows = -(-((F + 1) // 2) // cols) * C                    # texel rows that hold cells
    band = min(max(1, _chunk(chunk_size) // T), rows)
    face_id = torch.empty(band * T, dtype=torch.int32, device=dev)
    points = torch.empty(band * T, 3, dtype=torch.float32, device=dev)
    # the analytic gradient's feature comes from the training kernels; bake_material_atlas's from the inference ones
    shared = normals is None or model.geometry.grad_type == "finite_difference"
    for r0 in range(0, rows, band):
        n = min(band, rows - r0)
        pts = points[:n * T]
        L.call("rsdf_bake_texels", L.ptr(v_pos), L.ptr(t_pos_idx), F, T, r0, n, L.ptr(face_id), L.ptr(pts),
               L.stream())
        feature = None
        if normals is not None:
            _, grad, feature = model.geometry(pts, with_grad=True, with_feature=True)
            grad = grad.float().contiguous()
            L.call("rsdf_normal_pack", L.ptr(v_nrm), L.ptr(t_pos_idx), L.ptr(t_tangent), F, T, r0, n, L.ptr(grad),
                   L.ptr(normal_atlas.view(T * T, 3)[r0 * T:(r0 + n) * T]), L.stream())
        if materials:
            _materials(model, pts, face_id[:n * T], atlas.view(T * T, 5)[r0 * T:(r0 + n) * T],
                       feature if shared else None)
    return atlas, normal_atlas


@torch.no_grad()
def bake_material_atlas(model, v_pos, t_pos_idx, texture_size=8192, chunk_size=1 << 20):
    """The material atlas of the mesh (v_pos float32 [V, 3], t_pos_idx int64 [F, 3], CUDA): float32 [T, T, 5] of
    (albedo rgb, roughness, metallic), row 0 on top, 0 where no face owns the texel; UVs from `atlas_uv`.  Bands of
    max(1, chunk_size // T) texel rows are evaluated one at a time, over the rows that hold cells only."""
    return _bake_bands(model, v_pos, t_pos_idx, texture_size, chunk_size, True, None)[0]


@torch.no_grad()
def bake_normal_atlas(model, v_pos, t_pos_idx, v_nrm, t_tangent, texture_size=8192, chunk_size=1 << 20):
    """The tangent-space normal atlas of the mesh: float32 [T, T, 3], per texel the unit field normal
    normalize(model.geometry(point, with_grad=True)) at its surface point in the frame of the interpolated vertex
    normal `v_nrm` [V, 3] and corner tangents `t_tangent` [F, 3, 4] (`atlas_tangents`): (x along T, y along
    B = w cross(N, T), z along N); (0, 0, 1) where no face owns the texel.  Banded like `bake_material_atlas`."""
    return _bake_bands(model, v_pos, t_pos_idx, texture_size, chunk_size, False, (v_nrm, t_tangent))[1]


@torch.no_grad()
def bake_atlases(model, v_pos, t_pos_idx, v_nrm, t_tangent, texture_size=8192, chunk_size=1 << 20):
    """(`bake_material_atlas`, `bake_normal_atlas`) of the mesh from one geometry evaluation per band.  With the
    split-sum config's finite-difference gradient the material atlas is bit-identical to `bake_material_atlas`'s."""
    return _bake_bands(model, v_pos, t_pos_idx, texture_size, chunk_size, True, (v_nrm, t_tangent))
