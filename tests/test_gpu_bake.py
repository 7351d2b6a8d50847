"""Material baking for `SplitMixedOCCModel.export()` on the B200: csrc/bake.cu against the float32 layout oracle (bit for
bit), the baked atlas against the op-by-op torch material path and the fp64 CPU oracle, the atlas against the
per-vertex materials, the end-to-end export and its glTF file, and the band's memory and read-back bounds."""
import json
import struct

import numpy as np
import pytest
import torch

from oracle import bake as ob
from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import bake, formats

pytestmark = pytest.mark.gpu


def _split_model(base_res=64):
    """the seeded split-sum test model of tests/test_gpu_splitsum.py, in stage 1 with every hash-grid level on"""
    from rise_sdf_b200.split_mixed_occ import SplitMixedOCCModel, split_mixed_occ_config
    torch.manual_seed(0)
    cfg = split_mixed_occ_config()
    cfg["light"]["envlight_config"]["base_res"] = base_res
    m = SplitMixedOCCModel(cfg).cuda()
    with torch.no_grad():
        m.geometry.network.layers[0].weight_v[:, 3:].normal_(0.0, 0.05)
        m.variance.variance.fill_(0.5)
        m.geometry.encoding.encoding.encoding.params.uniform_(-0.02, 0.02)
    m.eval()
    m.update_step(0, 20000)
    assert m.stage == 1
    return m


@pytest.fixture(scope="module")
def model():
    return _split_model()


def _texels(v, f, T, row0, n_rows):
    face = torch.empty(n_rows * T, dtype=torch.int32, device="cuda")
    pts = torch.empty(n_rows * T, 3, dtype=torch.float32, device="cuda")
    L.call("rsdf_bake_texels", L.ptr(v), L.ptr(f), f.shape[0], T, row0, n_rows, L.ptr(face), L.ptr(pts), L.stream())
    return face, pts


def test_bake_kernels_match_oracle():
    rng = np.random.default_rng(0)
    V, F = 500, 777                                            # odd: the last pair has no triangle B
    v_np = (rng.standard_normal((V, 3)) * 3).astype(np.float32)
    f_np = rng.integers(0, V, (F, 3))
    v, f = torch.from_numpy(v_np).cuda(), torch.from_numpy(f_np).cuda()
    for T in (80, 97, 256):
        C, cols = bake.atlas_layout(F, T)
        uv = bake.atlas_uv(F, T, "cuda").cpu().numpy()
        assert np.array_equal(uv.view(np.uint32), ob.uv(F, T).view(np.uint32))
        want_face, want_pts = ob.texels(v_np, f_np, T, 0, T)
        for band in (T, C + 3):                                # C + 3: bands cut through cells
            got = [_texels(v, f, T, r0, min(band, T - r0)) for r0 in range(0, T, band)]
            face = torch.cat([g[0] for g in got]).cpu().numpy()
            pts = torch.cat([g[1] for g in got]).cpu().numpy()
            assert np.array_equal(face, want_face)
            assert np.array_equal(pts.view(np.uint32), want_pts.view(np.uint32))
    with pytest.raises(RuntimeError, match="bad argument"):
        L.call("rsdf_bake_uv", F, 16, L.ptr(torch.empty(F, 3, 2, device="cuda")), L.stream())


def _op_by_op_materials(m, pts):
    """albedo, roughness, metallic of the unfused torch material path (texture.material, stage 1)"""
    with torch.no_grad():
        _, feat = m.geometry(pts, with_grad=False, with_feature=True)
        nrm = torch.zeros_like(pts)
        nrm[:, 2] = 1.0
        m.texture.fused_shade = False
        try:
            mat = m.texture.material(feat, -nrm, nrm, pts, stage=1)
        finally:
            del m.texture.fused_shade
    return torch.cat([mat["albedo"], mat["roughness"], mat["metallic"]], -1), feat, nrm


def test_atlas_matches_torch_and_fp64_oracle(model):
    from helpers import split_oracle_params
    from oracle import split as osplit
    m = model
    mesh = m.geometry.isosurface(64)
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    T = 512
    atlas = bake.bake_material_atlas(m, v, f, T, chunk_size=1 << 16)
    face, pts = _texels(v, f, T, 0, T)
    owned = torch.nonzero(face >= 0)[:, 0]
    g = torch.Generator(device="cpu").manual_seed(1)
    pick = owned[torch.randperm(owned.numel(), generator=g)[:4096].cuda()]
    got = atlas.view(-1, 5)[pick]
    want, feat, nrm = _op_by_op_materials(m, pts[pick])
    assert float((got - want).abs().max()) <= 1e-5
    assert torch.equal(bake.material_at(m, pts[pick]), got)
    with torch.no_grad():
        m.emitter.build_mips()
    P = split_oracle_params(m).to(torch.float64)
    P.specular = [t.detach().cpu().double() for t in m.emitter.specular]
    P.diffuse = m.emitter.diffuse.detach().cpu().double()
    d = lambda t: t.detach().cpu().double()
    ref = osplit.texture_forward(P, d(feat), d(-nrm), d(nrm), d(pts[pick]), stage=1)
    ref = torch.cat([ref[:, 19:22], ref[:, 23:24], ref[:, 22:23]], -1)      # albedo, roughness, metallic
    assert float((got.cpu().double() - ref).abs().max()) <= 1e-4
    assert float(atlas.view(-1, 5)[face < 0].abs().max()) == 0.0


def _read_glb_json(path):
    buf = open(path, "rb").read()
    magic, version, length = struct.unpack_from("<III", buf, 0)
    assert magic == 0x46546C67 and version == 2 and length == len(buf)
    jlen, _ = struct.unpack_from("<II", buf, 12)
    return json.loads(buf[20:20 + jlen])


def test_export_end_to_end(model, tmp_path):
    m = model
    T = 1024
    out = m.export(chunk_size=1 << 16, resolution=128, texture_size=T)
    mesh = m.geometry.isosurface(128)
    v, f = out["v_pos"], out["t_pos_idx"]
    assert torch.equal(v, mesh["v_pos"]) and torch.equal(f, mesh["t_pos_idx"])
    V, F = v.shape[0], f.shape[0]
    assert V > 1000 and F > 1000
    assert out["v_nrm"].shape == (V, 3) and out["v_albedo"].shape == (V, 3)
    assert out["v_roughness"].shape == (V, 1) and out["v_metallic"].shape == (V, 1)
    assert out["t_uv"].shape == (F, 3, 2) and out["material_atlas"].shape == (T, T, 5)
    atlas = out["material_atlas"]
    for k in ("v_albedo", "v_roughness", "v_metallic", "material_atlas"):
        assert float(out[k].min()) >= 0.0 and float(out[k].max()) <= 1.0
    face, _ = _texels(v, f, T, 0, T)
    assert float(atlas.view(-1, 5)[face < 0].abs().max()) == 0.0
    # the texel at each face corner's UV is the vertex itself: it holds the per-vertex materials
    tex = torch.round(out["t_uv"] * T - 0.5).long()                               # [F, 3, 2] (column, row)
    at_corner = atlas[tex[..., 1], tex[..., 0]]                                   # [F, 3, 5]
    v_mat = torch.cat([out["v_albedo"], out["v_roughness"], out["v_metallic"]], -1)[f]
    assert float((at_corner - v_mat).abs().max()) <= 1e-6
    assert torch.equal(face.view(T, T)[tex[..., 1], tex[..., 0]].long(),
                       torch.arange(F, device="cuda")[:, None].expand(F, 3))
    # deterministic
    again = m.export(chunk_size=1 << 16, resolution=128, texture_size=T)
    for k, t in out.items():
        assert torch.equal(t, again[k]), k
    path = formats.save_mesh_glb(str(tmp_path / "split.glb"), out)
    gltf = _read_glb_json(path)
    (prim,) = gltf["meshes"][0]["primitives"]
    acc = gltf["accessors"]
    assert acc[prim["attributes"]["POSITION"]]["count"] == 3 * F == acc[prim["indices"]]["count"]
    assert acc[prim["attributes"]["TEXCOORD_0"]]["count"] == 3 * F == acc[prim["attributes"]["NORMAL"]]["count"]
    assert len(gltf["images"]) == 2 and prim["material"] == 0


def _winding_agreement(mesh):
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    p = v[f]
    wn = torch.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0], dim=-1)
    return float(((wn * mesh["v_nrm"][f].mean(1)).sum(-1) > 0).float().mean())


def test_export_winding_agrees_with_normals(model):
    """The faces' winding agrees with the exported vertex normals.  The test model's U(-0.02, 0.02) hash table puts
    noise into the finest levels that dominates the finite-difference normal (eps = one finest-level cell, 3.7e-4):
    there about 71 % of the faces agree (B200).  With the table scaled by 0.01 the field is smooth at the mesh's scale and
    the normals test the winding (100 % agree on the B200)."""
    print(f"winding agreement, test model: {_winding_agreement(model.export(resolution=128, texture_size=1024)):.4f}")
    smooth = _split_model()
    with torch.no_grad():
        smooth.geometry.encoding.encoding.encoding.params.mul_(0.01)
    agree = _winding_agreement(smooth.export(resolution=128, texture_size=1024))
    print(f"winding agreement, smooth table: {agree:.4f}")
    assert agree >= 0.99


def test_band_memory_and_read_backs(model):
    m = model
    mesh = m.geometry.isosurface(128)
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    band = 1 << 18
    T = 2048

    def peak(chunk):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        atlas = bake.bake_material_atlas(m, v, f, T, chunk_size=chunk)
        torch.cuda.synchronize()
        extra = torch.cuda.max_memory_allocated() - base - atlas.numel() * 4
        del atlas
        return extra

    bake.bake_material_atlas(m, v, f, T, chunk_size=band)                 # warm-up: weight caches
    banded, whole = peak(band), peak(T * T)
    print(f"peak beyond atlas + mesh: band of {band} texels {banded / band:.0f} B/texel, whole atlas "
          f"{whole / band:.0f} B per band texel")
    assert banded <= 4096 * band
    assert whole > 4096 * band

    def d2h(T):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            bake.bake_material_atlas(m, v, f, T, chunk_size=band)
            torch.cuda.synchronize()
        return sum(e.count for e in prof.key_averages() if "DtoH" in e.key or "Device -> Pageable" in e.key)

    def n_bands(T):
        C, cols = bake.atlas_layout(f.shape[0], T)
        rows = -(-((f.shape[0] + 1) // 2) // cols) * C
        return -(-rows // max(1, band // T))

    assert n_bands(4096) > n_bands(1024)
    assert d2h(1024) == d2h(4096)


def test_export_errors(model):
    m = model
    with pytest.raises(ValueError, match="texels per side"):
        m.export(resolution=64, texture_size=16)
    with pytest.raises(NotImplementedError, match="Only support cuda inputs."):
        bake.material_at(m, torch.zeros(4, 3))
    cpu = _split_model(base_res=16).cpu()
    with pytest.raises(NotImplementedError, match="Only support cuda inputs."):
        cpu.export(resolution=32)
