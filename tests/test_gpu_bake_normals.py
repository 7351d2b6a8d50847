"""The normal map of `SplitMixedOCCModel.export(normal_map=True)` on the B200: csrc/bake.cu's `rsdf_bake_tangents` and
`rsdf_normal_pack` against the float32 oracle (bit for bit), the baked map decoded as a glTF viewer does against the
field normal it stores (float and after the 8-bit PNG of the `.glb`), the map against the interpolated vertex normals,
the export's other entries, and the band's memory and read-back bounds."""
import math

import cv2
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bake_normals as obn
from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import bake, formats
from test_gpu_bake import _split_model, _texels
from test_mesh_glb import read_glb, view_bytes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    return _split_model()


@pytest.fixture(scope="module")
def smooth():
    """the test model with its hash table scaled by 0.01: smooth at the mesh's scale (test_export_winding_agrees_with_normals)"""
    m = _split_model()
    with torch.no_grad():
        m.geometry.encoding.encoding.encoding.params.mul_(0.01)
    return m


def _pack(v_nrm, f, t_tangent, T, row0, n_rows, grad):
    out = torch.empty(n_rows * T, 3, dtype=torch.float32, device="cuda")
    L.call("rsdf_normal_pack", L.ptr(v_nrm), L.ptr(f), L.ptr(t_tangent), f.shape[0], T, row0, n_rows, L.ptr(grad),
           L.ptr(out), L.stream())
    return out


def test_normal_kernels_match_oracle():
    rng = np.random.default_rng(0)
    V, Fn = 500, 777                                           # odd: the last pair has no triangle B
    v_np = (rng.standard_normal((V, 3)) * 3).astype(np.float32)
    f_np = rng.integers(0, V, (Fn, 3))
    f_np[:7, 1] = f_np[:7, 0]                                  # zero e1: fallback tangents, w = +1
    n_np = rng.standard_normal((V, 3)).astype(np.float32)
    n_np[:V // 2] /= np.linalg.norm(n_np[:V // 2], axis=1, keepdims=True)
    n_np[:5] = 0.0                                             # zero normals
    n_np[5] = [1.0, 0.0, 0.0]
    v_pos, f, v_nrm = (torch.from_numpy(a).cuda() for a in (v_np, f_np, n_np))
    for T in (80, 97, 256):
        C, cols = bake.atlas_layout(Fn, T)
        tan = bake.atlas_tangents(v_pos, f, v_nrm, T)
        want_tan = obn.tangents(v_np, f_np, n_np)
        assert np.array_equal(tan.cpu().numpy().view(np.uint32), want_tan.view(np.uint32))
        grad_np = (rng.standard_normal((T * T, 3)) * 2).astype(np.float32)
        grad_np[::17] = 0.0                                    # zero gradients: flat
        grad = torch.from_numpy(grad_np).cuda()
        want = obn.normal_pack(n_np, f_np, want_tan, T, 0, T, grad_np)
        for band in (T, C + 3):                                # C + 3: bands cut through cells
            got = torch.cat([_pack(v_nrm, f, tan, T, r0, min(band, T - r0), grad[r0 * T:(r0 + min(band, T - r0)) * T])
                             for r0 in range(0, T, band)]).cpu().numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    out = torch.empty(Fn, 3, 4, device="cuda")
    with pytest.raises(RuntimeError, match="bad argument"):
        L.call("rsdf_bake_tangents", L.ptr(v_pos), L.ptr(f), L.ptr(v_nrm), Fn, 16, L.ptr(out), L.stream())
    with pytest.raises(RuntimeError, match="bad argument"):
        L.call("rsdf_normal_pack", L.ptr(v_nrm), L.ptr(f), L.ptr(tan), Fn, 256, 250, 7, L.ptr(grad), L.ptr(out),
               L.stream())


def _field_normal(m, pts):
    with torch.no_grad():
        _, g = m.geometry(pts, with_grad=True, with_feature=False)
    return F.normalize(g.double(), dim=-1).cpu().numpy()


def _decode_at_texels(out, T, enc):
    """(owned texel indices, decoded world normals float64 [n, 3], texel points) of an export's atlas texels"""
    f = out["t_pos_idx"]
    face, pts = _texels(out["v_pos"], f, T, 0, T)
    face_np, b = obn.texel_barycentrics(f.shape[0], T, 0, T)
    assert np.array_equal(face.cpu().numpy(), face_np)
    own = np.flatnonzero(face_np >= 0)
    fo = face_np[own]
    f_np = f.cpu().numpy()
    dec = obn.decode(out["v_nrm"].cpu().numpy()[f_np[fo]], out["t_tangent"].cpu().numpy()[fo], b[own], enc[own])
    return own, dec, pts[torch.from_numpy(own).cuda()], b[own], f_np[fo]


def _angle(a, b):
    return np.arccos(np.clip(np.sum(a * b, -1), -1.0, 1.0))


def test_normal_map_decodes_to_the_field_normal(smooth, tmp_path):
    m = smooth
    T = 1024
    out = m.export(chunk_size=1 << 16, resolution=128, texture_size=T, normal_map=True)
    Fn = out["t_pos_idx"].shape[0]
    assert out["t_tangent"].shape == (Fn, 3, 4) and out["normal_atlas"].shape == (T, T, 3)
    w = out["t_tangent"][..., 3]
    assert torch.unique(w).numel() == 1 and float(w[0, 0]) in (-1.0, 1.0)        # one handedness for all faces
    atlas = out["normal_atlas"].view(-1, 3).cpu().numpy()
    own, dec, pts, _, _ = _decode_at_texels(out, T, atlas)
    unowned = np.setdiff1d(np.arange(T * T), own)
    assert np.all(atlas[unowned] == np.array([0, 0, 1], np.float32))
    want = _field_normal(m, pts)
    err = np.abs(dec - want).max()
    print(f"float normal map: max |decoded - field normal| = {err:.2e} over {len(own)} texels")
    assert err <= 1e-5
    # through the .glb: 8-bit channels round(255 (x / 2 + 1/2)) are off by at most 1/255 each in [-1, 1], a vector error
    # of at most sqrt(3) / 255, so the decoded direction is within asin(sqrt(3) / 255) (+ the float map's error)
    path = formats.save_mesh_glb(str(tmp_path / "n.glb"), out)
    gltf, binary = read_glb(path)
    (prim,) = gltf["meshes"][0]["primitives"]
    assert gltf["accessors"][prim["attributes"]["TANGENT"]]["count"] == 3 * Fn
    assert gltf["materials"][0]["normalTexture"] == {"index": 2, "texCoord": 0}
    img = gltf["images"][gltf["textures"][2]["source"]]
    png = cv2.imdecode(np.frombuffer(view_bytes(gltf, binary, img["bufferView"]), np.uint8), cv2.IMREAD_UNCHANGED)
    enc8 = png[..., ::-1].reshape(-1, 3).astype(np.float64) / 255.0 * 2.0 - 1.0
    _, dec8, _, _, _ = _decode_at_texels(out, T, enc8)
    bound = math.asin(math.sqrt(3) / 255) + 1e-5
    ang = _angle(dec8, want)
    print(f"8-bit normal map: max angle {ang.max():.2e} rad, bound {bound:.2e} rad")
    assert ang.max() <= bound


def _bilinear(atlas, uv):
    """bilinear sample (glTF LINEAR) of atlas [T, T, 3] at UVs [n, 2]; float64"""
    T = atlas.shape[0]
    x, y = uv[:, 0] * T - 0.5, uv[:, 1] * T - 0.5
    x0, y0 = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    fx, fy = (x - x0)[:, None], (y - y0)[:, None]
    a = atlas.astype(np.float64)
    return ((1 - fy) * ((1 - fx) * a[y0, x0] + fx * a[y0, x0 + 1]) + fy * ((1 - fx) * a[y0 + 1, x0] + fx * a[y0 + 1, x0 + 1]))


def test_normal_map_beats_vertex_normals(model, smooth):
    """At a coarse resolution the mesh's interpolated vertex normals miss the field's detail; the map holds it."""
    # noisy test model: at the texel points, where the map stores the field normal
    T = 2048
    out = model.export(chunk_size=1 << 18, resolution=48, texture_size=T, normal_map=True)
    atlas = out["normal_atlas"].view(-1, 3).cpu().numpy()
    own, dec, pts, b, corners = _decode_at_texels(out, T, atlas)
    want = _field_normal(model, pts)
    vn = out["v_nrm"].double().cpu().numpy()[corners]
    interp = np.einsum("nk,nkc->nc", b.astype(np.float64), vn)
    interp /= np.linalg.norm(interp, axis=-1, keepdims=True)
    map_err, vert_err = _angle(dec, want).mean(), _angle(interp, want).mean()
    print(f"noisy model, resolution 48, T {T}: mean angle to the field normal at the texel points: normal map "
          f"{map_err:.2e} rad, interpolated vertex normals {vert_err:.2e} rad")
    assert map_err < 0.01 * vert_err
    # smooth model: between the texels too, bilinear map samples as a viewer reads them
    T = 1024
    out = smooth.export(chunk_size=1 << 18, resolution=48, texture_size=T, normal_map=True)
    f = out["t_pos_idx"]
    rng = np.random.default_rng(0)
    bs = rng.dirichlet(np.ones(3), size=f.shape[0]).astype(np.float32)               # one point per face
    f_np = f.cpu().numpy()
    v = out["v_pos"].cpu().numpy()[f_np]
    pts = np.einsum("nk,nkc->nc", bs, v).astype(np.float32)
    uv = np.einsum("nk,nkc->nc", bs.astype(np.float64), out["t_uv"].double().cpu().numpy())
    enc = _bilinear(out["normal_atlas"].cpu().numpy(), uv)
    dec = obn.decode(out["v_nrm"].cpu().numpy()[f_np], out["t_tangent"].cpu().numpy(), bs, enc)
    want = _field_normal(smooth, torch.from_numpy(pts).cuda())
    vn = np.einsum("nk,nkc->nc", bs.astype(np.float64), out["v_nrm"].double().cpu().numpy()[f_np])
    vn /= np.linalg.norm(vn, axis=-1, keepdims=True)
    map_err, vert_err = _angle(dec, want).mean(), _angle(vn, want).mean()
    print(f"smooth model, resolution 48, T {T}: mean angle to the field normal inside the faces: bilinear normal map "
          f"{map_err:.2e} rad, interpolated vertex normals {vert_err:.2e} rad")
    assert map_err < vert_err


def test_export_with_normal_map_keeps_the_other_entries(model):
    m = model
    T = 1024
    plain = m.export(chunk_size=1 << 16, resolution=128, texture_size=T)
    out = m.export(chunk_size=1 << 16, resolution=128, texture_size=T, normal_map=True)
    assert set(out) == set(plain) | {"t_tangent", "normal_atlas"}
    for k, t in plain.items():
        assert torch.equal(out[k], t), k
    atlas = bake.bake_material_atlas(m, out["v_pos"], out["t_pos_idx"], T, 1 << 16)
    assert torch.equal(out["material_atlas"], atlas)
    # the shared band loop at other band sizes, and the normal atlas on its own
    for chunk in (T * 7 + 5, 1 << 20):
        mat, nrm = bake.bake_atlases(m, out["v_pos"], out["t_pos_idx"], out["v_nrm"], out["t_tangent"], T, chunk)
        assert torch.equal(mat, atlas) and torch.equal(nrm, out["normal_atlas"])
    assert torch.equal(bake.bake_normal_atlas(m, out["v_pos"], out["t_pos_idx"], out["v_nrm"], out["t_tangent"], T,
                                              1 << 16), out["normal_atlas"])
    again = m.export(chunk_size=1 << 16, resolution=128, texture_size=T, normal_map=True)
    for k, t in out.items():
        assert torch.equal(t, again[k]), k
    empty = m.export(resolution=32, threshold=1e4, texture_size=16, normal_map=True)
    assert empty["v_pos"].shape[0] == 0 and empty["t_tangent"].shape == (0, 3, 4)
    assert torch.equal(empty["normal_atlas"], torch.tensor([0.0, 0.0, 1.0], device="cuda").expand(16, 16, 3))
    with pytest.raises(ValueError, match="texels per side"):
        m.export(resolution=64, texture_size=16, normal_map=True)


def test_normal_band_memory_and_read_backs(model):
    m = model
    mesh = m.geometry.isosurface(128)
    v, f = mesh["v_pos"], mesh["t_pos_idx"]
    with torch.no_grad():
        _, g = m.geometry(v, with_grad=True, with_feature=False)
    v_nrm = F.normalize(g, dim=-1)
    band = 1 << 18
    T = 2048
    tan = bake.atlas_tangents(v, f, v_nrm, T)

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        atlases = fn()
        torch.cuda.synchronize()
        extra = torch.cuda.max_memory_allocated() - base - sum(a.numel() * 4 for a in atlases)
        del atlases
        return extra

    both = lambda chunk: bake.bake_atlases(m, v, f, v_nrm, tan, T, chunk)
    both(band)                                                           # warm-up: weight caches
    shared = peak(lambda: both(band))
    materials = peak(lambda: (bake.bake_material_atlas(m, v, f, T, band),))
    normals = peak(lambda: (bake.bake_normal_atlas(m, v, f, v_nrm, tan, T, band),))
    print(f"peak beyond the atlases, per band texel: materials {materials / band:.0f} B, normals {normals / band:.0f} B, "
          f"both in one pass {shared / band:.0f} B")
    assert shared <= 8192 * band and normals <= 8192 * band

    def d2h(T):
        t = bake.atlas_tangents(v, f, v_nrm, T)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            bake.bake_atlases(m, v, f, v_nrm, t, T, band)
            torch.cuda.synchronize()
        return sum(e.count for e in prof.key_averages() if "DtoH" in e.key or "Device -> Pageable" in e.key)

    def n_bands(T):
        C, cols = bake.atlas_layout(f.shape[0], T)
        rows = -(-((f.shape[0] + 1) // 2) // cols) * C
        return -(-rows // max(1, band // T))

    assert n_bands(4096) > n_bands(1024)
    assert d2h(1024) == d2h(4096)
