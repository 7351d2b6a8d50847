"""The normal map in `formats.save_mesh_glb`: TANGENT accessor, third embedded PNG and the material's `normalTexture`,
read back with the parser of test_mesh_glb.py; files without the normal-map keys keep their exact bytes.  CPU only."""
import hashlib

import cv2
import numpy as np
import pytest
import torch

from rise_sdf_b200 import formats
from test_mesh_glb import accessor, read_glb, view_bytes


def _textured(seed, V=40, F=61, T=48):
    rng = np.random.default_rng(seed)
    v = rng.standard_normal((V, 3)).astype(np.float32)
    f = rng.integers(0, V, (F, 3))
    n = rng.standard_normal((V, 3)).astype(np.float32)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    uv = rng.random((F, 3, 2)).astype(np.float32)
    atlas = rng.random((T, T, 5)).astype(np.float32)
    return {"v_pos": torch.from_numpy(v), "t_pos_idx": torch.from_numpy(f), "v_nrm": torch.from_numpy(n),
            "t_uv": torch.from_numpy(uv), "material_atlas": torch.from_numpy(atlas)}


def test_normal_map_glb_round_trip(tmp_path):
    mesh = _textured(0)
    F, T = mesh["t_pos_idx"].shape[0], mesh["material_atlas"].shape[0]
    rng = np.random.default_rng(1)
    tangent = rng.standard_normal((F, 3, 4)).astype(np.float32)
    tangent[..., 3] = np.where(rng.random((F, 1)) < 0.5, -1.0, 1.0)
    normals = rng.standard_normal((T, T, 3)).astype(np.float32)
    normals /= np.linalg.norm(normals, axis=-1, keepdims=True)
    normals[0, :3] = [[1.5, -1.5, 0.0], [-1.0, 1.0, 1.0], [0.0, 0.0, 1.0]]       # out of range clamps; exact ends
    path = formats.save_mesh_glb(str(tmp_path / "n.glb"), {**mesh, "t_tangent": torch.from_numpy(tangent),
                                                          "normal_atlas": torch.from_numpy(normals)})
    gltf, binary = read_glb(path)
    (prim,) = gltf["meshes"][0]["primitives"]
    assert set(prim["attributes"]) == {"POSITION", "NORMAL", "TEXCOORD_0", "TANGENT"}
    a = gltf["accessors"][prim["attributes"]["TANGENT"]]
    assert a["type"] == "VEC4" and a["componentType"] == 5126 and a["count"] == 3 * F
    data = np.frombuffer(view_bytes(gltf, binary, a["bufferView"]), "<f4").reshape(3 * F, 4)
    assert np.array_equal(data, tangent.reshape(-1, 4))
    pos = accessor(gltf, binary, prim["attributes"]["POSITION"], "VEC3", 5126)
    assert len(pos) == 3 * F
    (mat,) = gltf["materials"]
    assert mat["normalTexture"] == {"index": 2, "texCoord": 0}
    assert len(gltf["images"]) == 3 and gltf["textures"][2] == {"sampler": 0, "source": 2}
    img = gltf["images"][2]
    assert img["mimeType"] == "image/png"
    png = cv2.imdecode(np.frombuffer(view_bytes(gltf, binary, img["bufferView"]), np.uint8), cv2.IMREAD_UNCHANGED)
    png = png[..., ::-1]                                                            # BGR -> RGB
    want = np.round(np.clip(normals * np.float32(0.5) + np.float32(0.5), 0, 1) * np.float32(255)).astype(np.uint8)
    assert png.shape == (T, T, 3) and np.array_equal(png, want)
    assert list(png[0, 0]) == [255, 0, 128] and list(png[0, 1]) == [0, 255, 255] and list(png[0, 2]) == [128, 128, 255]
    # the other two textures are those of the file without the normal map
    plain, plain_bin = read_glb(formats.save_mesh_glb(str(tmp_path / "p.glb"), mesh))
    for i in (0, 1):
        assert view_bytes(gltf, binary, gltf["images"][i]["bufferView"]) == \
            view_bytes(plain, plain_bin, plain["images"][i]["bufferView"])


# sha256 of the files the writer produced before the normal map existed, for the meshes below, with `png_bytes` replaced
# by the raw pixels (the PNG encoder is shared and unchanged; this keeps the digests independent of the zlib build)
_BEFORE = {"textured": "71e825da72c486f5fdd2e2e389dfeaa4804a856785b083c70db54d37f0d9ab1f",
           "plain": "4912dc184bd6c83f77dbca94874e54efc000bc74a8a7c9886eb3d82a2fc4456e"}


def test_files_without_normal_map_are_unchanged(tmp_path, monkeypatch):
    monkeypatch.setattr(formats, "png_bytes", lambda a: np.ascontiguousarray(a, np.uint8).tobytes())
    digest = lambda m: hashlib.sha256(open(formats.save_mesh_glb(str(tmp_path / "u.glb"), m), "rb").read()).hexdigest()
    textured = _textured(3)
    plain = {k: _textured(4)[k] for k in ("v_pos", "t_pos_idx", "v_nrm")}
    assert digest(textured) == _BEFORE["textured"]
    assert digest(plain) == _BEFORE["plain"]
    F, T = textured["t_pos_idx"].shape[0], textured["material_atlas"].shape[0]
    # one of the two keys alone, or either key on a plain mesh, changes nothing
    assert digest({**textured, "t_tangent": torch.zeros(F, 3, 4)}) == _BEFORE["textured"]
    assert digest({**textured, "normal_atlas": torch.zeros(T, T, 3)}) == _BEFORE["textured"]
    assert digest({**plain, "t_tangent": torch.zeros(F, 3, 4), "normal_atlas": torch.zeros(T, T, 3)}) == \
        _BEFORE["plain"]


def test_normal_map_size_guard(tmp_path, monkeypatch):
    mesh = _textured(5, V=10, F=12, T=16)
    F = mesh["t_pos_idx"].shape[0]
    full = {**mesh, "t_tangent": torch.zeros(F, 3, 4), "normal_atlas": torch.zeros(16, 16, 3)}
    need = 12 + 8 + 8 + 4 * (3 + 3 + 2 + 4) * 3 * F + 4 * 3 * F          # attributes incl. TANGENT, indices
    monkeypatch.setattr(formats, "GLB_MAX_BYTES", need - 1)
    with pytest.raises(ValueError, match=f"at least {need} bytes"):
        formats.save_mesh_glb(str(tmp_path / "big.glb"), full)
