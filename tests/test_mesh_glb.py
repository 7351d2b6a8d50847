"""glTF binary writer (`formats.save_mesh_glb`) read back with a small independent parser, and the PNG encoder it shares
with `save_png`.  CPU only."""
import json
import struct
import zlib

import cv2
import numpy as np
import pytest
import torch

from rise_sdf_b200 import formats

COMP = {5126: ("<f4", 4), 5125: ("<u4", 4)}
NCOMP = {"SCALAR": 1, "VEC2": 2, "VEC3": 3}


def read_glb(path):
    """(json dict, bin bytes or None) after checking the container: header, chunk types, lengths and alignment."""
    buf = open(path, "rb").read()
    magic, version, length = struct.unpack_from("<III", buf, 0)
    assert magic == 0x46546C67 and version == 2 and length == len(buf) and length % 4 == 0
    jlen, jtype = struct.unpack_from("<II", buf, 12)
    assert jtype == 0x4E4F534A and jlen % 4 == 0
    js = buf[20:20 + jlen]
    assert js.rstrip(b" ") == js.rstrip() and js.decode("utf-8")
    gltf = json.loads(js)
    pos = 20 + jlen
    binary = None
    if pos < length:
        blen, btype = struct.unpack_from("<II", buf, pos)
        assert btype == 0x004E4942 and blen % 4 == 0 and pos + 8 + blen == length
        binary = buf[pos + 8:pos + 8 + blen]
        assert gltf["buffers"] == [{"byteLength": blen}]
    assert gltf["asset"]["version"] == "2.0"
    return gltf, binary


def view_bytes(gltf, binary, i):
    v = gltf["bufferViews"][i]
    assert v["buffer"] == 0 and v["byteOffset"] % 4 == 0 and v["byteOffset"] + v["byteLength"] <= len(binary)
    return binary[v["byteOffset"]:v["byteOffset"] + v["byteLength"]]


def accessor(gltf, binary, i, kind, comp):
    a = gltf["accessors"][i]
    assert a["type"] == kind and a["componentType"] == comp and a.get("byteOffset", 0) == 0
    dt, size = COMP[comp]
    data = view_bytes(gltf, binary, a["bufferView"])
    assert len(data) == a["count"] * NCOMP[kind] * size
    return np.frombuffer(data, dtype=dt).reshape(a["count"], NCOMP[kind]) if kind != "SCALAR" \
        else np.frombuffer(data, dtype=dt)


def _mesh(rng, V=40, F=61):
    v = rng.standard_normal((V, 3)).astype(np.float32)
    f = rng.integers(0, V, (F, 3))
    n = rng.standard_normal((V, 3)).astype(np.float32)
    return v, f, n / np.linalg.norm(n, axis=1, keepdims=True)


def _srgb(x):
    from rise_sdf_b200.light import rgb_to_srgb
    return rgb_to_srgb(torch.from_numpy(x)).numpy()


def test_textured_glb_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    v, f, n = _mesh(rng)
    T = 48
    uv = rng.random((len(f), 3, 2)).astype(np.float32)
    atlas = rng.random((T, T, 5)).astype(np.float32)
    atlas[:5] = 0.0
    atlas[5, :, 0] = np.linspace(-0.1, 1.1, T)                  # out-of-range values clamp
    mesh = {"v_pos": torch.from_numpy(v), "t_pos_idx": torch.from_numpy(f), "v_nrm": torch.from_numpy(n),
            "t_uv": torch.from_numpy(uv), "material_atlas": torch.from_numpy(atlas),
            "v_albedo": torch.zeros(len(v), 3)}
    path = formats.save_mesh_glb(str(tmp_path / "m.glb"), mesh)
    gltf, binary = read_glb(path)
    (prim,) = gltf["meshes"][0]["primitives"]
    assert gltf["scenes"][gltf["scene"]]["nodes"] == [0] and gltf["nodes"][0]["mesh"] == 0
    assert prim["mode"] == 4 and set(prim["attributes"]) == {"POSITION", "NORMAL", "TEXCOORD_0"}
    corners = f.reshape(-1)
    pos = accessor(gltf, binary, prim["attributes"]["POSITION"], "VEC3", 5126)
    nrm = accessor(gltf, binary, prim["attributes"]["NORMAL"], "VEC3", 5126)
    tc = accessor(gltf, binary, prim["attributes"]["TEXCOORD_0"], "VEC2", 5126)
    idx = accessor(gltf, binary, prim["indices"], "SCALAR", 5125)
    assert len(pos) == len(nrm) == len(tc) == 3 * len(f)
    assert np.array_equal(pos, v[corners]) and np.array_equal(nrm, n[corners])     # unwelded through t_pos_idx
    assert np.array_equal(tc, uv.reshape(-1, 2))
    assert np.array_equal(idx, np.arange(3 * len(f)))
    a = gltf["accessors"][prim["attributes"]["POSITION"]]
    assert np.array_equal(np.float32(a["min"]), v[corners].min(0)) and np.array_equal(np.float32(a["max"]),
                                                                                      v[corners].max(0))
    # material: two embedded PNG textures, linear / clamped sampler, unit factors
    (mat,) = gltf["materials"]
    pbr = mat["pbrMetallicRoughness"]
    assert pbr["metallicFactor"] == 1.0 and pbr["roughnessFactor"] == 1.0
    assert pbr.get("baseColorFactor", [1, 1, 1, 1]) == [1, 1, 1, 1] and prim["material"] == 0
    (smp,) = gltf["samplers"]
    assert smp == {"magFilter": 9729, "minFilter": 9729, "wrapS": 33071, "wrapT": 33071}

    def image(tex):
        t = gltf["textures"][tex["index"]]
        assert t["sampler"] == 0 and tex.get("texCoord", 0) == 0
        img = gltf["images"][t["source"]]
        assert img["mimeType"] == "image/png"
        data = np.frombuffer(view_bytes(gltf, binary, img["bufferView"]), np.uint8)
        return cv2.imdecode(data, cv2.IMREAD_UNCHANGED)[..., ::-1]          # BGR -> RGB

    base, mr = image(pbr["baseColorTexture"]), image(pbr["metallicRoughnessTexture"])
    q = lambda x: np.round(np.clip(x, 0, 1) * np.float32(255)).astype(np.uint8)
    want_base = q(_srgb(atlas[..., :3]))
    assert base.shape == (T, T, 3) and np.array_equal(base, want_base)
    assert mr.shape == (T, T, 3) and (mr[..., 0] == 0).all()
    assert np.array_equal(mr[..., 1], q(atlas[..., 3])) and np.array_equal(mr[..., 2], q(atlas[..., 4]))
    assert (base[:5] == 0).all() and (mr[:5] == 0).all()


def test_plain_glb_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    v, f, n = _mesh(rng, 33, 50)
    rgb = rng.random((33, 3)).astype(np.float32)
    for extra in ({}, {"v_rgb": torch.from_numpy(rgb)}, {"v_nrm": torch.from_numpy(n), "v_rgb": torch.from_numpy(rgb)}):
        path = formats.save_mesh_glb(str(tmp_path / "p.glb"), {"v_pos": torch.from_numpy(v),
                                                               "t_pos_idx": torch.from_numpy(f), **extra})
        gltf, binary = read_glb(path)
        (prim,) = gltf["meshes"][0]["primitives"]
        want = {"POSITION"} | ({"COLOR_0"} if "v_rgb" in extra else set()) | ({"NORMAL"} if "v_nrm" in extra else set())
        assert set(prim["attributes"]) == want and "material" not in prim and "images" not in gltf
        assert np.array_equal(accessor(gltf, binary, prim["attributes"]["POSITION"], "VEC3", 5126), v)
        assert np.array_equal(accessor(gltf, binary, prim["indices"], "SCALAR", 5125), f.reshape(-1))
        a = gltf["accessors"][prim["attributes"]["POSITION"]]
        assert np.array_equal(np.float32(a["min"]), v.min(0)) and np.array_equal(np.float32(a["max"]), v.max(0))
        if "v_rgb" in extra:
            assert np.array_equal(accessor(gltf, binary, prim["attributes"]["COLOR_0"], "VEC3", 5126), rgb)
        if "v_nrm" in extra:
            assert np.array_equal(accessor(gltf, binary, prim["attributes"]["NORMAL"], "VEC3", 5126), n)


def test_empty_mesh_glb(tmp_path):
    for extra in ({}, {"t_uv": torch.zeros(0, 3, 2), "material_atlas": torch.zeros(16, 16, 5),
                       "v_nrm": torch.zeros(0, 3)}):
        path = formats.save_mesh_glb(str(tmp_path / "e.glb"), {"v_pos": torch.zeros(0, 3),
                                                               "t_pos_idx": torch.zeros(0, 3, dtype=torch.int64),
                                                               **extra})
        gltf, binary = read_glb(path)
        assert binary is None and gltf["scenes"][gltf["scene"]] == {"nodes": []}
        assert "meshes" not in gltf and "buffers" not in gltf


def test_glb_size_guard(tmp_path, monkeypatch):
    rng = np.random.default_rng(2)
    v, f, _ = _mesh(rng, 10, 12)
    mesh = {"v_pos": torch.from_numpy(v), "t_pos_idx": torch.from_numpy(f)}
    gltf_len = len(open(formats.save_mesh_glb(str(tmp_path / "ok.glb"), mesh), "rb").read())
    monkeypatch.setattr(formats, "GLB_MAX_BYTES", gltf_len - 1)
    with pytest.raises(ValueError, match="glTF binary holds at most"):
        formats.save_mesh_glb(str(tmp_path / "big.glb"), mesh)
    monkeypatch.setattr(formats, "GLB_MAX_BYTES", 200)                  # the attribute data alone is too large
    with pytest.raises(ValueError, match="bytes; a .glb holds at most"):
        formats.save_mesh_glb(str(tmp_path / "big.glb"), mesh)
    monkeypatch.setattr(formats, "GLB_MAX_BYTES", gltf_len)
    formats.save_mesh_glb(str(tmp_path / "ok.glb"), mesh)


def _save_png_before_png_bytes(path, img):
    """`formats.save_png` as it was before its encoder became `formats.png_bytes`."""
    a = img.detach().cpu().numpy() if hasattr(img, "detach") else np.asarray(img)
    if a.ndim == 2:
        a = a[..., None]
    a = (np.clip(a, 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8)
    h, w, c = a.shape
    assert c in (1, 3)
    raw = b"".join(b"\x00" + a[y].tobytes() for y in range(h))

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)
    png = (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2 if c == 3 else 0, 0, 0, 0))
           + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))
    with open(path, "wb") as f:
        f.write(png)


def test_save_png_bytes_unchanged(tmp_path):
    rng = np.random.default_rng(7)
    imgs = [rng.random((13, 17, 3)).astype(np.float32) * 1.2 - 0.1, rng.random((9, 5)).astype(np.float32),
            torch.from_numpy(rng.random((4, 6, 1)).astype(np.float32)),
            np.linspace(0, 1, 64 * 3, dtype=np.float64).reshape(8, 8, 3)]
    for k, img in enumerate(imgs):
        formats.save_png(str(tmp_path / f"new{k}.png"), img)
        _save_png_before_png_bytes(str(tmp_path / f"old{k}.png"), img)
        new = open(tmp_path / f"new{k}.png", "rb").read()
        assert new == open(tmp_path / f"old{k}.png", "rb").read()
        dec = cv2.imdecode(np.frombuffer(new, np.uint8), cv2.IMREAD_UNCHANGED)
        assert dec is not None and dec.shape[:2] == np.asarray(img).shape[:2]
