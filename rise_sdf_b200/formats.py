"""On-disk formats either side of the hot path (SURVEY.md §8f row f4), so that RISE-SDF's own checkpoints,
BSDF table and HDR environment maps run through the B200 path unchanged.

* Lightning `.ckpt`: `torch.load(path)['state_dict']` with keys `model.<module path>` (`launch.py:100-119`,
  `systems/base.py` wraps the model as `self.model`).  Our host mirrors use the reference's module paths
  (`geometry.encoding.encoding.params`, `geometry.network.layers.N.weight_{g,v}`, `emitter.base`,
  `occupancy_grid.{resolution,aabbs,occs,binaries}`, `variance.variance`), so loading is a prefix strip +
  dtype normalisation; tiny-cuda-nn stores `params` flat in level-major order, which is also our table order.
* `load/bsdf/bsdf_256_256.bin`: raw little-endian fp32 `[1,256,256,2]` (`models/texture.py:285`).
* `.hdr` (Radiance RGBE, the format of the published env maps; `lib/pbr/utils/nvdiffrecmc_util.py:380-406`):
  a self-contained numpy reader / writer (flat and new-style RLE scanlines); `.exr` goes through cv2 when the
  image ships it, like the reference's pyexr path.

Pure host code (numpy + torch serialization): nothing here touches the device.
"""
import os
import struct

import numpy as np
import torch

MODEL_PREFIX = "model."
LIGHTNING_VERSION = "1.9.5"          # requirements.txt pins pytorch-lightning<2


# --------------------------------------------------------------------------------------------- checkpoints
def to_reference_state_dict(model):
    """state_dict of the Lightning system that owns `model` (`systems/base.py`: `self.model = models.make(..)`)."""
    return {MODEL_PREFIX + k: v.detach().clone() for k, v in model.state_dict().items()}


def load_reference_state_dict(model, state_dict, strict=False):
    """`system.load_state_dict(torch.load(ckpt)['state_dict'], strict=False)` (`launch.py:109,119`) for a bare
    model: accepts keys with or without the `model.` prefix, casts fp16 tiny-cuda-nn parameters to the fp32
    master copy and 0/1 occupancy bytes to bool.  Returns (missing_keys, unexpected_keys); with strict=True any
    mismatch raises like `nn.Module.load_state_dict`."""
    own = model.state_dict()
    picked, unexpected = {}, []
    for k, v in state_dict.items():
        name = k[len(MODEL_PREFIX):] if k.startswith(MODEL_PREFIX) else k
        if name not in own:
            unexpected.append(k)
            continue
        tgt = own[name]
        v = torch.as_tensor(v)
        if tgt.numel() == v.numel() and tgt.shape != v.shape:
            v = v.reshape(tgt.shape)          # e.g. occs [n_cells] vs [levels*n_cells], tcnn params [n] vs [n,1]
        if tgt.shape != v.shape:
            raise RuntimeError(f"size mismatch for {name}: checkpoint {tuple(v.shape)} vs model {tuple(tgt.shape)}")
        picked[name] = v.to(dtype=tgt.dtype)
    missing = [k for k in own if k not in picked]
    if strict and (missing or unexpected):
        raise RuntimeError(f"load_reference_state_dict: missing {missing}, unexpected {unexpected}")
    model.load_state_dict(picked, strict=False)       # runs the modules' own load hooks (occupancy box, bit cache)
    return missing, unexpected


def save_checkpoint(path, model, optimizer=None, scheduler=None, epoch=0, global_step=0):
    """Writes the subset of a pytorch-lightning 1.x checkpoint the reference reads back (`launch.py:100-119`):
    `state_dict` (+ `optimizer_states`, `lr_schedulers`, `epoch`, `global_step`)."""
    ckpt = {"epoch": int(epoch), "global_step": int(global_step), "pytorch-lightning_version": LIGHTNING_VERSION,
            "state_dict": to_reference_state_dict(model)}
    if optimizer is not None:
        ckpt["optimizer_states"] = [optimizer.state_dict()]
    if scheduler is not None:
        ckpt["lr_schedulers"] = [scheduler.state_dict()]
    tmp = path + ".tmp"
    torch.save(ckpt, tmp)
    os.replace(tmp, path)               # a crash mid-write never leaves a truncated checkpoint behind
    return path


def load_checkpoint(path, model, optimizer=None, scheduler=None, weights_only=False, strict=False):
    """`--resume` (`launch.py:100-102`): weights, then -- unless `weights_only` (`--resume_weights_only`) -- the
    optimizer / scheduler state.  Returns the checkpoint dict's bookkeeping (`epoch`, `global_step`, key report)."""
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    missing, unexpected = load_reference_state_dict(model, ckpt["state_dict"], strict=strict)
    if not weights_only:
        if optimizer is not None and ckpt.get("optimizer_states"):
            optimizer.load_state_dict(ckpt["optimizer_states"][0])
        if scheduler is not None and ckpt.get("lr_schedulers"):
            scheduler.load_state_dict(ckpt["lr_schedulers"][0])
    return {"epoch": ckpt.get("epoch", 0), "global_step": ckpt.get("global_step", 0), "missing": missing,
            "unexpected": unexpected}


# --------------------------------------------------------------------------------------------- BSDF table
def load_bsdf_lut(path="load/bsdf/bsdf_256_256.bin", res=256):
    """`np.fromfile(path, float32).reshape(1, 256, 256, 2)` (`models/texture.py:285`) -> torch tensor."""
    raw = np.fromfile(path, dtype="<f4")
    if raw.size != res * res * 2:
        raise ValueError(f"{path}: expected {res * res * 2} float32 values, found {raw.size}")
    return torch.from_numpy(raw.reshape(1, res, res, 2).astype(np.float32))


def save_bsdf_lut(path, lut):
    arr = (lut.detach().cpu().numpy() if isinstance(lut, torch.Tensor) else np.asarray(lut)).astype("<f4")
    arr.reshape(-1).tofile(path)
    return path


# --------------------------------------------------------------------------------------------- Radiance .hdr
def _rgbe_to_float(rgbe):
    """[..., 4] uint8 -> [..., 3] float32: value = mantissa * 2^(e-136), e == 0 is black -- OpenCV's `rgbe2float`
    (no +0.5 on the mantissa), because cv2 is the decoder the reference runs its env maps through."""
    e = rgbe[..., 3].astype(np.int32)
    scale = np.ldexp(np.float32(1.0), e - (128 + 8)).astype(np.float32)
    out = rgbe[..., :3].astype(np.float32) * scale[..., None]
    out[e == 0] = 0.0
    return out


def _float_to_rgbe(rgb):
    rgb = np.maximum(np.asarray(rgb, dtype=np.float32), 0.0)
    m = rgb.max(axis=-1)
    mant, exp = np.frexp(m)                    # m = mant * 2^exp, mant in [0.5, 1)
    scale = np.where(m > 1e-32, mant * 256.0 / np.maximum(m, 1e-38), 0.0).astype(np.float32)
    out = np.zeros(rgb.shape[:-1] + (4,), dtype=np.uint8)
    out[..., :3] = np.clip(np.floor(rgb * scale[..., None]), 0, 255).astype(np.uint8)
    out[..., 3] = np.where(m > 1e-32, exp + 128, 0).astype(np.uint8)
    return out


def _read_scanline_rle(buf, pos, width):
    """One new-style RLE scanline (4 planes of `width` bytes); returns ([width,4] uint8, new position)."""
    line = np.empty((4, width), dtype=np.uint8)
    for c in range(4):
        x = 0
        while x < width:
            n = buf[pos]
            pos += 1
            if n > 128:                          # run
                n -= 128
                line[c, x:x + n] = buf[pos]
                pos += 1
            else:                                # literal
                line[c, x:x + n] = np.frombuffer(buf, dtype=np.uint8, count=n, offset=pos)
                pos += n
            if n == 0:
                raise ValueError("corrupt RLE scanline")
            x += n
        if x != width:
            raise ValueError("RLE scanline overruns the image width")
    return line.T, pos


def read_hdr(path):
    """Radiance RGBE picture -> float32 [H, W, 3], RGB order, top row first (what the reference gets from
    `cv2.imdecode(..., IMREAD_UNCHANGED)` + BGR->RGB, `nvdiffrecmc_util.py:380-392`)."""
    with open(path, "rb") as f:
        buf = f.read()
    if not (buf.startswith(b"#?RADIANCE") or buf.startswith(b"#?RGBE")):
        raise ValueError(f"{path}: not a Radiance HDR file")
    pos, fmt_ok = 0, False
    while True:                                   # header lines up to the empty line
        end = buf.index(b"\n", pos)
        line = buf[pos:end]
        pos = end + 1
        if line.startswith(b"FORMAT="):
            fmt_ok = line.strip() == b"FORMAT=32-bit_rle_rgbe"
        if line.strip() == b"":
            break
    if not fmt_ok:
        raise ValueError(f"{path}: only FORMAT=32-bit_rle_rgbe is supported")
    end = buf.index(b"\n", pos)
    res = buf[pos:end].split()
    pos = end + 1
    if len(res) != 4 or res[0] != b"-Y" or res[2] != b"+X":
        raise ValueError(f"{path}: unsupported orientation {buf[pos:end]!r} (expected '-Y H +X W')")
    h, w = int(res[1]), int(res[3])
    rgbe = np.empty((h, w, 4), dtype=np.uint8)
    for y in range(h):
        if 8 <= w < 32768 and buf[pos] == 2 and buf[pos + 1] == 2 and ((buf[pos + 2] << 8) | buf[pos + 3]) == w:
            rgbe[y], pos = _read_scanline_rle(buf, pos + 4, w)
        else:                                     # flat (or old-style) scanline: 4 bytes per pixel
            rgbe[y] = np.frombuffer(buf, dtype=np.uint8, count=4 * w, offset=pos).reshape(w, 4)
            pos += 4 * w
    return _rgbe_to_float(rgbe)


def _rle_plane(row):
    """Radiance run-length code of one byte plane (runs of >= 4 equal bytes, literals of <= 128)."""
    out, n, i = bytearray(), len(row), 0
    while i < n:
        run = 1
        while i + run < n and run < 127 and row[i + run] == row[i]:
            run += 1
        if run >= 4:
            out += bytes((128 + run, row[i]))
            i += run
            continue
        j = i
        while j < n and j - i < 128:
            r = 1
            while j + r < n and r < 4 and row[j + r] == row[j]:
                r += 1
            if r >= 4:
                break
            j += 1
        out += bytes((j - i,)) + bytes(row[i:j])
        i = j
    return out


def write_hdr(path, img, rle=True):
    """float [H, W, 3] RGB -> Radiance RGBE file (readable by cv2 / the reference's `read_hdr`)."""
    img = np.asarray(img, dtype=np.float32)
    h, w, _ = img.shape
    rgbe = _float_to_rgbe(img)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n" + f"-Y {h} +X {w}\n".encode())
        for y in range(h):
            if rle and 8 <= w < 32768:
                f.write(struct.pack(">BBH", 2, 2, w))
                for c in range(4):
                    f.write(_rle_plane(rgbe[y, :, c].tolist()))
            else:
                f.write(rgbe[y].tobytes())
    return path


def load_image(fn):
    """`nvdiffrecmc_util.load_image` (`:394-406`): `.hdr` / `.exr` -> float32 [H, W, 3]; 8-bit data / 255."""
    if fn.endswith("hdr"):
        img = read_hdr(fn)
    elif fn.endswith("exr"):
        os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
        import cv2
        bgr = cv2.imread(fn, cv2.IMREAD_UNCHANGED)
        if bgr is None:
            raise IOError(f"cannot read {fn} (OpenEXR support missing from this cv2 build?)")
        img = np.ascontiguousarray(bgr[..., 2::-1])
    else:
        raise NotImplementedError("wrong image type")
    return img if img.dtype == np.float32 else img.astype(np.float32) / 255


def load_env_latlong(fn, device="cuda"):
    """Lat-long environment map as the tensor `EnvironmentLightMipCube.relight` / `EnvSet` take
    (`lib/pbr/light.py:155-158`)."""
    return torch.tensor(load_image(fn).copy(), dtype=torch.float32, device=device)


# ---------------------------------------------------------------------------------------- image writers
def save_png(path, img):
    """utils/mixins.py `save_image_grid` / `save_rgb_image` write 8-bit PNGs through cv2; this is a dependency-free
    writer (zlib from the standard library) for rendered frames: img [H, W, 3|1] float in [0, 1] (torch or numpy)."""
    import struct
    import zlib
    import numpy as np
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


def save_exr_or_hdr(path, img):
    """Float frames (utils/mixins.py writes .exr through pyexr): `.hdr` through this module's own Radiance codec, `.exr`
    through OpenCV when its EXR codec is enabled."""
    a = img.detach().cpu().numpy() if hasattr(img, "detach") else img
    if path.lower().endswith(".hdr"):
        return write_hdr(path, a)
    import os
    os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
    import cv2
    if not cv2.imwrite(path, a[..., ::-1].astype("float32")):
        raise RuntimeError(f"OpenCV could not write {path}")


def save_mesh_obj(path, v_pos, t_pos_idx, v_rgb=None):
    """Wavefront OBJ of a triangle mesh (`VolumeSDF.isosurface` / `NeuSModel.export`): one `v x y z` line per vertex,
    `v x y z r g b` with vertex colours in [0, 1], then one 1-based `f a b c` line per face -- the plain layout mesh
    viewers and trimesh read."""
    host = lambda t: t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
    v = host(v_pos).astype(np.float64).reshape(-1, 3)
    f = host(t_pos_idx).astype(np.int64).reshape(-1, 3) + 1
    if v_rgb is not None:
        v = np.concatenate([v, host(v_rgb).astype(np.float64).reshape(-1, 3)], 1)
    vfmt = "v" + " %.9g" * v.shape[1]                 # 9 significant digits: float32 round-trips exactly
    with open(path, "w") as fh:
        if len(v):
            np.savetxt(fh, v, fmt=vfmt)
        if len(f):
            np.savetxt(fh, f, fmt="f %d %d %d")
    return path


def save_level_grid(path, level):
    """The isosurface level grid (VolumeSDF.isosurface_level) as a raw .npy volume for an external marching-cubes tool."""
    import numpy as np
    np.save(path, level.detach().cpu().numpy() if hasattr(level, "detach") else level)
