"""Relighting render (BASELINE configs[3]; systems/split_occ.py:331-458): 800x800 frames of a
split-sum model under new environment maps, pixels sharded across GPUs with NO communication
(SURVEY.md §8e): the pixels are interleaved over the ranks (rank r takes pixels r, r + world, ...; the
object is centred, so row blocks -- and even round-robin row bands -- would be imbalanced) and each shard
is rendered in `tile`-ray tiles; every rank holds the full model, occupancy grid, prefiltered mip
pyramids and LUT and keeps its result sharded (`frame[rank::world] = shard` assembles it)."""
import torch

from . import metrics
from . import synthetic as syn
from .light import blender_latlong_to_cubemap


class EnvSet:
    """Prefiltered pyramids for a list of lat-long HDR maps (built once per map: `base` is frozen
    when relighting, unlike training where build_mips runs every step)."""

    def __init__(self, model, latlongs):
        self.model = model
        self.maps = []
        em = model.emitter
        with torch.no_grad():
            for img in latlongs:
                em.base.data = blender_latlong_to_cubemap(img.to(em.base.device).float(), [512, 512])
                em.build_mips()
                self.maps.append(([t.detach().clone() for t in em.specular], em.diffuse.detach().clone()))

    def use(self, i):
        self.model.emitter.specular, self.model.emitter.diffuse = self.maps[i]


def my_tiles(n_rays, tile, rank, world):
    """contiguous tiles dealt round-robin (kept for callers that want row blocks; see `my_pixels`)"""
    return [(s, min(s + tile, n_rays)) for k, s in enumerate(range(0, n_rays, tile)) if k % world == rank]


def my_pixels(n_rays, rank, world):
    """Pixel-interleaved shard of a frame: rank r renders rays r, r + world, r + 2 world, ...  Every rank (and every
    tile inside a rank's shard) sees the whole image subsampled, so the work per rank is balanced whatever the
    object covers -- row blocks or round-robin row bands put the dense centre on a few ranks.  Returns the slice."""
    return slice(rank, n_rays, world)


# rays per forward_ call.  Every tile pays a fixed ~4 ms of host read-backs and launch latency (16 syncs, ~400 launches),
# so fewer, larger tiles are faster: 32768 -> 4.45, 65536 -> 5.0, 131072 -> 5.2-5.3 frames/s at 1 GPU, and the 80 000-ray
# shard of an 8-GPU run is one tile.  (Geometry is bit-identical across tile sizes; the largest evaluation batch at the
# config's initial variance, 28 M samples = 5.4 G feature elements, is beyond int32 element counts: offsets are 64-bit.)
# Tiles are multiples of the reference's 4096-ray chunk: its relighting recombination is decided per chunk
# (split_mixed_occ.py, "recombined"), and a tile boundary inside a chunk would change that decision.
MAX_TILE = 131072
REF_CHUNK = 4096


def balanced_tile(n_rays, world, max_tile=None, per_rank=1):
    """Tile size for a rank's shard of ceil(n_rays / world) rays: the fewest tiles of at most max_tile rays (every
    tile pays ~16 host read-backs; interleaved pixels already balance the ranks), all (almost) equal, whole reference
    chunks of 4096 rays: 640 000 rays -> 5 tiles of 131 072 on 1 GPU, one 81 920-ray tile for the 80 000-ray shard of 8
    GPUs."""
    max_tile = max_tile or MAX_TILE
    n = -(-n_rays // world)
    t = min(max_tile, -(-n // per_rank))
    t = -(-t // 64) * 64
    k = -(-n // t)
    t = -(-(-(-n // k)) // 64) * 64
    up = -(-t // REF_CHUNK) * REF_CHUNK          # whole reference chunks, if that does not add a tile's worth of rays
    return up if up <= max_tile else t


@torch.no_grad()
def render_frame_shard(model, rays, envs, rank=0, world=1, tile=None, keys=("comp_rgb_phys_full",),
                       share_across_envs=True):
    """Render this rank's pixels of one frame under every env map.  rays: [H*W, 6] on the device (the whole frame:
    the rank keeps `rays[rank::world]`).  Returns {env_index: {key: [n_my_rays, C]}} -- row i is pixel
    rank + i * world of the frame -- plus the tile list (ranges inside the shard).

    share_across_envs: a tile is rendered under all maps back to back with a tile cache installed on the model
    (`SplitMixedOCCModel._memo`): sampling, field evaluations, material networks and the secondary bounce run once
    per tile, only the emitter lookups, compositing and the third-bounce shading run per map.  The frames are
    bit-identical to rendering every map from scratch (share_across_envs=False, the reference's loop order)."""
    if world > 1:
        rays = rays[my_pixels(rays.shape[0], rank, world)]          # rows of the outputs follow this order
    if tile is None:
        tile = balanced_tile(rays.shape[0], 1)
    tiles = my_tiles(rays.shape[0], tile, 0, 1)
    n_env = len(envs.maps)
    parts = {e: {k: [] for k in keys} for e in range(n_env)}
    try:
        if share_across_envs:
            for a, b in tiles:
                model._tile_cache = {}
                for e in range(n_env):
                    envs.use(e)
                    o = model.forward_(rays[a:b], relighting=True)
                    for k in keys:
                        parts[e][k].append(o[k])
        else:
            for e in range(n_env):
                envs.use(e)
                for a, b in tiles:
                    o = model.forward_(rays[a:b], relighting=True)
                    for k in keys:
                        parts[e][k].append(o[k])
    finally:
        model._tile_cache = None
    out = {e: {k: torch.cat(v) if v else torch.zeros(0, 3, device=rays.device) for k, v in parts[e].items()}
           for e in range(n_env)}
    return out, tiles


EVAL_KEYS = ("comp_rgb_phys_full", "comp_albedo", "comp_normal")


@torch.no_grad()
def evaluate_frame(model, rays, hw, envs, targets):
    """Score one test view of a stage-1 SplitMixedOCCModel as SplitOccSystem.test_step does (systems/split_occ.py:
    331-458, scores at :417-424): one render_frame_shard on this GPU (the albedo and normal keys ride along with the
    env-shared tile cache), then the metrics of rise_sdf_b200.metrics.  rays: [H*W, 6] on the device, hw = (H, W),
    envs: an EnvSet.  targets (every key optional): "mask" [H,W] bool, "albedo" [H,W,3] linear, "normal" [H,W,3]
    world-space vectors in the model's frame, "relit" one [H,W,3] per env map in the model's output space (sRGB,
    background composited with model.background_color).  Without a mask, albedo and normal scores cover every pixel.

    Returns Python floats: albedo_scale (3 values: the per-channel median ratio), albedo_psnr (masked, after aligning
    the prediction by albedo_scale, without clamping), albedo_ssim (the aligned prediction and the target, both set to 0
    outside the mask: this project's choice), normal_mae (degrees, masked), relit_psnr / relit_ssim (one value per env
    map, full frame).  All scalars are stacked on the device and read back once.  Averaging over views is the caller's."""
    H, W = hw
    relit = targets.get("relit")
    if relit is not None and len(relit) != len(envs.maps):
        raise ValueError(f"{len(relit)} relit targets for {len(envs.maps)} env maps")
    out, _ = render_frame_shard(model, rays, envs, keys=EVAL_KEYS)
    img = lambda e, k: out[e][k].view(H, W, 3)
    mask = targets.get("mask")
    if mask is None and ("albedo" in targets or "normal" in targets):
        mask = torch.ones(H, W, dtype=torch.bool, device=rays.device)
    parts = []                                    # (name, device tensor [n]), read back together
    if "albedo" in targets:
        gt = targets["albedo"]
        scale = metrics.albedo_scale(img(0, "comp_albedo"), gt, mask)
        aligned = img(0, "comp_albedo") * scale
        m3 = mask[..., None]
        parts += [("albedo_scale", scale.double()), ("albedo_psnr", metrics.psnr(aligned, gt, mask)),
                  ("albedo_ssim", metrics.ssim(torch.where(m3, aligned, 0.0), torch.where(m3, gt, 0.0)))]
    if "normal" in targets:
        parts.append(("normal_mae", metrics.normal_mae(img(0, "comp_normal"), targets["normal"], mask)))
    for e, gt in enumerate(relit or []):
        rgb = img(e, "comp_rgb_phys_full")
        parts += [("relit_psnr", metrics.psnr(rgb, gt)), ("relit_ssim", metrics.ssim(rgb, gt))]
    if not parts:
        return {}
    flat = torch.cat([v.reshape(-1) for _, v in parts]).tolist()        # the frame's one device-to-host copy
    res, i = {}, 0
    for name, v in parts:
        vals, i = flat[i:i + v.numel()], i + v.numel()
        if name == "albedo_scale":
            res[name] = vals
        elif name in ("relit_psnr", "relit_ssim"):
            res.setdefault(name, []).extend(vals)
        else:
            res[name] = vals[0]
    return res


def synthetic_envs():
    return [syn.env_latlong("bridge", seed=1), syn.env_latlong("city", seed=2)]
