"""Drop-in for PyMCubes' `mcubes.marching_cubes(volume, isovalue)` (models/geometry.py:60), on the device.

The reference copies every level chunk to the host and meshes the 512^3 grid on the CPU, twice per `isosurface()`.
Here the grid stays resident: two passes of csrc/mcubes.cu over it with one host read-back of (V, F) in between.

Conventions (include/rsdf_b200.h, `rsdf_mc_count`):
  * a grid vertex is inside when value > isovalue, value = -volume with `negate=True` (no negated copy is made);
  * one welded vertex per grid edge whose ends differ, t = (iso - va) / (vb - va) from the edge's lower end, in fp32;
  * faces are wound so that right-hand normals point towards decreasing value (out of the object for -sdf);
  * vertices are ordered by the edge's lower grid corner's linear index, then axis x < y < z; faces by the cell's
    linear index, then triangle-table order.  The output is deterministic.
The triangle table comes from a face-walk rule that decides each ambiguous face from its own four signs, so the mesh
is closed and consistently oriented; it is not PyMCubes' table, so ambiguous cells may be split differently.

`marching_cubes` takes a dense volume of at most 2^31 - 1 grid edges (about 894^3).  `marching_cubes_slabs` meshes a
volume of any size from a callback that produces it one x-slab at a time (`rsdf_mc_slab_count` / `_emit`): each
slab's level values, scratch and mesh are bounded, and the concatenated result is the dense result, bit for bit.
"""
import operator

import torch

from . import _lib as L

TILE = 2048                    # grid vertices per block of csrc/mcubes.cu
SCRATCH_PER_TILE = 1048        # bytes of scratch per tile
MAX_EDGES = 2 ** 31 - 1        # 3 * nx * ny * nz must fit int32: vertex ids are int32 on the device
SLAB_BYTES = 1 << 30           # level values owned by one slab of `marching_cubes_slabs`
MAX_LAYERS = 1 << 24           # slab vertices sit at x0 + x in fp32, exact below 2^24


def scratch_bytes(shape):
    nx, ny, nz = shape
    return SCRATCH_PER_TILE * -(-(nx * ny * nz) // TILE)


def marching_cubes(volume, isovalue, negate=False):
    """volume: CUDA tensor [nx, ny, nz] (x-major, as `VolumeSDF.isosurface_level` returns it).  Returns
    (vertices float32 [V, 3] in index space, faces int64 [F, 3]) on the volume's device.  Raises ValueError when
    3 * nx * ny * nz exceeds 2^31 - 1 (about 894^3)."""
    L.require_cuda(volume)
    if volume.dim() != 3:
        raise ValueError(f"marching_cubes expects a 3-D volume, got shape {tuple(volume.shape)}")
    nx, ny, nz = volume.shape
    if 3 * nx * ny * nz > MAX_EDGES:
        raise ValueError(f"volume {tuple(volume.shape)} has {3 * nx * ny * nz} grid edges; at most {MAX_EDGES} "
                         "(3 * nx * ny * nz < 2^31) are supported")
    dev = volume.device
    if min(nx, ny, nz) < 2:
        return torch.zeros(0, 3, dtype=torch.float32, device=dev), torch.zeros(0, 3, dtype=torch.int64, device=dev)
    vol = volume.detach().to(torch.float32).contiguous()
    scratch = torch.empty(scratch_bytes(vol.shape), dtype=torch.uint8, device=dev)
    totals = torch.empty(2, dtype=torch.int64, device=dev)
    args = (L.ptr(vol), nx, ny, nz, float(isovalue), int(bool(negate)), L.ptr(scratch))
    L.call("rsdf_mc_count", *args, L.ptr(totals), L.stream())
    n_verts, n_faces = totals.tolist()                       # the one host read-back: sizes of the outputs
    verts = torch.empty(n_verts, 3, dtype=torch.float32, device=dev)
    faces = torch.empty(n_faces, 3, dtype=torch.int64, device=dev)
    if n_verts:
        L.call("rsdf_mc_emit", *args, L.ptr(verts), L.ptr(faces), L.stream())
    return verts, faces


def plan_slabs(shape, slab_layers=None):
    """[(x0, own, p)] for the x-slabs of a volume of `shape`: slab k owns layers [x0, x0 + own) and presents
    p = min(own + 2, nx - x0) layers to the kernels.  `own` is `slab_layers` (default: SLAB_BYTES of fp32 level values,
    at least one layer) capped so that 3 * p * ny * nz fits int32; a final slab of one layer is folded into the one
    before it, because the kernels need p >= 2."""
    nx, ny, nz = _check_shape(shape)
    if min(nx, ny, nz) < 2:
        return []
    max_p = MAX_EDGES // (3 * ny * nz)
    cap = nx if nx <= max_p else max_p - 2
    if cap < 1:
        raise ValueError(f"ny * nz = {ny * nz} is too large: even one owned layer with its two halo layers exceeds "
                         f"{MAX_EDGES} grid edges")
    if slab_layers is None:
        slab_layers = max(1, SLAB_BYTES // (4 * ny * nz))
    if int(slab_layers) < 1:
        raise ValueError(f"slab_layers must be positive, got {slab_layers}")
    own = min(int(slab_layers), cap)
    plan, x0 = [], 0
    while x0 < nx:
        n = min(own, nx - x0)
        if nx - x0 - n == 1:
            n += 1
        plan.append((x0, n, min(n + 2, nx - x0)))
        x0 += n
    return plan


def _check_shape(shape):
    try:
        dims = tuple(operator.index(d) for d in shape)
    except TypeError:
        dims = ()
    if len(dims) != 3 or min(dims) < 0:
        raise ValueError(f"shape must be three non-negative ints, got {shape!r}")
    shape = dims
    if shape[0] > MAX_LAYERS:
        raise ValueError(f"nx = {shape[0]} exceeds {MAX_LAYERS}: index-space x would not be exact in fp32")
    return shape


def marching_cubes_slab_iter(layers, shape, isovalue, negate=False, slab_layers=None):
    """Yields (vertices float32 [V_k, 3], faces int64 [F_k, 3]) of each x-slab in x order, on the device.  The
    volume [nx, ny, nz] = `shape` is never materialised: `layers(x0, n)` returns its layers [x0, x0 + n) as a
    contiguous CUDA float32 tensor [n, ny, nz] (it may reuse one buffer: the slab is consumed before the next call).
    Vertices are in the volume's index space and face ids are global, so concatenating the slabs gives
    `marching_cubes(volume, isovalue, negate)`.  One host read-back per slab (its V, F); one scratch buffer, sized for
    the largest slab, serves every slab."""
    nx, ny, nz = _check_shape(shape)
    plan = plan_slabs(shape, slab_layers)
    scratch = totals = dev = None
    vbase = 0
    for x0, own, p in plan:
        vol = layers(x0, p)
        if not isinstance(vol, torch.Tensor) or not vol.is_cuda or vol.dtype != torch.float32:
            raise ValueError(f"layers({x0}, {p}) must return a CUDA float32 tensor, got "
                             f"{type(vol).__name__ if not isinstance(vol, torch.Tensor) else (vol.dtype, vol.device)}")
        if tuple(vol.shape) != (p, ny, nz) or not vol.is_contiguous():
            raise ValueError(f"layers({x0}, {p}) must return a contiguous tensor of shape {(p, ny, nz)}, got "
                             f"{tuple(vol.shape)}{'' if vol.is_contiguous() else ' (not contiguous)'}")
        if dev is None:
            dev = vol.device
            scratch = torch.empty(scratch_bytes((max(q for _, _, q in plan), ny, nz)), dtype=torch.uint8, device=dev)
            totals = torch.empty(2, dtype=torch.int64, device=dev)
        elif vol.device != dev:
            raise ValueError(f"layers({x0}, {p}) returned a tensor on {vol.device}, earlier slabs were on {dev}")
        args = (L.ptr(vol), p, ny, nz, own)
        tail = (float(isovalue), int(bool(negate)), L.ptr(scratch))
        L.call("rsdf_mc_slab_count", *args, *tail, L.ptr(totals), L.stream())
        n_verts, n_faces = totals.tolist()                   # the slab's one host read-back
        verts = torch.empty(n_verts, 3, dtype=torch.float32, device=dev)
        faces = torch.empty(n_faces, 3, dtype=torch.int64, device=dev)
        if n_verts:
            L.call("rsdf_mc_slab_emit", *args, x0, vbase, *tail, L.ptr(verts), L.ptr(faces), L.stream())
        del vol
        yield verts, faces
        vbase += n_verts


def marching_cubes_slabs(layers, shape, isovalue, negate=False, slab_layers=None):
    """`marching_cubes` of the volume that `layers(x0, n)` produces slab by slab (see `marching_cubes_slab_iter`), at
    any size: (vertices float32 [V, 3], faces int64 [F, 3]) on the device, equal to the dense result bit for bit
    wherever that exists."""
    parts = list(marching_cubes_slab_iter(layers, shape, isovalue, negate, slab_layers))
    if not parts:
        return torch.zeros(0, 3, dtype=torch.float32, device="cuda"), torch.zeros(0, 3, dtype=torch.int64, device="cuda")
    if len(parts) == 1:
        return parts[0]
    verts = torch.cat([v for v, _ in parts])
    faces = torch.cat([f for _, f in parts])
    return verts, faces
