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
"""
import torch

from . import _lib as L

TILE = 2048                    # grid vertices per block of csrc/mcubes.cu
SCRATCH_PER_TILE = 1048        # bytes of scratch per tile
MAX_EDGES = 2 ** 31 - 1        # 3 * nx * ny * nz must fit int32: vertex ids are int32 on the device


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
