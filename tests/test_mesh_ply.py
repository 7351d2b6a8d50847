"""Binary PLY mesh writer (`formats.save_mesh_ply`): exact header, round trip through a small numpy reader with and
without vertex colours, empty mesh.  CPU only."""
import numpy as np
import pytest
import torch

from rise_sdf_b200 import formats


def read_ply(path):
    """(vertex record array, faces int64 [F, 3]) of a binary little-endian triangle-mesh PLY with float vertex
    properties and a `list uchar int` face property."""
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    counts, props, elem = {}, {"vertex": [], "face": []}, None
    for ln in lines[2:-1]:
        tok = ln.split()
        if tok[0] == "element":
            elem = tok[1]
            counts[elem] = int(tok[2])
        elif tok[0] == "property":
            props[elem].append(tok[1:])
    assert all(p[0] == "float" for p in props["vertex"])
    assert props["face"] == [["list", "uchar", "int", "vertex_indices"]]
    vdt = np.dtype([(p[1], "<f4") for p in props["vertex"]])
    nv, nf = counts["vertex"], counts["face"]
    verts = np.frombuffer(data, vdt, nv, end)
    faces = np.frombuffer(data, [("n", "u1"), ("i", "<i4", (3,))], nf, end + nv * vdt.itemsize)
    assert (faces["n"] == 3).all()
    assert len(data) == end + nv * vdt.itemsize + nf * 13
    return verts, faces["i"].astype(np.int64)


def test_round_trip_with_and_without_colours(tmp_path):
    rng = np.random.default_rng(0)
    v = rng.standard_normal((50, 3)).astype(np.float32)
    f = rng.integers(0, 50, (80, 3))
    c = rng.random((50, 3)).astype(np.float32)
    for rgb in (None, c):
        path = formats.save_mesh_ply(str(tmp_path / "m.ply"), torch.from_numpy(v), torch.from_numpy(f),
                                     None if rgb is None else torch.from_numpy(rgb))
        verts, faces = read_ply(path)
        assert np.array_equal(faces, f)
        assert np.array_equal(np.stack([verts["x"], verts["y"], verts["z"]], -1), v)
        if rgb is None:
            assert verts.dtype.names == ("x", "y", "z")
        else:
            assert np.array_equal(np.stack([verts["red"], verts["green"], verts["blue"]], -1), rgb)
    # numpy inputs are accepted as well
    verts, faces = read_ply(formats.save_mesh_ply(str(tmp_path / "n.ply"), v, f))
    assert np.array_equal(faces, f)


def test_exact_header(tmp_path):
    path = formats.save_mesh_ply(str(tmp_path / "h.ply"), torch.zeros(4, 3), torch.zeros(2, 3, dtype=torch.int64),
                                 torch.ones(4, 3))
    head = open(path, "rb").read().split(b"end_header\n")[0] + b"end_header\n"
    assert head == (b"ply\nformat binary_little_endian 1.0\nelement vertex 4\nproperty float x\nproperty float y\n"
                    b"property float z\nproperty float red\nproperty float green\nproperty float blue\n"
                    b"element face 2\nproperty list uchar int vertex_indices\nend_header\n")


def test_empty_mesh(tmp_path):
    path = formats.save_mesh_ply(str(tmp_path / "e.ply"), torch.zeros(0, 3), torch.zeros(0, 3, dtype=torch.int64))
    assert open(path, "rb").read() == (b"ply\nformat binary_little_endian 1.0\nelement vertex 0\nproperty float x\n"
                                       b"property float y\nproperty float z\nelement face 0\n"
                                       b"property list uchar int vertex_indices\nend_header\n")
    verts, faces = read_ply(path)
    assert len(verts) == 0 and faces.shape == (0, 3)


def test_colour_rows_must_match_vertices(tmp_path):
    with pytest.raises(ValueError, match="v_rgb"):
        formats.save_mesh_ply(str(tmp_path / "x.ply"), torch.zeros(4, 3), torch.zeros(1, 3, dtype=torch.int64),
                              torch.zeros(3, 3))
