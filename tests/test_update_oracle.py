"""CPU: the numpy restatement of Mesh::Mesh's normals (tests/update_oracle.py), which the vertex-update tests use as the
reference, equals the host front end's flattened face and vertex normals bit for bit (NaN alike) on every fixture."""
import numpy as np
import pytest

import kd_build_oracle as kb
import update_oracle as uo
from conftest import SMALL_SCENES, same_f32


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_normals_restatement_matches_front_end(name, loaded, crt):
    _, flat, _, _ = loaded[name]
    a = kb.scene_arrays(flat)
    fn, vn = uo.mesh_normals(a["vertex_position"], a["triangle_vertex"])
    assert same_f32(fn, a["triangle_normal"]).all()
    assert same_f32(vn, a["vertex_normal"]).all()
    assert np.array_equal(crt.scene_vertex_positions(flat).view(np.uint32), a["vertex_position"].view(np.uint32))


def test_signed_zero_fold_starts_at_plus_zero():
    """A vertex whose corners all add -0.0 components keeps +0.0 (the reference adds to a zero-initialised Vector); a
    degenerate triangle's zero normal stays zero."""
    vp = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [5, 5, 5]], np.float32)
    tv = np.array([[0, 1, 2], [3, 3, 3]], np.uint32)
    fn, vn = uo.mesh_normals(vp, tv)
    assert fn[0].tolist() == [0.0, 0.0, 1.0] and np.signbit(fn[0, :2]).tolist() == [False, False]
    assert (fn[1] == 0).all() and (vn[3] == 0).all()
    # edge (1, -0, 0) x (0, 1, 0) = (-0, +0, 1): every vertex normal's x is +0 + -0 = +0
    vp2 = np.array([[0, 0, 0], [1, -0.0, 0], [0, 1, 0]], np.float32)
    fn2, vn2 = uo.mesh_normals(vp2, np.array([[0, 1, 2]], np.uint32))
    assert fn2[0, 0] == 0 and np.signbit(fn2[0, 0])
    assert (vn2[:, 0] == 0).all() and not np.signbit(vn2[:, 0]).any()


def test_edited_scene_copies_everything_but_geometry(loaded, crt):
    _, flat, _, _ = loaded["hw11_room"]
    a = kb.scene_arrays(flat)
    moved = a["vertex_position"] + np.float32(0.25)
    e = uo.EditedScene(crt, flat, moved)
    b = kb.scene_arrays(e.ptr)
    assert np.array_equal(b["vertex_position"], moved)
    fn, vn = uo.mesh_normals(moved, a["triangle_vertex"])
    assert same_f32(b["triangle_normal"], fn).all() and same_f32(b["vertex_normal"], vn).all()
    for k in ("vertex_uv", "triangle_vertex", "materials", "textures", "texels", "lights"):
        assert np.array_equal(a[k], b[k]), k
    for f in ("material", "first_triangle", "n_triangles", "first_vertex", "n_vertices"):
        assert np.array_equal(a["meshes"][f], b["meshes"][f]), f
    assert e.scene.n_mesh_nodes == e.scene.n_top_nodes == 0 and not e.scene.mesh_nodes
