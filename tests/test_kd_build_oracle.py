"""CPU: pins the restatement of the KD build rules (tests/kd_build_oracle.py) against the host builder and the stored
reference trees, and the front end's geometry-only flatten against the full one.  The GPU tests of the device builder
(test_gpu_device_build.py) use the restatement for scenes that cannot be written as .crtscene files."""
import os

import numpy as np
import pytest

import kd_build_oracle as kb
from conftest import ROOT, SMALL_SCENES

GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_restatement_equals_host_builder(name, loaded):
    sf, flat, _, _ = loaded[name]
    kb.assert_trees_equal(kb.scene_trees(flat), kb.host_trees(flat))


@pytest.mark.parametrize("name", ["hw11_room", "hw14_small", "degenerate_uv"])
def test_restatement_equals_stored_reference_trees(name, loaded, ob, tmp_path):
    """The restatement against kdtrees_<name>.npz (the reference's --dump-tree format), node for node."""
    sf, flat, _, _ = loaded[name]
    dump = tmp_path / "trees.bin"
    dump.write_bytes(np.load(os.path.join(GOLDEN, "kdtrees_" + name + ".npz"))["dump"].tobytes())
    ref_meshes, ref_top = ob.read_reference_trees(str(dump))
    t = kb.scene_trees(flat)
    assert len(ref_meshes) == len(t["mesh_fields"])

    def check(ref_nodes, nodes, refs):
        assert len(ref_nodes) == len(nodes)
        for k, (box, c0, c1, idx) in enumerate(ref_nodes):
            assert np.array_equal(kb.box_bits(nodes[k:k + 1])[0], box.view(np.uint32))
            assert tuple(nodes[k]["child"]) == (c0, c1)
            assert list(refs[nodes[k]["leaf_start"]:nodes[k]["leaf_start"] + nodes[k]["leaf_count"]]) == list(idx)

    for m, (fn, nn, fr, nr) in enumerate(t["mesh_fields"]):
        check(ref_meshes[m], t["mesh_nodes"][fn:fn + nn], t["mesh_leaf_refs"][fr:fr + nr])
    check(ref_top, t["top_nodes"], t["top_leaf_refs"])


def test_restatement_edge_rules():
    """What the exact rules say on inputs no .crtscene has: signed zeros keep the first one's bits, NaN never enters a
    box, an empty mesh has a 0-element leaf root with the empty box, coincident triangles run to depth-25 leaves."""
    vp = np.array([[-0.0, 0, 0], [1, 0, 0], [0, 1, 0], [0.0, 0, 0], [1, 1, 0], [np.nan, 2, 0]], np.float32)
    t = kb.build_scene_trees(vp, [[0, 1, 2], [3, 4, 5]], [(0, 1), (1, 1), (2, 0)])
    root0 = t["mesh_nodes"][0]
    assert np.float32(root0["box_min"][0]).view(np.uint32) == 0x80000000  # -0.0 first
    root1 = t["mesh_nodes"][t["mesh_fields"][1][0]]
    assert np.float32(root1["box_min"][0]).view(np.uint32) == 0 and root1["box_max"][0] == 1  # NaN ignored
    empty = t["mesh_nodes"][t["mesh_fields"][2][0]]
    assert empty["leaf_count"] == 0 and empty["box_min"][0] == kb.FLT_MAX and empty["box_max"][0] == -kb.FLT_MAX
    assert np.float32(t["top_nodes"][0]["box_min"][0]).view(np.uint32) == 0x80000000
    vp, tv = kb.coincident_triangles(10)
    c = kb.build_scene_trees(vp, tv, [(0, 11)])
    # one chain of 25 inner nodes, each with a leaf holding the big triangle alone, ends in a depth-25 leaf of all 11
    assert len(c["mesh_nodes"]) == 51 and np.sort(c["mesh_nodes"]["leaf_count"])[-2:].tolist() == [1, 11]


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_geometry_flatten_equals_full_flatten_without_trees(name, built, scene_dir):
    """crtfe_scene_flatten_geometry: every non-tree array equal to crtfe_scene_flatten's, tree counts 0, tree arrays
    NULL, the meshes' tree fields 0; and it leaves the full flatten as it was."""
    sf = built.SceneFile(name + ".crtscene", scene_dir)
    full = kb.scene_arrays(sf.flatten())
    g_ptr = sf.flatten(trees=False)
    geo = kb.scene_arrays(g_ptr)
    s = g_ptr.contents
    assert (s.n_mesh_nodes, s.n_mesh_leaf_refs, s.n_top_nodes, s.n_top_leaf_refs) == (0, 0, 0, 0)
    assert not s.mesh_nodes and not s.mesh_leaf_refs and not s.top_nodes and not s.top_leaf_refs
    for k in ("vertex_position", "vertex_normal", "vertex_uv", "triangle_vertex", "triangle_normal", "materials", "textures",
              "texels", "lights"):
        assert geo[k].tobytes() == full[k].tobytes(), k
    for f in ("material", "first_triangle", "n_triangles", "first_vertex", "n_vertices"):
        assert np.array_equal(geo["meshes"][f], full["meshes"][f]), f
    for f in ("first_node", "n_nodes", "first_leaf_ref", "n_leaf_refs"):
        assert not geo["meshes"][f].any(), f
    f = sf.flatten().contents
    assert (s.width, s.height, list(s.background)) == (f.width, f.height, list(f.background))
    assert kb.scene_arrays(sf.flatten())["mesh_nodes"].tobytes() == full["mesh_nodes"].tobytes()
    sf.close()
