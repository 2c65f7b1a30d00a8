"""CPU restatement of the KD build rules (DESIGN.md 3.11; the host builder csrc/frontend/crt_kdtree.cpp and the device
builder csrc/crt_build.cuh both follow them): TriangleKDTree(mesh, 25, 8) per mesh and ObjectKDTree(scene, 25, 4)
(AccelerationStructure.cpp:12-50), in binary32, numbered and flattened as buildFlatScene does.  Also the helpers the
tests use to read a crtb200_scene into numpy arrays and to make one from arrays.

Test infrastructure only."""
import ctypes as C

import numpy as np

FLT_MAX = np.float32(np.finfo(np.float32).max)
INVALID = 0xFFFFFFFF
MAX_DEPTH = 25
KDNODE_DTYPE = np.dtype([("box_min", np.float32, 3), ("box_max", np.float32, 3), ("child", np.uint32, 2),
                         ("leaf_start", np.uint32), ("leaf_count", np.uint32)])


def triangle_boxes(p):
    """p: (n, 3 vertices, 3) float32.  BoundingBox(const Triangle&): grown over vertices 0, 1, 2 from {FLT_MAX, -FLT_MAX}
    with mn = (v < mn) ? v : mn, mx = (mx < v) ? v : mx -- a NaN coordinate never enters."""
    mn = np.full(p.shape[:1] + (3,), FLT_MAX, np.float32)
    mx = np.full(p.shape[:1] + (3,), -FLT_MAX, np.float32)
    for k in range(3):
        v = p[:, k]
        mn = np.where(v < mn, v, mn)
        mx = np.where(mx < v, v, mx)
    return mn, mx


def fold_boxes(mn, mx):
    """The serial fold of boxes (n, 3) in order from {FLT_MAX, -FLT_MAX}: per bound the FIRST value among those that
    compare equal to the extreme wins (so -0.0 / +0.0 keep the bits of the first one)."""
    out_mn = np.full(3, FLT_MAX, np.float32)
    out_mx = np.full(3, -FLT_MAX, np.float32)
    for a in range(3):
        v = mn[:, a]
        cand = v < FLT_MAX
        if cand.any():
            i = np.flatnonzero(cand & (v == v[cand].min()))[0]
            out_mn[a] = v[i]
        v = mx[:, a]
        cand = -FLT_MAX < v
        if cand.any():
            i = np.flatnonzero(cand & (v == v[cand].max()))[0]
            out_mx[a] = v[i]
    return out_mn, out_mx


def build_tree(emn, emx, root_mn, root_mx, max_leaf):
    """KDTree<T>::build (KDTree.cpp:10-46): (nodes KDNODE_DTYPE in pre-order, child 0's subtree first; leaf refs)."""
    nodes, refs = [], []
    with np.errstate(over="ignore", invalid="ignore"):
        def rec(bmn, bmx, depth, idx):
            me = len(nodes)
            nodes.append([bmn, bmx, INVALID, INVALID, 0, 0])
            if depth >= MAX_DEPTH or len(idx) <= max_leaf:
                nodes[me][4], nodes[me][5] = len(refs), len(idx)
                refs.extend(idx.tolist())
                return me
            axis = depth % 3
            middle = np.float32(np.float32(bmx[axis] - bmn[axis]) / np.float32(2))
            plane = np.float32(bmn[axis] + middle)
            c0mx, c1mn = bmx.copy(), bmn.copy()
            c0mx[axis] = plane
            c1mn[axis] = plane
            a_mn, a_mx = emn[idx], emx[idx]
            e0 = idx[~((bmn > a_mx) | (c0mx < a_mn)).any(axis=1)]
            e1 = idx[~((c1mn > a_mx) | (bmx < a_mn)).any(axis=1)]
            if len(e0):
                nodes[me][2] = rec(bmn, c0mx, depth + 1, e0)
            if len(e1):
                nodes[me][3] = rec(c1mn, bmx, depth + 1, e1)
            return me

        rec(np.asarray(root_mn, np.float32), np.asarray(root_mx, np.float32), 0, np.arange(len(emn), dtype=np.int64))
    out = np.zeros(len(nodes), KDNODE_DTYPE)
    for k, (bmn, bmx, c0, c1, ls, lc) in enumerate(nodes):
        out[k] = (bmn, bmx, (c0, c1), ls, lc)
    return out, np.array(refs, np.uint32)


def build_scene_trees(vertex_position, triangle_vertex, mesh_ranges):
    """All trees of a scene, flattened as buildFlatScene flattens them.  vertex_position (V, 3) f32, triangle_vertex
    (T, 3) global vertex ids, mesh_ranges [(first_triangle, n_triangles)] in mesh order.  Returns a dict with
    'mesh_fields' (M x 4: first_node, n_nodes, first_leaf_ref, n_leaf_refs), 'mesh_nodes', 'mesh_leaf_refs' (mesh-local),
    'top_nodes', 'top_leaf_refs'."""
    vp = np.asarray(vertex_position, np.float32).reshape(-1, 3)
    tv = np.asarray(triangle_vertex, np.int64).reshape(-1, 3)
    mesh_nodes, mesh_refs, fields, root_mn, root_mx = [], [], [], [], []
    n_nodes = n_refs = 0
    for first, n in mesh_ranges:
        mn, mx = triangle_boxes(vp[tv[first:first + n]])
        rmn, rmx = fold_boxes(mn, mx)
        nodes, refs = build_tree(mn, mx, rmn, rmx, 8)
        fields.append((n_nodes, len(nodes), n_refs, len(refs)))
        n_nodes += len(nodes)
        n_refs += len(refs)
        mesh_nodes.append(nodes)
        mesh_refs.append(refs)
        root_mn.append(rmn)
        root_mx.append(rmx)
    bmn = np.array(root_mn, np.float32).reshape(-1, 3)
    bmx = np.array(root_mx, np.float32).reshape(-1, 3)
    smn, smx = fold_boxes(bmn, bmx)  # BoundingBox(scene): the fold over all triangles in order, regrouped by mesh
    top, top_refs = build_tree(bmn, bmx, smn, smx, 4)
    return {"mesh_fields": np.array(fields, np.uint32).reshape(-1, 4),
            "mesh_nodes": np.concatenate(mesh_nodes) if mesh_nodes else np.zeros(0, KDNODE_DTYPE),
            "mesh_leaf_refs": np.concatenate(mesh_refs) if mesh_refs else np.zeros(0, np.uint32),
            "top_nodes": top, "top_leaf_refs": top_refs}


def coincident_triangles(n):
    """One triangle spanning [0, 1]^3 and n coincident tiny triangles inside it, away from every split plane: the node
    holding them never drops to 8 elements, so it runs to a depth-25 leaf (without making the tree grow wide)."""
    big = [[0, 0, 0], [1, 0, 1], [0, 1, 1]]
    tiny = [[0.3, 0.3, 0.3], [0.3000001, 0.3, 0.3], [0.3, 0.3000001, 0.3]]
    vp = np.array(big + tiny * n, np.float32)
    return vp, np.arange(3 * (n + 1), dtype=np.uint32).reshape(-1, 3)


def _arr(ptr, n, dtype, per=1):
    if n == 0 or not ptr:
        return np.zeros((n, per) if per > 1 else n, dtype)
    a = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n * per * np.dtype(dtype).itemsize,))
    a = a.view(dtype).copy()
    return a.reshape(n, per) if per > 1 else a


MESH_FIELDS = ("material", "first_triangle", "n_triangles", "first_vertex", "n_vertices", "first_node", "n_nodes",
               "first_leaf_ref", "n_leaf_refs")
MESH_DTYPE = np.dtype([(n, np.uint32) for n in MESH_FIELDS])


def scene_arrays(scene_ptr):
    """Copies of every array of a crtb200_scene (a ctypes POINTER(Scene))."""
    s = scene_ptr.contents
    return {
        "vertex_position": _arr(s.vertex_position, s.n_vertices, np.float32, 3),
        "vertex_normal": _arr(s.vertex_normal, s.n_vertices, np.float32, 3),
        "vertex_uv": _arr(s.vertex_uv, s.n_vertices if s.vertex_uv else 0, np.float32, 3),
        "triangle_vertex": _arr(s.triangle_vertex, s.n_triangles, np.uint32, 3),
        "triangle_normal": _arr(s.triangle_normal, s.n_triangles, np.float32, 3),
        "meshes": _arr(s.meshes, s.n_meshes, MESH_DTYPE),
        "materials": _arr(s.materials, s.n_materials, np.uint8, 28),
        "textures": _arr(s.textures, s.n_textures, np.uint8, 48),
        "texels": _arr(s.texels, s.n_texels, np.float32, 3),
        "lights": _arr(s.lights, s.n_lights, np.uint8, 16),
        "mesh_nodes": _arr(s.mesh_nodes, s.n_mesh_nodes, KDNODE_DTYPE),
        "mesh_leaf_refs": _arr(s.mesh_leaf_refs, s.n_mesh_leaf_refs, np.uint32),
        "top_nodes": _arr(s.top_nodes, s.n_top_nodes, KDNODE_DTYPE),
        "top_leaf_refs": _arr(s.top_leaf_refs, s.n_top_leaf_refs, np.uint32),
    }


def host_trees(scene_ptr):
    """The trees a flattened scene carries, in build_scene_trees' form (only the tree arrays are copied)."""
    s = scene_ptr.contents
    m = _arr(s.meshes, s.n_meshes, MESH_DTYPE)
    return {"mesh_fields": np.stack([m["first_node"], m["n_nodes"], m["first_leaf_ref"], m["n_leaf_refs"]], axis=1).reshape(-1, 4),
            "mesh_nodes": _arr(s.mesh_nodes, s.n_mesh_nodes, KDNODE_DTYPE),
            "mesh_leaf_refs": _arr(s.mesh_leaf_refs, s.n_mesh_leaf_refs, np.uint32),
            "top_nodes": _arr(s.top_nodes, s.n_top_nodes, KDNODE_DTYPE),
            "top_leaf_refs": _arr(s.top_leaf_refs, s.n_top_leaf_refs, np.uint32)}


def device_trees(t):
    """Context.scene_trees() in build_scene_trees' form."""
    m = t["meshes"]
    return {"mesh_fields": np.stack([m["first_node"], m["n_nodes"], m["first_leaf_ref"], m["n_leaf_refs"]], axis=1).reshape(-1, 4),
            **{k: t[k] for k in ("mesh_nodes", "mesh_leaf_refs", "top_nodes", "top_leaf_refs")}}


def box_bits(nodes):
    return np.concatenate([nodes["box_min"], nodes["box_max"]], axis=1).view(np.uint32)


def assert_trees_equal(got, exp):
    """Trees in build_scene_trees' form: boxes as bits, children, leaf ranges, references, per-mesh ranges."""
    for k in ("mesh_nodes", "top_nodes"):
        assert len(got[k]) == len(exp[k]), k
        assert np.array_equal(box_bits(got[k]), box_bits(exp[k])), k
        for f in ("child", "leaf_start", "leaf_count"):
            assert np.array_equal(got[k][f], exp[k][f]), (k, f)
    for k in ("mesh_leaf_refs", "top_leaf_refs", "mesh_fields"):
        assert np.array_equal(np.asarray(got[k], np.uint32), np.asarray(exp[k], np.uint32)), k


def scene_trees(scene_ptr):
    """build_scene_trees of a flattened scene's geometry."""
    a = scene_arrays(scene_ptr)
    m = a["meshes"]
    return build_scene_trees(a["vertex_position"], a["triangle_vertex"], list(zip(m["first_triangle"].tolist(), m["n_triangles"].tolist())))


class ArrayScene:
    """A crtb200_scene made from numpy arrays (kept alive by this object): one diffuse material, one light, vertex normals
    = 0, face normals the geometric unit normals computed in float64 and rounded (or given).  trees: None for
    crtb200_upload_geometry, or a build_scene_trees result for crtb200_upload_scene."""

    def __init__(self, crt, vertex_position, triangle_vertex, mesh_ranges, trees=None, width=32, height=18, face_normals=None):
        self.keep = []
        vp = np.ascontiguousarray(vertex_position, np.float32).reshape(-1, 3)
        tv = np.ascontiguousarray(triangle_vertex, np.uint32).reshape(-1, 3)
        if face_normals is None:
            with np.errstate(all="ignore"):
                p = vp[tv].astype(np.float64)
                cr = np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])
                ln = np.linalg.norm(cr, axis=1, keepdims=True)
                fn = np.where(ln > 0, cr / np.where(ln > 0, ln, 1), 0).astype(np.float32)
        else:
            fn = np.ascontiguousarray(face_normals, np.float32).reshape(-1, 3)
        vn = np.zeros_like(vp)
        meshes = (crt.Mesh * max(1, len(mesh_ranges)))()
        for i, (first, n) in enumerate(mesh_ranges):
            meshes[i].material = 0
            meshes[i].first_triangle = first
            meshes[i].n_triangles = n
            if trees is not None:
                f = trees["mesh_fields"][i]
                meshes[i].first_node, meshes[i].n_nodes, meshes[i].first_leaf_ref, meshes[i].n_leaf_refs = (int(x) for x in f)
        mat = crt.Material(0, 0, INVALID, (C.c_float * 3)(0.8, 0.8, 0.8), 1.0)
        light = crt.Light((C.c_float * 3)(0.0, 5.0, 0.0), 100)
        s = crt.Scene()
        s.abi_version = crt.core().crtb200_abi_version()
        s.width, s.height = width, height
        s.n_vertices = len(vp)
        s.vertex_position = self._p(vp, C.c_float)
        s.vertex_normal = self._p(vn, C.c_float)
        s.n_triangles = len(tv)
        s.triangle_vertex = self._p(tv, C.c_uint32)
        s.triangle_normal = self._p(fn, C.c_float)
        s.n_meshes = len(mesh_ranges)
        s.meshes = C.cast(meshes, C.POINTER(crt.Mesh))
        s.n_materials = 1
        s.materials = C.pointer(mat)
        s.n_lights = 1
        s.lights = C.pointer(light)
        if trees is not None:
            for k, typ in (("mesh_nodes", crt.KdNode), ("top_nodes", crt.KdNode), ("mesh_leaf_refs", C.c_uint32), ("top_leaf_refs", C.c_uint32)):
                a = np.ascontiguousarray(trees[k])
                setattr(s, "n_" + k, len(a))
                setattr(s, k, self._p(a, typ) if len(a) else None)
        self.keep += [meshes, mat, light, s]
        self.scene = s
        self.ptr = C.pointer(s)

    def _p(self, a, typ):
        a = np.ascontiguousarray(a)
        self.keep.append(a)
        return C.cast(a.ctypes.data, C.POINTER(typ))
