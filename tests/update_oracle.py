"""CPU restatement of Mesh::Mesh's normals (Scene.cpp:5-30; csrc/frontend/crt_scene.cpp) in numpy binary32, and a
flattened scene copied with its vertex positions replaced: what crtb200_update_vertices_device must leave on the device
(DESIGN.md 3.14) is what crtb200_upload_geometry leaves for such a copy.

Test infrastructure only."""
import ctypes as C

import numpy as np

import kd_build_oracle as kb


def _normalize(v):
    """Vector::normalize (Vector.cpp:97-106) row by row: len = sqrt((x*x + y*y) + z*z); unchanged when len == 0, else
    every component times 1.0f / len.  Every operation rounds to binary32 (numpy ufuncs never contract)."""
    x, y, z = v[:, 0], v[:, 1], v[:, 2]
    ln = np.sqrt(x * x + y * y + z * z)
    inv = np.float32(1.0) / np.where(ln == 0, np.float32(1.0), ln)
    out = v * inv[:, None]
    return np.where((ln == 0)[:, None], v, out).astype(np.float32)


def mesh_normals(vertex_position, triangle_vertex):
    """(face normals (T, 3), vertex normals (V, 3)) as Mesh::Mesh computes them, over global vertex ids: face normal
    n = cross(p1 - p0, p2 - p0) normalised; each vertex normal starts at +0.0 and adds, for every triangle in order and
    its corners 0, 1, 2, the face normal at that corner's vertex, then is normalised."""
    vp = np.ascontiguousarray(vertex_position, np.float32).reshape(-1, 3)
    tv = np.ascontiguousarray(triangle_vertex, np.int64).reshape(-1, 3)
    with np.errstate(all="ignore"):
        p0, p1, p2 = vp[tv[:, 0]], vp[tv[:, 1]], vp[tv[:, 2]]
        a, b = p1 - p0, p2 - p0
        cr = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                       a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1).astype(np.float32)
        fn = _normalize(cr)
        vn = np.zeros_like(vp)  # +0.0
        np.add.at(vn, tv.reshape(-1), np.repeat(fn, 3, axis=0))  # unbuffered, in index order: the serial fold
        vn = _normalize(vn)
    return fn, vn


def tri_geom(vertex_position, triangle_vertex, face_normals):
    """The device's triangle records (T, 3, 4): per corner k the position and face-normal component k."""
    vp = np.asarray(vertex_position, np.float32).reshape(-1, 3)
    tv = np.asarray(triangle_vertex, np.int64).reshape(-1, 3)
    out = np.zeros((len(tv), 3, 4), np.float32)
    out[:, :, :3] = vp[tv]
    out[:, :, 3] = face_normals
    return out


class EditedScene:
    """A copy of a flattened crtb200_scene (a ctypes POINTER(Scene)) whose vertex positions are `positions` and whose
    face and vertex normals are mesh_normals' of them; everything else is shared with the original, which must outlive
    this object.  trees: None for crtb200_upload_geometry (tree arrays NULL), or a kd_build_oracle.build_scene_trees
    result for crtb200_upload_scene and the CPU oracle."""

    def __init__(self, crt, scene_ptr, positions, trees=None):
        src = scene_ptr.contents
        s = crt.Scene()
        C.memmove(C.byref(s), C.byref(src), C.sizeof(crt.Scene))
        self.positions = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
        assert len(self.positions) == src.n_vertices
        tv = kb._arr(src.triangle_vertex, src.n_triangles, np.uint32, 3)
        self.face_normals, self.vertex_normals = mesh_normals(self.positions, tv)
        self.keep = [self.positions, self.face_normals, self.vertex_normals]
        s.vertex_position = self._p(self.positions, C.c_float)
        s.vertex_normal = self._p(self.vertex_normals, C.c_float)
        s.triangle_normal = self._p(self.face_normals, C.c_float)
        meshes = kb._arr(src.meshes, src.n_meshes, kb.MESH_DTYPE)
        for k in ("first_node", "n_nodes", "first_leaf_ref", "n_leaf_refs"):
            meshes[k] = 0
        for k in ("mesh_nodes", "top_nodes", "mesh_leaf_refs", "top_leaf_refs"):
            setattr(s, "n_" + k, 0)
            setattr(s, k, None)
        if trees is not None:
            f = trees["mesh_fields"]
            for i, k in enumerate(("first_node", "n_nodes", "first_leaf_ref", "n_leaf_refs")):
                meshes[k] = f[:, i]
            for k, typ in (("mesh_nodes", crt.KdNode), ("top_nodes", crt.KdNode), ("mesh_leaf_refs", C.c_uint32),
                           ("top_leaf_refs", C.c_uint32)):
                a = np.ascontiguousarray(trees[k])
                setattr(s, "n_" + k, len(a))
                setattr(s, k, self._p(a, typ) if len(a) else None)
        s.meshes = self._p(meshes, crt.Mesh) if len(meshes) else None
        self.scene = s
        self.ptr = C.pointer(s)

    def _p(self, a, typ):
        a = np.ascontiguousarray(a)
        self.keep.append(a)
        return C.cast(a.ctypes.data, C.POINTER(typ))


def with_trees(crt, scene_ptr, positions):
    """EditedScene carrying the trees kd_build_oracle builds for the edited positions (the CPU oracle walks them)."""
    src = scene_ptr.contents
    tv = kb._arr(src.triangle_vertex, src.n_triangles, np.uint32, 3)
    m = kb._arr(src.meshes, src.n_meshes, kb.MESH_DTYPE)
    trees = kb.build_scene_trees(positions, tv, list(zip(m["first_triangle"].tolist(), m["n_triangles"].tolist())))
    return EditedScene(crt, scene_ptr, positions, trees)
