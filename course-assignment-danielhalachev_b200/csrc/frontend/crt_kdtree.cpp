#include "crt_kdtree.hpp"

#include <algorithm>
#include <chrono>
#include <future>
#include <limits>
#include <thread>

namespace crt {

namespace {

constexpr unsigned AXIS_COUNT = 3;  // KDTree.h:27

struct Builder {
  const std::vector<Box> &elems;
  unsigned maxDepth, maxLeaf;

  // BoundingBox::intersects(const BoundingBox&)  BoundingBox.h:75-83 -- inclusive on both sides
  static bool overlaps(const Box &a, const Box &b) {
    for (int i = 0; i < 3; i++)
      if ((a.mn[i] > b.mx[i]) || (a.mx[i] < b.mn[i])) return false;
    return true;
  }
  static crtb200_kdnode makeNode(const Box &b) {
    crtb200_kdnode n;
    for (int i = 0; i < 3; i++) {
      n.box_min[i] = b.mn[i];
      n.box_max[i] = b.mx[i];
    }
    n.child[0] = n.child[1] = CRTB200_INVALID;
    n.leaf_start = 0;
    n.leaf_count = 0;
    return n;
  }
  // BoundingBox::split  BoundingBox.h:60-69
  static void split(const Box &b, unsigned axis, Box &first, Box &second) {
    float middle = (b.mx[axis] - b.mn[axis]) / 2;
    float plane = b.mn[axis] + middle;
    first = b;
    second = b;
    first.mx[axis] = plane;
    second.mn[axis] = plane;
  }

  // Serial build of one subtree appended to `out` in the reference's DFS pre-order; `self` already exists in out.
  void buildSerial(KDTreeData &out, uint32_t self, unsigned depth, std::vector<uint32_t> &&elements) const {
    if (depth >= maxDepth || elements.size() <= maxLeaf) {  // KDTree.cpp:13-16
      out.nodes[self].leaf_start = static_cast<uint32_t>(out.refs.size());
      out.nodes[self].leaf_count = static_cast<uint32_t>(elements.size());
      out.refs.insert(out.refs.end(), elements.begin(), elements.end());
      return;
    }
    Box box{{out.nodes[self].box_min[0], out.nodes[self].box_min[1], out.nodes[self].box_min[2]},
            {out.nodes[self].box_max[0], out.nodes[self].box_max[1], out.nodes[self].box_max[2]}};
    Box b0, b1;
    split(box, depth % AXIS_COUNT, b0, b1);
    std::vector<uint32_t> e0, e1;
    e0.reserve(elements.size() / 2);
    e1.reserve(elements.size() / 2);
    for (uint32_t e : elements) {
      if (overlaps(b0, elems[e])) e0.push_back(e);
      if (overlaps(b1, elems[e])) e1.push_back(e);
    }
    std::vector<uint32_t>().swap(elements);
    if (!e0.empty()) {
      uint32_t c = static_cast<uint32_t>(out.nodes.size());
      out.nodes.push_back(makeNode(b0));
      out.nodes[self].child[0] = c;
      buildSerial(out, c, depth + 1, std::move(e0));
    }
    if (!e1.empty()) {
      uint32_t c = static_cast<uint32_t>(out.nodes.size());
      out.nodes.push_back(makeNode(b1));
      out.nodes[self].child[1] = c;
      buildSerial(out, c, depth + 1, std::move(e1));
    }
  }

  static void append(KDTreeData &dst, uint32_t parent, int which, KDTreeData &&sub) {
    const uint32_t nodeOff = static_cast<uint32_t>(dst.nodes.size());
    const uint32_t refOff = static_cast<uint32_t>(dst.refs.size());
    dst.nodes[parent].child[which] = nodeOff;
    for (crtb200_kdnode n : sub.nodes) {
      if (n.child[0] != CRTB200_INVALID) n.child[0] += nodeOff;
      if (n.child[1] != CRTB200_INVALID) n.child[1] += nodeOff;
      if (n.leaf_count) n.leaf_start += refOff;
      dst.nodes.push_back(n);
    }
    dst.refs.insert(dst.refs.end(), sub.refs.begin(), sub.refs.end());
  }

  // Subtree rooted at a node with box `box`; large shallow subtrees fork their two children.
  KDTreeData buildTask(const Box &box, unsigned depth, std::vector<uint32_t> &&elements, unsigned forkLevels) const {
    KDTreeData out;
    out.nodes.push_back(makeNode(box));
    if (forkLevels == 0 || elements.size() < 65536 || depth >= maxDepth || elements.size() <= maxLeaf) {
      buildSerial(out, 0, depth, std::move(elements));
      return out;
    }
    Box b0, b1;
    split(box, depth % AXIS_COUNT, b0, b1);
    std::vector<uint32_t> e0, e1;
    e0.reserve(elements.size() / 2);
    e1.reserve(elements.size() / 2);
    for (uint32_t e : elements) {
      if (overlaps(b0, elems[e])) e0.push_back(e);
      if (overlaps(b1, elems[e])) e1.push_back(e);
    }
    std::vector<uint32_t>().swap(elements);
    std::future<KDTreeData> f0;
    const bool has0 = !e0.empty(), has1 = !e1.empty();
    if (has0)
      f0 = std::async(std::launch::async,
                      [this, b0, depth, forkLevels](std::vector<uint32_t> e) {
                        return buildTask(b0, depth + 1, std::move(e), forkLevels - 1);
                      },
                      std::move(e0));
    KDTreeData s1;
    if (has1) s1 = buildTask(b1, depth + 1, std::move(e1), forkLevels - 1);
    if (has0) append(out, 0, 0, f0.get());
    if (has1) append(out, 0, 1, std::move(s1));
    return out;
  }
};

unsigned forkLevelsFor(unsigned threads) {
  unsigned levels = 0;
  while ((1u << levels) < threads * 2 && levels < 8) levels++;
  return threads <= 1 ? 0 : levels;
}

}  // namespace

KDTreeData buildKDTree(const std::vector<Box> &elementBoxes, const Box &rootBox, unsigned maxDepth,
                       unsigned maxElementsInLeaf, unsigned threads) {
  Builder b{elementBoxes, maxDepth, maxElementsInLeaf};
  std::vector<uint32_t> all(elementBoxes.size());
  for (size_t i = 0; i < all.size(); i++) all[i] = static_cast<uint32_t>(i);  // std::iota, AccelerationStructure.cpp:17
  return b.buildTask(rootBox, 0, std::move(all), forkLevelsFor(threads));
}

static Box emptyBox() {  // BoundingBox::initializeMinMaxPoints  BoundingBox.h:15-20
  Box b;
  for (int i = 0; i < 3; i++) {
    b.mn[i] = std::numeric_limits<float>::max();
    b.mx[i] = std::numeric_limits<float>::lowest();
  }
  return b;
}
static inline void grow(Box &b, const Vector &p) {  // std::min / std::max as written, BoundingBox.h:31-32
  const float v[3] = {p.x, p.y, p.z};
  for (int i = 0; i < 3; i++) {
    b.mn[i] = std::min(b.mn[i], v[i]);
    b.mx[i] = std::max(b.mx[i], v[i]);
  }
}

void buildFlatScene(const Scene &scene, FlatScene &out, unsigned threads, bool trees) {
  auto t0 = std::chrono::steady_clock::now();
  if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
  out = FlatScene();
  const size_t nMesh = scene.objects.size();
  out.meshes.resize(nMesh);
  bool anyUV = false;
  for (auto &m : scene.objects) anyUV = anyUV || !m.uvs.empty();

  std::vector<Box> meshBoxes(nMesh);
  Box sceneBox = emptyBox();
  uint32_t vtxBase = 0, triBase = 0;
  for (size_t mi = 0; mi < nMesh; mi++) {
    const Mesh &mesh = scene.objects[mi];
    crtb200_mesh &fm = out.meshes[mi];
    fm.material = mesh.materialIndex;
    fm.first_vertex = vtxBase;
    fm.n_vertices = static_cast<uint32_t>(mesh.positions.size());
    fm.first_triangle = triBase;
    fm.n_triangles = static_cast<uint32_t>(mesh.triangleCount());
    for (size_t v = 0; v < mesh.positions.size(); v++) {
      const Vector &p = mesh.positions[v], &n = mesh.normals[v];
      out.vertexPosition.insert(out.vertexPosition.end(), {p.x, p.y, p.z});
      out.vertexNormal.insert(out.vertexNormal.end(), {n.x, n.y, n.z});
      if (anyUV) {
        Vector uv = v < mesh.uvs.size() ? mesh.uvs[v] : Vector();
        out.vertexUV.insert(out.vertexUV.end(), {uv.x, uv.y, uv.z});
      }
    }
    // per-triangle boxes (BoundingBox(const Triangle&), BoundingBox.h:50-58) and the mesh root box
    // (BoundingBox(const std::vector<Triangle>&), BoundingBox.h:26-34: only vertices referenced by triangles)
    std::vector<Box> triBoxes(trees ? fm.n_triangles : 0);
    Box root = emptyBox();
    for (uint32_t t = 0; t < fm.n_triangles; t++) {
      Box b = emptyBox();
      for (int k = 0; k < 3; k++) {
        const uint32_t vi = mesh.indices[3 * t + k];
        if (trees) {
          grow(b, mesh.positions[vi]);
          grow(root, mesh.positions[vi]);
          grow(sceneBox, mesh.positions[vi]);
        }
        out.triangleVertex.push_back(vtxBase + vi);
      }
      if (trees) triBoxes[t] = b;
      const Vector &fn = mesh.faceNormals[t];
      out.triangleNormal.insert(out.triangleNormal.end(), {fn.x, fn.y, fn.z});
    }
    vtxBase += fm.n_vertices;
    triBase += fm.n_triangles;
    if (!trees) {  // geometry only (crtb200_upload_geometry builds the trees): tree fields 0
      fm.first_node = fm.n_nodes = fm.first_leaf_ref = fm.n_leaf_refs = 0;
      continue;
    }
    // TriangleKDTree(mesh, 25, 8)  AccelerationStructure.h:10-11
    KDTreeData tree = buildKDTree(triBoxes, root, 25, 8, threads);
    fm.first_node = static_cast<uint32_t>(out.meshNodes.size());
    fm.n_nodes = static_cast<uint32_t>(tree.nodes.size());
    fm.first_leaf_ref = static_cast<uint32_t>(out.meshLeafRefs.size());
    fm.n_leaf_refs = static_cast<uint32_t>(tree.refs.size());
    out.meshNodes.insert(out.meshNodes.end(), tree.nodes.begin(), tree.nodes.end());
    out.meshLeafRefs.insert(out.meshLeafRefs.end(), tree.refs.begin(), tree.refs.end());
    // ObjectKDTreeSubTree::getBoundingBox = tree root box  AccelerationStructure.cpp:21-23
    meshBoxes[mi] = root;
  }
  if (trees) {
    // ObjectKDTree(scene, 25, 4): root box = BoundingBox(scene)  AccelerationStructure.cpp:27-45, BoundingBox.h:36-48
    KDTreeData top = buildKDTree(meshBoxes, sceneBox, 25, 4, 1);
    out.topNodes = std::move(top.nodes);
    out.topLeafRefs = std::move(top.refs);
  }

  for (const Material &m : scene.materials) {
    crtb200_material fm;
    fm.type = static_cast<uint32_t>(m.type);
    fm.smooth_shading = m.smoothShading ? 1u : 0u;
    fm.texture = m.texture < 0 ? CRTB200_INVALID : static_cast<uint32_t>(m.texture);
    fm.albedo[0] = m.albedo.x;
    fm.albedo[1] = m.albedo.y;
    fm.albedo[2] = m.albedo.z;
    fm.ior = m.ior;
    out.materials.push_back(fm);
  }
  for (const Texture &t : scene.textures) {
    crtb200_texture ft{};
    ft.kind = static_cast<uint32_t>(t.kind);
    for (int i = 0; i < 3; i++) {
      ft.color_a[i] = t.colorA[i];
      ft.color_b[i] = t.colorB[i];
    }
    ft.scalar = t.scalar;
    ft.width = static_cast<uint32_t>(t.width);
    ft.height = static_cast<uint32_t>(t.height);
    ft.texel_offset = out.texels.size() / 3;
    for (const Color &c : t.buffer) out.texels.insert(out.texels.end(), {c.x, c.y, c.z});
    out.textures.push_back(ft);
  }
  for (const Light &l : scene.lights) {
    crtb200_light fl;
    fl.position[0] = l.position.x;
    fl.position[1] = l.position.y;
    fl.position[2] = l.position.z;
    fl.intensity = l.intensity;
    out.lights.push_back(fl);
  }

  crtb200_scene &a = out.abi;
  a.abi_version = CRTB200_ABI_VERSION;
  a.width = scene.sceneSettings.image.width;
  a.height = scene.sceneSettings.image.height;
  for (int i = 0; i < 3; i++) a.background[i] = scene.sceneSettings.sceneBackgroundColor[i];
  a.n_vertices = vtxBase;
  a.vertex_position = out.vertexPosition.data();
  a.vertex_normal = out.vertexNormal.data();
  a.vertex_uv = anyUV ? out.vertexUV.data() : nullptr;
  a.n_triangles = triBase;
  a.triangle_vertex = out.triangleVertex.data();
  a.triangle_normal = out.triangleNormal.data();
  a.n_meshes = static_cast<uint32_t>(nMesh);
  a.meshes = out.meshes.data();
  a.n_materials = static_cast<uint32_t>(out.materials.size());
  a.materials = out.materials.data();
  a.n_textures = static_cast<uint32_t>(out.textures.size());
  a.textures = out.textures.data();
  a.n_texels = out.texels.size() / 3;
  a.texels = out.texels.data();
  a.n_lights = static_cast<uint32_t>(out.lights.size());
  a.lights = out.lights.data();
  a.n_mesh_nodes = static_cast<uint32_t>(out.meshNodes.size());
  a.mesh_nodes = trees ? out.meshNodes.data() : nullptr;
  a.n_mesh_leaf_refs = static_cast<uint32_t>(out.meshLeafRefs.size());
  a.mesh_leaf_refs = trees ? out.meshLeafRefs.data() : nullptr;
  a.n_top_nodes = static_cast<uint32_t>(out.topNodes.size());
  a.top_nodes = trees ? out.topNodes.data() : nullptr;
  a.n_top_leaf_refs = static_cast<uint32_t>(out.topLeafRefs.size());
  a.top_leaf_refs = trees ? out.topLeafRefs.data() : nullptr;
  out.buildSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace crt
