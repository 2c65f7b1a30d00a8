// Host KD-tree build + flattening into the C ABI's arrays (host component H1 of SURVEY.md 2.2).
//
// The build reproduces the reference's trees NODE FOR NODE (same boxes, same numbering, same leaf contents):
//   KDTree<Triangle>::build / KDTree<ObjectKDTreeSubTree>::build   src/KDTree.cpp:10-46, 89-125
//   BoundingBox ctors / split / intersects                         include/tracer/BoundingBox.h:24-83
//   TriangleKDTree / ObjectKDTree ctors                            src/AccelerationStructure.cpp:12-50
// because under the reference's visit-all traversal the visited-node set affects results (SURVEY App. B-7).
// Unlike the reference (single-threaded, 11 s for 1 M triangles) independent subtrees are built on a thread pool
// and stitched back in the reference's DFS pre-order.
#pragma once
#include <cstdint>
#include <vector>

#include "../../../include/crtb200.h"
#include "crt_scene.hpp"

namespace crt {

struct Box {
  float mn[3], mx[3];
};

struct KDTreeData {
  std::vector<crtb200_kdnode> nodes;  // reference numbering, children relative to nodes[0]
  std::vector<uint32_t> refs;         // leaf element indices
};

// Generic builder over element boxes (triangles: their own AABB; meshes: their tree's root box).
KDTreeData buildKDTree(const std::vector<Box> &elementBoxes, const Box &rootBox, unsigned maxDepth,
                       unsigned maxElementsInLeaf, unsigned threads);

// Everything crtb200_upload_scene needs, owning the storage the crtb200_scene pointers refer to.
struct FlatScene {
  std::vector<float> vertexPosition, vertexNormal, vertexUV;
  std::vector<uint32_t> triangleVertex;
  std::vector<float> triangleNormal;
  std::vector<crtb200_mesh> meshes;
  std::vector<crtb200_material> materials;
  std::vector<crtb200_texture> textures;
  std::vector<float> texels;
  std::vector<crtb200_light> lights;
  std::vector<crtb200_kdnode> meshNodes, topNodes;
  std::vector<uint32_t> meshLeafRefs, topLeafRefs;
  crtb200_scene abi{};
  double buildSeconds = 0;
};

// AccelerationStructure(scene) + flattening.  threads = 0 -> hardware_concurrency.  trees = false: the flattened arrays
// alone (tree counts 0, tree arrays NULL, the meshes' tree fields 0), for crtb200_upload_geometry.
void buildFlatScene(const Scene &scene, FlatScene &out, unsigned threads = 0, bool trees = true);

}  // namespace crt
