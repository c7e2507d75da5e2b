// bvh_build.h — the mesh index (lower.h BvhNode) built ON THE DEVICE at ftb_scene_create time.
//
// The reference builds its BSP by lazily re-evaluated clipping (BspMesh.fs:30-65); what the render kernel needs from a
// mesh is only its (clipped) triangle set and the enumeration order (lower.h).  The index over that set is this library's
// own and is built where the triangles are going anyway: parallel locally-ordered clustering (PLOC: Morton-sort the
// triangles, then repeatedly merge every pair of clusters that are each other's nearest neighbour within a window of the
// sorted order, nearest = smallest surface area of the joint box), which gives trees close to a top-down SAH build in a
// few dozen small launches.  Subtrees of <= 4 triangles become the leaves.  The host builder (lower.cpp buildMeshIndex,
// binned SAH) stays: for small meshes, where it takes 0.2-3 ms against the device build's 2-10 ms of fixed cost and gives
// 3-9 % faster walks; and as the fallback (tree deeper than the traversal stack).
// Measured on the 355 k-triangle mesh: index in 4.9 ms of device time (host: 135 ms), frames 8 % slower than on the host's tree.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "lower.h"

namespace ftb {

struct DeviceBuildStats {
    double build_ms = 0;  // device time of the build kernels, all meshes (CUDA events)
    double total_ms = 0;  // wall time including the transfers either way
    int max_depth = 0;
};

// Builds the index of every used mesh of the scene on the current device and appends it to L (bvh_nodes, bvh_tri,
// bvh_seq, mesh_root, max_bvh_depth) in the same form lower.cpp's host builder produces.  `order[m]` = the triangles
// of mesh m in the reference's enumeration order (lower.cpp enumerateMeshes).  Returns false (L untouched) on any CUDA
// error or when a tree comes out deeper than max_depth_allowed; err says why.  radius = window of the nearest-neighbour search
// (either side, in Morton order): wider windows merge by area over longer distances, which on meshes full of clipped slivers
// gives deeper trees (window 40 on the 355 k-triangle mesh: deeper than the 64-entry stack; window 16: fine).
bool buildMeshIndexDevice(const double* triangles, int n_triangles, const std::vector<std::vector<int32_t>>& order, int max_depth_allowed, int radius, Lowered& L,
                          DeviceBuildStats& stats, std::string& err);

}  // namespace ftb
