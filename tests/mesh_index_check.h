// The mesh index invariants, shared by the probes of tests/test_lowering_cpu.py (the host build) and
// tests/test_gpu_mesh_index.py (the device build).  For every mesh a bspMesh primitive uses: the walk from its root reaches
// every triangle slot exactly once, each child box (FP32 and FP64) contains every double-precision vertex below it, leaves
// hold 1..max_leaf slots, and `seq` ranks the mesh's triangles in BspMesh.intersect's right-before-left order (`order`, from
// enumerateMeshes) with bvh_tri naming them.  Returns the number of triangle slots checked, or a negative code naming the
// first violation; *walk_depth = the deepest link the walk met (root = 0).
#pragma once
#include <algorithm>
#include <cfloat>
#include <functional>
#include <utility>
#include <vector>

inline long checkMeshIndex(const ftb_scene_desc* d, const ftb::Lowered& L, const std::vector<std::vector<int32_t>>& order, int max_leaf, int* walk_depth)
{
    std::vector<int> seen(L.bvh_tri.size(), 0);
    long checked = 0;
    int maxDepth = 0;
    if (L.mesh_root.size() != order.size()) return -20;
    for (size_t m = 0; m < order.size(); ++m) {
        if (!L.mesh_used[m]) continue;
        std::vector<std::pair<int32_t, int32_t>> bySeq;  // (seq, triangle)
        // returns the box of everything below `link` in double
        std::function<int(int32_t, int, double*, double*)> walk = [&](int32_t link, int depth, double* lo, double* hi) -> int {
            if (depth > maxDepth) maxDepth = depth;
            for (int k = 0; k < 3; ++k) { lo[k] = DBL_MAX; hi[k] = -DBL_MAX; }
            if (link < 0) {
                const int code = ~link, first = code >> 3, count = code & 7;
                if (count < 1 || count > max_leaf || first < 0 || (size_t)(first + count) > L.bvh_tri.size()) return -10;
                for (int s = first; s < first + count; ++s) {
                    if (seen[(size_t)s]++) return -11;
                    const int32_t tri = L.bvh_tri[(size_t)s];
                    if (tri < 0 || tri >= d->n_triangles) return -12;
                    bySeq.push_back({L.bvh_seq[(size_t)s], tri});
                    for (int v = 0; v < 3; ++v)
                        for (int k = 0; k < 3; ++k) {
                            const double x = d->triangles[9 * (size_t)tri + 3 * v + k];
                            if (x < lo[k]) lo[k] = x;
                            if (x > hi[k]) hi[k] = x;
                        }
                    ++checked;
                }
                return 0;
            }
            if ((size_t)link >= L.bvh_nodes.size()) return -13;
            const ftb::BvhNode& n = L.bvh_nodes[(size_t)link];
            for (int c = 0; c < 2; ++c) {
                double clo[3], chi[3];
                const int rc = walk(n.child[c], depth + 1, clo, chi);
                if (rc) return rc;
                for (int k = 0; k < 3; ++k) {
                    if (!((double)n.lo[c][k] <= clo[k] && (double)n.hi[c][k] >= chi[k])) return -14;  // the FP32 box must contain its subtree
                    if (!(n.dlo[c][k] <= clo[k] && n.dhi[c][k] >= chi[k])) return -15;                // and so must the FP64 one
                    if (clo[k] < lo[k]) lo[k] = clo[k];
                    if (chi[k] > hi[k]) hi[k] = chi[k];
                }
            }
            return 0;
        };
        double lo[3], hi[3];
        const int rc = walk(L.mesh_root[m], 0, lo, hi);
        if (rc) return rc;
        std::sort(bySeq.begin(), bySeq.end());
        if (bySeq.size() != order[m].size()) return -16;
        for (size_t i = 0; i < bySeq.size(); ++i)
            if (bySeq[i].first != (int32_t)i || bySeq[i].second != order[m][i]) return -17;  // seq = rank in the reference's enumeration
    }
    for (size_t s = 0; s < seen.size(); ++s) if (seen[s] != 1) return -18;
    *walk_depth = maxDepth;
    return checked;
}
