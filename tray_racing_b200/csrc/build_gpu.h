// build_gpu.h — internal interface between the C ABI (tray_cuda.cu) and the device-side builder (build_gpu.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "tray_cuda.h"

namespace tray_build {

struct Result {
    uint8_t* d_nodes;            // n_nodes x 80 bytes (allocation holds n_tris + 1 nodes); caller owns (cudaFree)
    uint64_t n_nodes;
    uint8_t* d_tris;             // n_tris x tri_stride, BVH order; caller owns
    uint32_t* d_prim_indices;    // BVH slot -> input triangle; caller owns
    uint32_t* d_blas_offsets;    // two-level builds: node index of the BLAS behind TLAS leaf k; caller owns
    uint32_t n_instances, tlas_start;
    bool force_exact;            // some node scale >= 2^40 (see tray_scene::force_exact)
    tray_build_stats stats;
};

// Builds on the current device, synchronously with respect to `st`.  Returns 0, or a negative code with a message in `err`.
int build(const float* tris9_host, uint64_t n_tris, uint32_t tri_stride, uint32_t max_prims_per_leaf, uint32_t search_radius,
          cudaStream_t st, Result* out, char* err, size_t errlen);

// Two-level build: one BLAS per object (object k = triangles [object_offsets[k], object_offsets[k + 1])) + a TLAS over them.
int build_tlas(const float* tris9_host, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects, uint32_t tri_stride,
               uint32_t max_prims_per_leaf, uint32_t search_radius, cudaStream_t st, Result* out, char* err, size_t errlen);

// Refit (tray_cuda_scene_refit): what a scene keeps of its trees' topology after one walk from the roots, and the boxes a refit
// passes from level to level.  Owned by the scene; refit_free releases it.
struct RefitTopology {
    uint2* d_items = nullptr;                // the reachable nodes as (node, tree base), level after level
    std::vector<uint32_t> level_off;         // level L = d_items[level_off[L], level_off[L + 1]); BLAS (or flat) levels first
    uint32_t n_blas_levels = 0;              // the TLAS levels follow
    int4* d_node_box = nullptr;              // per node: min, max as ordered ints (two int4)
    int4* d_slot_box = nullptr;              // per triangle slot: the same
    uint32_t* d_flag = nullptr;
    bool unreached_exact = false;            // a node no root reaches (never rewritten) has an exponent byte >= 167
    uint64_t bytes = 0;                      // device memory held
};

// The walk: level-by-level BFS from node 0, or from the distinct blas_offsets and then tlas_start.  Returns 0, -1 (with a
// message) for a tree it cannot refit — a node reached twice, a child or leaf index outside its array, a blas_offsets entry
// outside the node array — or -2 for a CUDA error.  Synchronous on `st`.
int refit_walk(const void* d_nodes, uint64_t n_nodes, uint64_t n_tris, const uint32_t* d_blas, uint32_t n_instances, uint32_t tlas_start,
               cudaStream_t st, RefitTopology* out, char* err, size_t errlen);
void refit_free(RefitTopology* t);
// *bad = some coordinate of d_tris9 is not finite, or the vertices' extent on some axis (max - min in f32) is not: then a box
// extent could overflow and could not be encoded
int refit_check(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, cudaStream_t st, bool* bad, char* err, size_t errlen);
// Rewrites the triangle records (slot k <- d_tris9[d_prim_indices ? d_prim_indices[k] : k]) and p, exponents and used q bytes
// of every reachable node, tight over the new triangles.  *exact = some node's exponent byte is >= 167.  Synchronous on `st`.
int refit_run(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, const uint32_t* d_prim_indices, uint32_t tri_stride,
              void* d_nodes, void* d_tris, const uint32_t* d_blas, cudaStream_t st, bool* exact, char* err, size_t errlen);

}  // namespace tray_build
