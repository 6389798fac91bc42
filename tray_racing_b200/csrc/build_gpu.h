// build_gpu.h — internal interface between the C ABI (tray_cuda.cu) and the device-side builder (build_gpu.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <memory>
#include <vector>

#include "tray_cuda.h"

namespace tray {
// The fused node test needs 2^23 * scale * |1/d| finite, i.e. below 2^105 on the x axis.  Rays with |1/d| >= 2^64 on some axis
// (RayConst::wide) and scenes with an exponent byte >= EXACT_EXP_BYTE (scale >= 2^40) take the unfused test: together the two
// guards keep 2^23 * A below 2^23 * 2^39 * 2^64 = 2^126, two bits short of the overflow.  The builder and the refit report such
// nodes; scene creation scans uploaded ones.
constexpr uint32_t EXACT_EXP_BYTE = 167;
__host__ __device__ __forceinline__ bool node_needs_exact(uint32_t exp_bytes3) {    // the three exponent bytes of a node (byte 12..14)
    return (exp_bytes3 & 0xffu) >= EXACT_EXP_BYTE || ((exp_bytes3 >> 8) & 0xffu) >= EXACT_EXP_BYTE || ((exp_bytes3 >> 16) & 0xffu) >= EXACT_EXP_BYTE;
}
}  // namespace tray

namespace tray_build {

// device memory freed with cudaFree when its owner goes
struct CudaFree { void operator()(void* p) const { cudaFree(p); } };
template <typename T> using DevPtr = std::unique_ptr<T, CudaFree>;

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
// object_offsets == NULL: one flat BVH.  Otherwise a two-level build: one BLAS per object (object k = triangles
// [object_offsets[k], object_offsets[k + 1])) + a TLAS over them.
int build_tlas(const float* tris9_host, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects, uint32_t tri_stride,
               uint32_t max_prims_per_leaf, uint32_t search_radius, cudaStream_t st, Result* out, char* err, size_t errlen);

// Refit (tray_cuda_scene_refit): what a scene keeps of its trees' topology after one walk from the roots, and the boxes a refit
// passes from level to level.  Owned by the scene.
struct RefitTopology {
    DevPtr<uint2> d_items;                   // the reachable nodes as (node, tree base), level after level
    std::vector<uint32_t> level_off;         // level L = d_items[level_off[L], level_off[L + 1]); BLAS (or flat) levels first
    uint32_t n_blas_levels = 0;              // the TLAS levels follow
    DevPtr<int4> d_node_box;                 // per node: min, max as ordered ints (two int4)
    DevPtr<int4> d_slot_box;                 // per triangle slot: the same
    DevPtr<uint32_t> d_flag;
    bool unreached_exact = false;            // a node no root reaches (never rewritten) has an exponent byte >= 167
    uint64_t bytes = 0;                      // device memory held
};

// The walk: level-by-level BFS from node 0, or from the distinct blas_offsets and then tlas_start.  Returns 0, -1 (with a
// message) for a tree it cannot refit — a node reached twice, a child or leaf index outside its array, a blas_offsets entry
// outside the node array — or -2 for a CUDA error.  Synchronous on `st`.
int refit_walk(const void* d_nodes, uint64_t n_nodes, uint64_t n_tris, const uint32_t* d_blas, uint32_t n_instances, uint32_t tlas_start,
               cudaStream_t st, RefitTopology* out, char* err, size_t errlen);
// *bad = some coordinate of d_tris9 is not finite, or the vertices' extent on some axis (max - min in f32) is not: then a box
// extent could overflow and could not be encoded
int refit_check(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, cudaStream_t st, bool* bad, char* err, size_t errlen);
// Rewrites the triangle records (slot k <- d_tris9[d_prim_indices ? d_prim_indices[k] : k]) and p, exponents and used q bytes
// of every reachable node, tight over the new triangles.  *exact = some node's exponent byte is >= 167.  Synchronous on `st`.
int refit_run(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, const uint32_t* d_prim_indices, uint32_t tri_stride,
              void* d_nodes, void* d_tris, const uint32_t* d_blas, cudaStream_t st, bool* exact, char* err, size_t errlen);

}  // namespace tray_build
