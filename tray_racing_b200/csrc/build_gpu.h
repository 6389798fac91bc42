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
template <typename T> cudaError_t dev_alloc(DevPtr<T>& p, size_t bytes) { T* q = nullptr; const cudaError_t e = cudaMalloc(&q, bytes); p.reset(q); return e; }

// pinned host memory, freed with cudaFreeHost
struct CudaFreeHost { void operator()(void* p) const { cudaFreeHost(p); } };
template <typename T> using HostPtr = std::unique_ptr<T, CudaFreeHost>;
template <typename T> cudaError_t host_alloc(HostPtr<T>& p, size_t bytes) { T* q = nullptr; const cudaError_t e = cudaMallocHost(&q, bytes); p.reset(q); return e; }

// streams (non-blocking) and events, destroyed when their owner goes
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
inline cudaError_t make_stream(Stream& s) { cudaStream_t q = nullptr; const cudaError_t e = cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking); s.reset(q); return e; }
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
using Event = std::unique_ptr<CUevent_st, EventDestroy>;
inline cudaError_t make_event(Event& ev, unsigned flags = cudaEventDefault) { cudaEvent_t q = nullptr; const cudaError_t e = cudaEventCreateWithFlags(&q, flags); ev.reset(q); return e; }

// Device memory that grows and never shrinks, for n elements of T.  A growth frees the old allocation before it makes the new
// one, so that the peak is the new size alone, and keeps no contents.  A failed growth leaves the buffer empty (cap 0): the next
// call tries again.
template <typename T> struct DevBuf {
    DevPtr<T> p;
    uint64_t cap = 0;
    T* get() const { return p.get(); }
    cudaError_t reserve(uint64_t n) {
        if (n <= cap) return cudaSuccess;
        p.reset(); cap = 0;
        const cudaError_t e = dev_alloc(p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
};

struct Result {
    DevPtr<uint8_t> d_nodes;           // n_nodes x 80 bytes (the allocation holds node_cap nodes)
    uint64_t n_nodes = 0, node_cap = 0;
    DevPtr<uint8_t> d_tris;            // n_tris x tri_stride, BVH order
    DevPtr<uint32_t> d_prim_indices;   // BVH slot -> input triangle
    DevPtr<uint32_t> d_blas_offsets;   // two-level builds: node index of the BLAS behind TLAS leaf k
    uint32_t n_instances = 0, tlas_start = 0;
    bool force_exact = false;          // some node scale >= 2^40 (see tray_scene::force_exact)
    tray_build_stats stats{};
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
    uint64_t cap = 0;                        // nodes d_items and d_node_box have room for
    DevPtr<uint32_t> d_canon;                // two-level: blas_offsets sorted, i.e. the BLAS roots of the instances in canonical order
    std::vector<uint32_t> roots;             // two-level: the distinct blas_offsets of the walk, ascending (the valid instance roots)
    DevPtr<uint32_t> d_roots;                // the same on the device
    DevPtr<uint4> d_root_nodes;              // room for their nodes (root_nodes)
    DevPtr<char> d_tlas_arena;               // device scratch of the TLAS rebuilds (refit_reserve), kept from call to call
    size_t tlas_arena_bytes = 0;
    bool unreached_exact = false;            // a node no root reaches (never rewritten) has an exponent byte >= 167
    bool unreached_exact_blas = false;       // ... one below tlas_start
    bool blas_past_tlas = false;             // a node reached from a BLAS root has an index >= tlas_start
    bool blas_empty = false;                 // some BLAS reaches no triangle
    uint64_t bytes = 0;                      // device memory held
};

// The walk: level-by-level BFS from node 0, or from the distinct blas_offsets and then tlas_start.  Returns 0, -1 (with a
// message) for a tree it cannot refit — a node reached twice, a child or leaf index outside its array, a blas_offsets entry
// outside the node array — or -2 for a CUDA error.  Synchronous on `st`.  blas_past_tlas and blas_empty are not refusals here:
// a refit takes such trees, a TLAS rebuild does not.
int refit_walk(const void* d_nodes, uint64_t n_nodes, uint64_t n_tris, const uint32_t* d_blas, uint32_t n_instances, uint32_t tlas_start,
               cudaStream_t st, RefitTopology* out, char* err, size_t errlen);
// *bad = some coordinate of d_tris9 is not finite, or the vertices' extent on some axis (max - min in f32) is not: then a box
// extent could overflow and could not be encoded
int refit_check(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, cudaStream_t st, bool* bad, char* err, size_t errlen);
// Rewrites the triangle records (slot k <- d_tris9[d_prim_indices ? d_prim_indices[k] : k]) and p, exponents and used q bytes
// of every reachable node, tight over the new triangles.  *exact = some node's exponent byte is >= 167.  Synchronous on `st`.
// blas_only: the BLAS levels alone (a TLAS rebuild follows); *exact then leaves the TLAS nodes out.
int refit_run(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, const uint32_t* d_prim_indices, uint32_t tri_stride,
              void* d_nodes, void* d_tris, const uint32_t* d_blas, bool blas_only, cudaStream_t st, bool* exact, char* err, size_t errlen);
// What a TLAS rebuild of n_instances needs before its first write: room for `cap` nodes in the topology's arrays (the listed items
// kept), and the rebuild's scratch arena (n_instances x 384 B + 16 MiB), allocated by the first call and grown by a call with more
// instances than any before it.  Synchronous on `st`.
int refit_reserve(RefitTopology& t, uint64_t cap, uint32_t n_instances, cudaStream_t st, char* err, size_t errlen);
// The TLAS of an instanced scene (tray_cuda_scene_set_instances): the boxes of instance k are h_lo[k] / h_hi[k] (host memory, xyz),
// its InstanceRecord (traverse.cuh) d_in[4k .. 4k + 3] with the instance id k.
struct InstanceTlas { const float4* h_lo; const float4* h_hi; const uint4* d_in; uint4* d_rec; };
// TLAS rebuild (tray_cuda_scene_refit_rebuild_tlas), after refit_run(blas_only): the TLAS leg of build_tlas over the BLAS root
// boxes of the n instances in canonical order, written at node tlas_start of d_nodes; d_blas[j] = the root of TLAS leaf j; the
// topology's TLAS levels become the new tree's (refit_reserve(tlas_start + n + 1) first).  `written` (optional) is recorded
// behind the last TLAS write.  *n_tlas_nodes, and *exact = some new TLAS node's exponent byte is >= 167.  Synchronous on `st`.
// With `inst`: over the instances' boxes in instance order instead; d_rec[4j ..] = the InstanceRecord of TLAS leaf j.
int rebuild_tlas(RefitTopology& t, void* d_nodes, uint32_t tlas_start, uint32_t n, uint32_t* d_blas, uint32_t max_leaf, uint32_t radius,
                 cudaStream_t st, cudaEvent_t written, uint32_t* n_tlas_nodes, bool* exact, char* err, size_t errlen,
                 const InstanceTlas* inst = nullptr);
// The first 80-byte node of each of t.roots, as 5 uint4 per root in `out`.  Synchronous on `st`.
int root_nodes(const RefitTopology& t, const void* d_nodes, cudaStream_t st, std::vector<uint4>* out, char* err, size_t errlen);
// *exact = some node below tlas_start has an exponent byte >= 167 (tray::node_needs_exact).  Synchronous on `st`.
int blas_exact(const RefitTopology& t, const void* d_nodes, uint32_t tlas_start, cudaStream_t st, bool* exact, char* err, size_t errlen);

}  // namespace tray_build
