// build_gpu.cu — device-side CWBVH builder (SURVEY.md §8 f3): triangles in, the 80-byte CwBvhNode array + BVH-ordered
// triangle records out, all resident in HBM, so that a scene can be traced without the host ever holding a BVH.
//
// The reference builds on the CPU with obvhs' `ploc_cwbvh` (src/cwbvh.rs:24-105: PLOC BVH2 -> collapse -> CWBVH; 0.95-2.9 s
// multi-threaded for its large scenes, BASELINE.md).  obvhs is an un-vendored dependency, so nothing here is derived from
// its code; the pipeline below is the published algorithm family laid out for a GPU:
//   1. per-triangle boxes + scene bounds                              (one pass, atomics on ordered ints)
//   2. 63-bit Morton codes of the box centres, radix sort              (cub::DeviceRadixSort — library code, like the
//                                                                        prefix sums; the builder is not the hot path)
//   3. PLOC (Meister & Bittner 2018): every cluster looks `radius` neighbours left and right in Morton order for the
//      partner with the smallest merged surface area; mutual pairs merge; compaction by prefix sum; repeat until one
//      cluster is left.  radius defaults to 14 = obvhs' `search_distance` default (src/main.rs:563-587).
//   4. collapse to 8-wide, level by level: a wide node starts from a BVH2 node's two children and keeps opening the
//      largest-area subtree that must stay inner (> max_prims_per_leaf) until it has 8 children, then spends free
//      slots on splitting small subtrees into tighter leaves; children are placed in slots by octant
//      (embree/src/bvh_embree.rs:284-349) and encoded exactly as the in-tree encoder does
//      (embree/src/bvh_embree_to_cwbvh.rs:85-186: p / exponent / floor-ceil quantisation / child_meta).
//      Node and primitive indices come from prefix sums, not atomics: the same triangles give the same bytes on every
//      GPU, so N ranks that each build their replica agree on every primitive id.
// Same collapse rule, slot assignment and encoder as the host producer in host/cwbvh_build.cpp; only the BVH2 differs
// (PLOC here, binned SAH there).
#include <cub/cub.cuh>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <utility>

#include "build_gpu.h"
#include "host_copy.h"

namespace tray_build {

namespace {

#define BCU(call)                                                                                                  \
    do {                                                                                                           \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess) {                                                                                   \
            snprintf(err, errlen, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);     \
            cudaGetLastError();                                                                                    \
            return -2;                                                                                             \
        }                                                                                                          \
    } while (0)

constexpr int TPB = 256;
inline unsigned blocks(uint64_t n) { return (unsigned)((n + TPB - 1) / TPB); }

// ---- sign of zero ----------------------------------------------------------------------------------------------
// fminf / fmaxf (min.f32 / max.f32) order -0.0 below +0.0 whatever the argument order, and so do the ordered-int atomics of
// the scene bounds: every box corner that is zero is -0.0 when some primitive below it has -0.0 there (minimum) and +0.0 when
// some has +0.0 (maximum).  A node's p is therefore its primitives' minimum bit for bit.  oracle/build_ref.c states the same
// rule, and the host producer (host/cwbvh_build.cpp) follows it.

// ---- ordered-int float atomics ------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int f2o(float f) { int i; memcpy(&i, &f, 4); return i >= 0 ? i : i ^ 0x7fffffff; }
__host__ __device__ __forceinline__ float o2f(int i) { i = i >= 0 ? i : i ^ 0x7fffffff; float f; memcpy(&f, &i, 4); return f; }
// bounds before the first box: minima +max, maxima -max (ordered)
constexpr int EMPTY_BOUNDS[6] = { 0x7f7fffff, 0x7f7fffff, 0x7f7fffff, (int)0x80800000, (int)0x80800000, (int)0x80800000 };

// the warp's minimum of mn and maximum of mx per axis, merged into lo[0..2] / hi[0..2] by one ordered-int atomic per warp
__device__ __forceinline__ void warp_bounds(const float mn[3], const float mx[3], int* lo, int* hi) {
#pragma unroll
    for (int a = 0; a < 3; a++) {
        float l = mn[a], h = mx[a];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { l = fminf(l, __shfl_xor_sync(0xffffffffu, l, o)); h = fmaxf(h, __shfl_xor_sync(0xffffffffu, h, o)); }
        if ((threadIdx.x & 31) == 0) { atomicMin(lo + a, f2o(l)); atomicMax(hi + a, f2o(h)); }
    }
}

__device__ __forceinline__ void tri_box(const float* t, float mn[3], float mx[3]) {
#pragma unroll
    for (int a = 0; a < 3; a++) { mn[a] = fminf(t[a], fminf(t[3 + a], t[6 + a])); mx[a] = fmaxf(t[a], fmaxf(t[3 + a], t[6 + a])); }
}

// BVH2 node: lo = (min.xyz, left), hi = (max.xyz, right).  Leaf i (< n_prims): left = -1, right = primitive index.
struct Bvh2 {
    float4* lo; float4* hi; uint32_t* count;
};
__device__ __forceinline__ int node_left(const float4& lo) { return __float_as_int(lo.w); }
__device__ __forceinline__ int node_right(const float4& hi) { return __float_as_int(hi.w); }
__device__ __forceinline__ float half_area(const float4& lo, const float4& hi) {
    const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}
__device__ __forceinline__ float union_area(const float4& alo, const float4& ahi, const float4& blo, const float4& bhi) {
    const float dx = fmaxf(ahi.x, bhi.x) - fminf(alo.x, blo.x), dy = fmaxf(ahi.y, bhi.y) - fminf(alo.y, blo.y), dz = fmaxf(ahi.z, bhi.z) - fminf(alo.z, blo.z);
    return dx * dy + dy * dz + dz * dx;
}
// inner node `id` over children l and r with boxes (alo, ahi), (blo, bhi): the union of the boxes, the children in w
__device__ __forceinline__ void write_union(const Bvh2& b, int id, int l, int r, const float4& alo, const float4& ahi, const float4& blo,
                                            const float4& bhi) {
    b.lo[id] = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), __int_as_float(l));
    b.hi[id] = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), __int_as_float(r));
}

// ---- 1. boxes and scene bounds -----------------------------------------------------------------------------------
__global__ void tri_boxes_kernel(const float* __restrict__ tris9, uint32_t n, float4* __restrict__ plo, float4* __restrict__ phi) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float mn[3], mx[3];
    tri_box(tris9 + 9ull * i, mn, mx);
    plo[i] = make_float4(mn[0], mn[1], mn[2], 0.f);
    phi[i] = make_float4(mx[0], mx[1], mx[2], 0.f);
}

__global__ void box_bounds_kernel(const float4* __restrict__ plo, const float4* __restrict__ phi, uint32_t n, int* __restrict__ scene) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float mn[3] = { 3.4e38f, 3.4e38f, 3.4e38f }, mx[3] = { -3.4e38f, -3.4e38f, -3.4e38f };
    if (i < n) {
        const float4 lo = plo[i], hi = phi[i];
        mn[0] = lo.x; mn[1] = lo.y; mn[2] = lo.z; mx[0] = hi.x; mx[1] = hi.y; mx[2] = hi.z;
    }
    warp_bounds(mn, mx, scene, scene + 3);
}

__device__ __forceinline__ unsigned long long spread21(unsigned long long v) {
    v &= 0x1fffffull;
    v = (v | (v << 32)) & 0x1f00000000ffffull;
    v = (v | (v << 16)) & 0x1f0000ff0000ffull;
    v = (v | (v << 8)) & 0x100f00f00f00f00full;
    v = (v | (v << 4)) & 0x10c30c30c30c30c3ull;
    v = (v | (v << 2)) & 0x1249249249249249ull;
    return v;
}

// `prim_seg` (optional): segment (object) of every primitive; it becomes the top 21 bits of the key (42-bit Morton code
// below it), so that a sort groups every object's primitives and PLOC can be kept from merging across objects
__global__ void morton_kernel(const float4* __restrict__ plo, const float4* __restrict__ phi, uint32_t n, const int* __restrict__ scene,
                              const uint32_t* __restrict__ prim_seg, unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 lo = plo[i], hi = phi[i];
    const float c[3] = { 0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z) };
    unsigned long long q[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const float s0 = o2f(scene[a]), s1 = o2f(scene[3 + a]);
        const float ext = s1 - s0;
        float u = ext > 0.f ? (c[a] - s0) / ext : 0.f;
        u = fminf(fmaxf(u, 0.f), 1.f);
        q[a] = (unsigned long long)fminf(u * 2097152.f, 2097151.f);
    }
    unsigned long long key = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    if (prim_seg) key = ((unsigned long long)prim_seg[i] << 42) | (key >> 21);
    keys[i] = key;
    vals[i] = i;
}

__global__ void leaf_init_kernel(const float4* __restrict__ plo, const float4* __restrict__ phi, const uint32_t* __restrict__ sorted_prim, uint32_t n,
                                 const uint32_t* __restrict__ prim_seg, uint32_t* __restrict__ node_seg, Bvh2 b, int* __restrict__ cluster) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = sorted_prim[i];
    float4 lo = plo[p], hi = phi[p];
    lo.w = __int_as_float(-1); hi.w = __int_as_float((int)p);
    b.lo[i] = lo; b.hi[i] = hi; b.count[i] = 1u;
    if (node_seg) node_seg[i] = prim_seg[p];
    cluster[i] = (int)i;
}

// ---- 3. PLOC ----------------------------------------------------------------------------------------------------
// One step, run by the multi-kernel loop and by ploc_tail_kernel alike: nearest neighbours, keep / lead flags, parents.
// nearest neighbour of position i among positions [i - r, i + r] (box(j, lo, hi) and seg(j) read position j): smallest half-area
// of the merged box, ties to the lower position (so that "mutual" is well defined and the build is deterministic)
template <typename Box, typename Seg>
__device__ __forceinline__ int ploc_nearest(int i, uint32_t m, int r, Box box, Seg seg) {
    float4 lo, hi, l2, h2;
    box(i, lo, hi);
    const uint32_t s = seg(i);
    float best = 3.4e38f; int best_j = -1;
    const int j0 = max(0, i - r), j1 = min((int)m - 1, i + r);
    for (int j = j0; j <= j1; j++) {
        if (j == i || seg(j) != s) continue;          // clusters of different objects never merge
        box(j, l2, h2);
        const float a = union_area(lo, hi, l2, h2);
        if (a < best) { best = a; best_j = j; }
    }
    return best_j;
}
__device__ __forceinline__ void ploc_flags(const int* nn, uint32_t i, uint32_t& keep, uint32_t& lead) {
    const int j = nn[i];
    const bool mutual = j >= 0 && nn[j] == (int)i;
    keep = (mutual && (int)i > j) ? 0u : 1u;          // the higher position of a merged pair disappears
    lead = (mutual && (int)i < j) ? 1u : 0u;          // the lower one creates the parent
}
// node `id` over clusters l and r (boxes (alo, ahi), (blo, bhi)); its segment, when there are segments, is that of l: seg[k]
__device__ __forceinline__ void ploc_parent(const Bvh2& b, uint32_t* node_seg, int id, int l, int r, const float4& alo, const float4& ahi,
                                            const float4& blo, const float4& bhi, const uint32_t* seg, int k) {
    write_union(b, id, l, r, alo, ahi, blo, bhi);
    b.count[id] = b.count[l] + b.count[r];
    if (node_seg) node_seg[id] = seg[k];
}

__global__ void __launch_bounds__(TPB) ploc_nn_kernel(const int* __restrict__ cluster, uint32_t m, int r, Bvh2 b, const uint32_t* __restrict__ node_seg,
                                                      int* __restrict__ nn) {
    extern __shared__ float4 s_box[];                 // [(TPB + 2r) x 2] boxes, then [(TPB + 2r)] segments
    const int base = (int)(blockIdx.x * TPB) - r;
    const int span = TPB + 2 * r;
    uint32_t* s_seg = reinterpret_cast<uint32_t*>(s_box + 2 * span);
    for (int k = threadIdx.x; k < span; k += TPB) {
        const int pos = base + k;
        if (pos >= 0 && pos < (int)m) {
            const int c = cluster[pos]; s_box[2 * k] = b.lo[c]; s_box[2 * k + 1] = b.hi[c];
            s_seg[k] = node_seg ? node_seg[c] : 0u;
        }
    }
    __syncthreads();
    const int i = (int)(blockIdx.x * TPB + threadIdx.x);
    if (i >= (int)m) return;
    nn[i] = ploc_nearest(i, m, r, [&](int j, float4& lo, float4& hi) { lo = s_box[2 * (j - base)]; hi = s_box[2 * (j - base) + 1]; },
                         [&](int j) { return s_seg[j - base]; });
}

__global__ void ploc_flag_kernel(const int* __restrict__ nn, uint32_t m, uint32_t* __restrict__ keep, uint32_t* __restrict__ lead) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    uint32_t k, l;
    ploc_flags(nn, i, k, l);
    keep[i] = k; lead[i] = l;
}

__global__ void ploc_merge_kernel(const int* __restrict__ cluster, const int* __restrict__ nn, uint32_t m, const uint32_t* __restrict__ keep,
                                  const uint32_t* __restrict__ keep_pos, const uint32_t* __restrict__ lead, const uint32_t* __restrict__ lead_pos,
                                  uint32_t next_node, Bvh2 b, uint32_t* __restrict__ node_seg, int* __restrict__ cluster_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m || !keep[i]) return;
    int c = cluster[i];
    if (lead[i]) {
        const int l = c, rgt = cluster[nn[i]];
        const float4 a0 = b.lo[l], a1 = b.hi[l], b0 = b.lo[rgt], b1 = b.hi[rgt];
        const int id = (int)(next_node + lead_pos[i]);
        ploc_parent(b, node_seg, id, l, rgt, a0, a1, b0, b1, node_seg, l);
        c = id;
    }
    cluster_out[keep_pos[i]] = c;
}

// The last iterations of a PLOC run work on a handful of clusters each and are pure launch + synchronisation latency
// (68 iterations for 2.88 M triangles, ~55 of them below a thousand clusters).  Once m <= PLOC_TAIL they all run in ONE block:
// the same step, the same prefix-sum numbering of clusters and new nodes as the three kernels above, so the BVH2 is the one
// the multi-kernel loop would have produced.
constexpr int PLOC_TAIL = 1024;
struct PlocTailOut { uint32_t m, next_node, iters, stalled; };

__global__ void __launch_bounds__(PLOC_TAIL) ploc_tail_kernel(int* __restrict__ cluster, uint32_t m, int r, Bvh2 b, uint32_t* __restrict__ node_seg,
                                                              uint32_t next_node, PlocTailOut* __restrict__ out) {
    __shared__ float s_b[6][PLOC_TAIL];                       // min.xyz, max.xyz per cluster position
    __shared__ uint32_t s_seg[PLOC_TAIL];
    __shared__ int s_nn[PLOC_TAIL], s_cl[PLOC_TAIL], s_cl2[PLOC_TAIL];
    __shared__ uint32_t s_tot[2];
    typedef cub::BlockScan<uint32_t, PLOC_TAIL> Scan;
    __shared__ typename Scan::TempStorage s_scan;
    const auto box = [&](int j, float4& lo, float4& hi) {
        lo = make_float4(s_b[0][j], s_b[1][j], s_b[2][j], 0.f); hi = make_float4(s_b[3][j], s_b[4][j], s_b[5][j], 0.f);
    };
    const int i = (int)threadIdx.x;
    if (i < (int)m) s_cl[i] = cluster[i];
    __syncthreads();
    uint32_t iters = 0, stalled = 0;
    while (m > 1) {
        if (i < (int)m) {
            const int c = s_cl[i]; const float4 lo = b.lo[c], hi = b.hi[c];
            s_b[0][i] = lo.x; s_b[1][i] = lo.y; s_b[2][i] = lo.z; s_b[3][i] = hi.x; s_b[4][i] = hi.y; s_b[5][i] = hi.z;
            s_seg[i] = node_seg ? node_seg[c] : 0u;
        }
        __syncthreads();
        if (i < (int)m) s_nn[i] = ploc_nearest(i, m, r, box, [&](int j) { return s_seg[j]; });
        __syncthreads();
        uint32_t keep = 0, lead = 0;
        if (i < (int)m) ploc_flags(s_nn, (uint32_t)i, keep, lead);
        uint32_t keep_pos, lead_pos, tot_keep, tot_lead;
        Scan(s_scan).ExclusiveSum(keep, keep_pos, tot_keep);
        __syncthreads();
        Scan(s_scan).ExclusiveSum(lead, lead_pos, tot_lead);
        if (i < (int)m && keep) {
            int c = s_cl[i];
            if (lead) {
                const int j = s_nn[i];
                const int id = (int)(next_node + lead_pos);
                float4 alo, ahi, blo, bhi;
                box(i, alo, ahi); box(j, blo, bhi);
                ploc_parent(b, node_seg, id, c, s_cl[j], alo, ahi, blo, bhi, s_seg, i);
                c = id;
            }
            s_cl2[keep_pos] = c;
        }
        if (i == 0) { s_tot[0] = tot_keep; s_tot[1] = tot_lead; }
        __syncthreads();
        if (s_tot[1] == 0u) { stalled = 1; break; }           // no mutual pair left: every segment is down to one cluster (or an error, flat)
        next_node += s_tot[1]; m = s_tot[0]; iters++;
        if (i < (int)m) s_cl[i] = s_cl2[i];
        __syncthreads();
    }
    if (i < (int)m) cluster[i] = s_cl[i];
    if (i == 0) { out->m = m; out->next_node = next_node; out->iters = iters; out->stalled = stalled; }
}

// ---- 3b. reinsertion: BVH2 optimisation between PLOC and the collapse --------------------------------------------------
// obvhs runs a reinsertion pass over its PLOC tree before it collapses it (`reinsertion_batch_ratio`, `post_collapse_reinsertion`,
// reference src/main.rs:563-587); PLOC alone is greedy and pairs e.g. crossing ribbons of the hairball-like scene, which costs
// ~17 % more node visits per ray than the host's binned-SAH tree.  This is the published parallel formulation (Meister & Bittner,
// "Parallel Reinsertion for Bounding Volume Hierarchy Optimization", 2018) laid out on this builder's arrays:
//   find   every node v looks for the position x that lowers the tree's SAH cost (sum of inner-node areas) most if the subtree of
//          v is cut out and re-inserted as the sibling of x: it climbs from its parent to the root and searches the subtree on the
//          other side of every ancestor with branch and bound (the induced growth of the boxes on the way down is the bound)
//   lock   the moves are ordered by (gain, node): each claims the six nodes it rewires with atomicMax; a move that still owns all
//          six wins, unless its target sits inside the subtree a higher-ranked winner moves (that could close a cycle)
//   apply  the winners rewire their pointers concurrently
//   refit  boxes and primitive counts bottom-up
// All of it is deterministic (the lock key is a total order), so replicas built on different GPUs still agree byte for byte.
struct OptArrays { int* parent; float* gain; int* target; unsigned long long* lock; uint32_t* visits; uint8_t* win; };

__global__ void opt_parent_kernel(Bvh2 b, uint32_t first_inner, uint32_t n_nodes, int* __restrict__ parent) {
    const uint32_t i = first_inner + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    parent[node_left(b.lo[i])] = (int)i; parent[node_right(b.hi[i])] = (int)i;
}

__device__ __forceinline__ int sibling_of(const Bvh2& b, const int* parent, int x) {
    const int p = parent[x];
    const int l = node_left(b.lo[p]);
    return l == x ? node_right(b.hi[p]) : l;
}

__global__ void __launch_bounds__(128) opt_find_kernel(Bvh2 b, uint32_t n_nodes, OptArrays o, uint32_t max_visits) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    o.gain[v] = 0.f; o.target[v] = -1;
    const int p = o.parent[v];
    if (p < 0 || o.parent[p] < 0) return;                   // the root and its children stay where they are
    const float4 Llo = b.lo[v], Lhi = b.hi[v];
    const float aL = half_area(Llo, Lhi);
    float best = 0.f; int best_x = -1;
    float d = half_area(b.lo[p], b.hi[p]);                  // removing v deletes its parent
    const int s = sibling_of(b, o.parent, (int)v);
    float4 pblo = b.lo[s], pbhi = b.hi[s];                  // box of the path node once v is gone
    int pivot = p, region = s;
    bool skip_root_of_region = true;                        // re-inserting next to the own sibling is the identity
    uint32_t visits = 0;
    int stack_n[48]; float stack_c[48];
    for (;;) {
        // ---- branch and bound over the subtree `region`: cost of inserting at x = area(x U v) + induced growth on the way down
        int sp = 0; stack_n[sp] = region; stack_c[sp] = 0.f; sp++;
        while (sp && visits < max_visits) {
            sp--; const int x = stack_n[sp]; const float cind = stack_c[sp];
            visits++;
            const float4 xlo = b.lo[x], xhi = b.hi[x];
            const float m = union_area(xlo, xhi, Llo, Lhi);
            if (!(skip_root_of_region && x == region)) {
                const float g = d - (cind + m);
                if (g > best) { best = g; best_x = x; }
            }
            const int xl = node_left(xlo);
            if (xl >= 0) {
                const float cchild = cind + m - half_area(xlo, xhi);
                if (d - (cchild + aL) > best && sp + 2 <= 48) {          // a descendant could still beat the best
                    stack_n[sp] = node_right(xhi); stack_c[sp] = cchild; sp++;
                    stack_n[sp] = xl; stack_c[sp] = cchild; sp++;
                }
            }
        }
        skip_root_of_region = false;
        // ---- climb: the pivot becomes a node between the new common ancestor and v's old place
        const int up = o.parent[pivot];
        if (up < 0 || visits >= max_visits) break;
        if (pivot != p) d += half_area(b.lo[pivot], b.hi[pivot]) - half_area(pblo, pbhi);
        region = sibling_of(b, o.parent, pivot);
        const float4 rlo = b.lo[region], rhi = b.hi[region];
        // (the search of `region` uses the d of the new pivot `up`: nodes strictly between up and p have shrunk)
        pivot = up;
        // run the region search first (next loop iteration), then the path node itself; to keep one loop, handle the path node here
        // with the box it will have: pb' = pb U region
        float4 nlo = make_float4(fminf(pblo.x, rlo.x), fminf(pblo.y, rlo.y), fminf(pblo.z, rlo.z), 0.f);
        float4 nhi = make_float4(fmaxf(pbhi.x, rhi.x), fmaxf(pbhi.y, rhi.y), fmaxf(pbhi.z, rhi.z), 0.f);
        if (o.parent[pivot] >= 0) {                         // insert above the path node `pivot` (never above the root)
            const float g = d - half_area(nlo, nhi);
            if (g > best) { best = g; best_x = pivot; }
        }
        pblo = nlo; pbhi = nhi;
    }
    if (o.visits) o.visits[v] = visits;
    if (best_x >= 0 && best > aL * 1e-6f) { o.gain[v] = best; o.target[v] = best_x; }
}

// The six nodes a move rewires: v (parent), its parent p (children, parent), its sibling s (parent), its grandparent g (child), the
// target x (parent) and x's parent q (child).  Moves are ordered by key = (gain, v): each claims its six nodes with atomicMax, and
// a move that still owns all six after everybody has claimed is a winner of the pass.
template <typename F>
__device__ __forceinline__ void opt_six(const Bvh2& b, const int* parent, int v, int x, F f) {
    const int p = parent[v];
    f(v); f(p); f(sibling_of(b, parent, v)); f(parent[p]); f(x);
    if (parent[x] >= 0) f(parent[x]);
}
__device__ __forceinline__ unsigned long long opt_key(const OptArrays& o, uint32_t v) {
    return ((unsigned long long)__float_as_uint(o.gain[v]) << 32) | v;
}

// `dirty` marks the nodes earlier rounds of this pass have rewired: a move found before those rounds is still a valid move as
// long as none of its six nodes is dirty and its target has not ended up inside the subtree it moves (re-checked by a walk up).
__global__ void opt_lock_kernel(Bvh2 b, uint32_t n_nodes, OptArrays o, const uint8_t* __restrict__ dirty, int round) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes || o.target[v] < 0) return;
    if (round > 0) {
        bool stale = false;
        opt_six(b, o.parent, (int)v, o.target[v], [&](int y) { if (dirty[y]) stale = true; });
        int guard = 0;
        for (int a = o.target[v]; a >= 0 && guard < (1 << 20) && !stale; a = o.parent[a], guard++) if ((uint32_t)a == v) stale = true;
        if (stale || o.parent[o.parent[v]] < 0) { o.target[v] = -1; return; }
    }
    const unsigned long long key = opt_key(o, v);
    opt_six(b, o.parent, (int)v, o.target[v], [&](int y) { atomicMax(o.lock + y, key); });
}

__global__ void opt_check_kernel(Bvh2 b, uint32_t n_nodes, OptArrays o) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes || o.target[v] < 0) return;
    const unsigned long long key = opt_key(o, v);
    bool mine = true;
    opt_six(b, o.parent, (int)v, o.target[v], [&](int y) { if (o.lock[y] != key) mine = false; });
    o.win[v] = mine ? 1 : 0;
}

// Disjoint pointer sets are not enough: if A's target lies inside the subtree B moves and B's target inside the subtree A moves,
// applying both ties the two subtrees into a cycle.  A winner whose target has a HIGHER-keyed winner's moving node among its
// ancestors steps back for this pass; around any would-be cycle at least one edge points to a higher key, so no cycle survives.
__global__ void opt_cycle_kernel(uint32_t n_nodes, OptArrays o, uint8_t* __restrict__ drop) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    drop[v] = 0;
    if (o.target[v] < 0 || !o.win[v]) return;
    const unsigned long long key = opt_key(o, v);
    int guard = 0;
    for (int a = o.target[v]; a >= 0 && guard < (1 << 20); a = o.parent[a], guard++)
        if ((uint32_t)a != v && o.target[a] >= 0 && o.win[a] && opt_key(o, (uint32_t)a) > key) { drop[v] = 1; return; }
}

// winners own disjoint sets of nodes, so they rewire concurrently
__global__ void opt_apply_kernel(Bvh2 b, uint32_t n_nodes, OptArrays o, const uint8_t* __restrict__ drop, uint8_t* __restrict__ dirty,
                                 uint32_t* __restrict__ n_applied) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes || o.target[v] < 0 || !o.win[v] || drop[v]) return;
    opt_six(b, o.parent, (int)v, o.target[v], [&](int y) { dirty[y] = 1; });
    const int x = o.target[v];
    const int s = sibling_of(b, o.parent, (int)v);
    const int p = o.parent[v], g = o.parent[p];
    // cut: s takes p's place under g
    if (node_left(b.lo[g]) == p) b.lo[g].w = __int_as_float(s); else b.hi[g].w = __int_as_float(s);
    o.parent[s] = g;
    // paste: p becomes the parent of (x, v) where x was (x's parent read AFTER the cut: it may be g)
    const int q = o.parent[x];
    if (node_left(b.lo[q]) == x) b.lo[q].w = __int_as_float(p); else b.hi[q].w = __int_as_float(p);
    o.parent[p] = q;
    b.lo[p].w = __int_as_float(x); b.hi[p].w = __int_as_float((int)v);
    o.parent[x] = p;
    o.target[v] = -1;                                       // done for this pass
    atomicAdd(n_applied, 1u);
}

// boxes and primitive counts bottom-up: the second thread to reach a node computes it (the first leaves)
__global__ void opt_refit_kernel(Bvh2 b, uint32_t n_leaves, const int* __restrict__ parent, uint32_t* __restrict__ arrived) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_leaves) return;
    int x = parent[i];
    while (x >= 0) {
        __threadfence();
        if (atomicAdd(arrived + x, 1u) == 0u) return;
        const int l = node_left(b.lo[x]), r = node_right(b.hi[x]);
        const volatile float4* vlo = b.lo; const volatile float4* vhi = b.hi;
        const float lx0 = vlo[l].x, ly0 = vlo[l].y, lz0 = vlo[l].z, lx1 = vhi[l].x, ly1 = vhi[l].y, lz1 = vhi[l].z;
        const float rx0 = vlo[r].x, ry0 = vlo[r].y, rz0 = vlo[r].z, rx1 = vhi[r].x, ry1 = vhi[r].y, rz1 = vhi[r].z;
        write_union(b, x, l, r, make_float4(lx0, ly0, lz0, 0.f), make_float4(lx1, ly1, lz1, 0.f), make_float4(rx0, ry0, rz0, 0.f),
                    make_float4(rx1, ry1, rz1, 0.f));
        b.count[x] = ((volatile uint32_t*)b.count)[l] + ((volatile uint32_t*)b.count)[r];
        x = parent[x];
    }
}

__global__ void opt_cost_kernel(Bvh2 b, uint32_t first_inner, uint32_t n_nodes, double* __restrict__ cost) {
    const uint32_t i = first_inner + blockIdx.x * blockDim.x + threadIdx.x;
    float a = i < n_nodes ? half_area(b.lo[i], b.hi[i]) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0 && a != 0.f) atomicAdd(cost, (double)a);
}

// ---- 4. collapse to 8-wide ------------------------------------------------------------------------------------------
struct Kids { int id[8]; int n; };

// children of the wide node that replaces BVH2 subtree `root` (same rule as Collapser::run in host/cwbvh_build.cpp)
__device__ void gather_kids(const Bvh2& b, int root, uint32_t max_leaf, Kids& k) {
    const float4 rlo = b.lo[root], rhi = b.hi[root];
    k.n = 0;
    if (b.count[root] <= max_leaf || node_left(rlo) < 0) { k.id[k.n++] = root; }
    else { k.id[k.n++] = node_left(rlo); k.id[k.n++] = node_right(rhi); }
    for (int phase = 0; phase < 2; phase++) {
        while (k.n < 8) {
            int best = -1; float best_a = -1.f;
            for (int i = 0; i < k.n; i++) {
                const int c = k.id[i];
                const float4 lo = b.lo[c];
                if (node_left(lo) < 0) continue;                      // a single primitive cannot be opened
                const uint32_t cnt = b.count[c];
                const bool big = cnt > max_leaf;
                if ((phase == 0) != big) continue;
                const float a = half_area(lo, b.hi[c]) * (phase == 0 ? 1.f : (float)cnt);
                if (a > best_a) { best_a = a; best = i; }
            }
            if (best < 0) break;
            const int c = k.id[best];
            k.id[best] = node_left(b.lo[c]); k.id[k.n++] = node_right(b.hi[c]);
        }
    }
}

__global__ void collapse_count_kernel(const int* __restrict__ items, uint32_t n_items, Bvh2 b, uint32_t max_leaf,
                                      uint32_t* __restrict__ n_inner, uint32_t* __restrict__ n_tris) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    Kids k; gather_kids(b, items[i], max_leaf, k);
    uint32_t ni = 0, nt = 0;
    for (int c = 0; c < k.n; c++) {
        const uint32_t cnt = b.count[k.id[c]];
        if (cnt > max_leaf) ni++; else nt += cnt;
    }
    n_inner[i] = ni; n_tris[i] = nt;
}

// smallest power of two 2^k with 255 * 2^k >= extent (bvh_embree_to_cwbvh.rs:97-110)
__device__ int quant_exponent(float extent) {
    extent = fmaxf(extent, 1e-20f);
    int k = (int)ceil(log2((double)extent / 255.0));
    while (ldexp(255.0, k) < (double)extent) k++;
    while (ldexp(255.0, k - 1) >= (double)extent) k--;
    return k;
}

// The encoder (bvh_embree_to_cwbvh.rs:85-186), shared by the collapse and the refit: over the node box [nmn, nmx], p = its
// minimum and one power-of-two scale per axis, then the floor / ceil q bytes (in double, clamped to 0 .. 255) of every slot in
// `used`, whose box child_box(s, cmn, cmx) gives.  Writes nothing else of the node.  Returns whether some scale is >= 2^40
// (exponent byte >= tray::EXACT_EXP_BYTE: the traversal must use its unfused node test).
template <typename ChildBox>
__device__ __forceinline__ bool encode_bounds(uint32_t w[20], const float nmn[3], const float nmx[3], uint32_t used, ChildBox child_box) {
    uint8_t* nb = reinterpret_cast<uint8_t*>(w);
    double scale[3];
    bool exact = false;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        w[a] = __float_as_uint(nmn[a]);
        const int ke = quant_exponent(nmx[a] - nmn[a]);
        nb[12 + a] = (uint8_t)(ke + 127);
        exact |= ke + 127 >= (int)tray::EXACT_EXP_BYTE;
        scale[a] = ldexp(1.0, ke);
    }
#pragma unroll
    for (int s = 0; s < 8; s++) {
        if (!((used >> s) & 1u)) continue;
        float cmn[3], cmx[3];
        child_box(s, cmn, cmx);
#pragma unroll
        for (int a = 0; a < 3; a++) {
            double ql = floor(((double)cmn[a] - (double)nmn[a]) / scale[a]);
            double qh = ceil(((double)cmx[a] - (double)nmn[a]) / scale[a]);
            ql = fmin(255.0, fmax(0.0, ql)); qh = fmin(255.0, fmax(0.0, qh));
            nb[32 + 16 * a + s] = (uint8_t)ql; nb[40 + 16 * a + s] = (uint8_t)qh;
        }
    }
    return exact;
}

template <int STRIDE>
__device__ void write_tri_record(const float* __restrict__ tris9, uint32_t prim, uint8_t* __restrict__ out, uint64_t slot) {
    const float* t = tris9 + 9ull * prim;
    float v0[3] = { t[0], t[1], t[2] }, e1[3], e2[3];
#pragma unroll
    for (int a = 0; a < 3; a++) { e1[a] = __fsub_rn(t[a], t[3 + a]); e2[a] = __fsub_rn(t[6 + a], t[a]); }
    if (STRIDE == 24) {
        // RtCompressedTriangle (src/rt_gpu/mod.rs:39-43): v0 f32 x 3, e[k] = half(v2 - v0) | half(v1 - v0) << 16
        uint32_t* rec = reinterpret_cast<uint32_t*>(out + slot * 24ull);
#pragma unroll
        for (int a = 0; a < 3; a++) {
            rec[a] = __float_as_uint(v0[a]);
            rec[3 + a] = (uint32_t)__half_as_ushort(__float2half_rn(e2[a])) | ((uint32_t)__half_as_ushort(__float2half_rn(__fsub_rn(t[3 + a], t[a]))) << 16);
        }
    } else {
        float4* rec = reinterpret_cast<float4*>(out + slot * (uint64_t)STRIDE);
        rec[0] = make_float4(v0[0], v0[1], v0[2], 0.f);
        rec[1] = make_float4(e1[0], e1[1], e1[2], 0.f);
        rec[2] = make_float4(e2[0], e2[1], e2[2], 0.f);
        if (STRIDE == 64)     // ng = cross(e1, e2): mul, mul, sub, each rounded
            rec[3] = make_float4(__fsub_rn(__fmul_rn(e1[1], e2[2]), __fmul_rn(e1[2], e2[1])), __fsub_rn(__fmul_rn(e1[2], e2[0]), __fmul_rn(e1[0], e2[2])),
                                 __fsub_rn(__fmul_rn(e1[0], e2[1]), __fmul_rn(e1[1], e2[0])), 0.f);
    }
}

template <int STRIDE>
__global__ void collapse_emit_kernel(const int* __restrict__ items, uint32_t n_items, Bvh2 b, uint32_t max_leaf,
                                     const uint32_t* __restrict__ inner_off, const uint32_t* __restrict__ tri_off,
                                     uint32_t level_base, uint32_t next_base, uint32_t prim_base,
                                     const float* __restrict__ tris9, uint8_t* __restrict__ nodes, uint8_t* __restrict__ tri_out,
                                     uint32_t* __restrict__ prim_indices, int* __restrict__ items_next, uint32_t* __restrict__ flags,
                                     const uint32_t* __restrict__ items_root, uint32_t* __restrict__ items_root_next) {
    // items_root (forest builds): node index of the root of the BLAS this item belongs to — child_base_idx is stored
    // relative to it, because the two-level traversal adds the BLAS offset to every node index (query_tlas.hlsl:383)
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const int root = items[i];
    const uint32_t my_root = items_root ? (level_base == 0u ? i : items_root[i]) : 0u;
    Kids k; gather_kids(b, root, max_leaf, k);
    const float4 nlo = b.lo[root], nhi = b.hi[root];
    const float nmn[3] = { nlo.x, nlo.y, nlo.z }, nmx[3] = { nhi.x, nhi.y, nhi.z };
    // slot assignment by octant (bvh_embree.rs:284-349): greedy min-cost matching of (child centre - node centre) . (+-1,+-1,+-1)
    float cost[8][8];
    for (int c = 0; c < k.n; c++) {
        const float4 lo = b.lo[k.id[c]], hi = b.hi[k.id[c]];
        const float d0 = 0.5f * (lo.x + hi.x) - 0.5f * (nmn[0] + nmx[0]), d1 = 0.5f * (lo.y + hi.y) - 0.5f * (nmn[1] + nmx[1]),
                    d2 = 0.5f * (lo.z + hi.z) - 0.5f * (nmn[2] + nmx[2]);
        for (int s = 0; s < 8; s++)
            cost[c][s] = d0 * ((s & 4) ? -1.f : 1.f) + d1 * ((s & 2) ? -1.f : 1.f) + d2 * ((s & 1) ? -1.f : 1.f);
    }
    int slot_child[8]; unsigned child_done = 0, slot_used = 0;
    for (int s = 0; s < 8; s++) slot_child[s] = -1;
    for (int r = 0; r < k.n; r++) {
        float bc = 3.4e38f; int bi = -1, bs = -1;
        for (int c = 0; c < k.n; c++) if (!((child_done >> c) & 1u))
            for (int s = 0; s < 8; s++) if (!((slot_used >> s) & 1u) && cost[c][s] < bc) { bc = cost[c][s]; bi = c; bs = s; }
        child_done |= 1u << bi; slot_used |= 1u << bs; slot_child[bs] = bi;
    }
    // encode (bvh_embree_to_cwbvh.rs:85-186)
    uint32_t w[20];
#pragma unroll
    for (int q = 0; q < 20; q++) w[q] = 0u;
    uint8_t* nb = reinterpret_cast<uint8_t*>(w);
    const bool exact = encode_bounds(w, nmn, nmx, slot_used, [&](int s, float cmn[3], float cmx[3]) {
        const int c = k.id[slot_child[s]];
        const float4 lo = b.lo[c], hi = b.hi[c];
        cmn[0] = lo.x; cmn[1] = lo.y; cmn[2] = lo.z; cmx[0] = hi.x; cmx[1] = hi.y; cmx[2] = hi.z;
    });
    if (exact) atomicOr(flags, 1u);
    w[4] = next_base + inner_off[i] - my_root;              // child_base_idx
    w[5] = prim_base + tri_off[i];                          // primitive_base_idx
    uint32_t tri_local = 0, n_in = 0, imask = 0;
    for (int s = 0; s < 8; s++) {
        if (slot_child[s] < 0) continue;
        const int c = k.id[slot_child[s]];
        const uint32_t cnt = b.count[c];
        if (cnt > max_leaf) {
            imask |= 1u << s;
            nb[24 + s] = (uint8_t)((24 + s) | 0x20);
            items_next[inner_off[i] + n_in] = c;
            if (items_root_next) items_root_next[inner_off[i] + n_in] = my_root;
            n_in++;
        } else {
            const uint8_t unary = cnt == 1 ? 0x20 : cnt == 2 ? 0x60 : 0xE0;
            nb[24 + s] = (uint8_t)(unary | tri_local);
            // primitives of the small subtree, left to right
            int stack[4]; int sp = 0; stack[sp++] = c;
            while (sp) {
                const int x = stack[--sp];
                const float4 xl = b.lo[x];
                if (node_left(xl) < 0) {
                    const uint32_t prim = (uint32_t)node_right(b.hi[x]);
                    const uint64_t slot = (uint64_t)prim_base + tri_off[i] + tri_local;
                    prim_indices[slot] = prim;
                    if (STRIDE != 0) write_tri_record<STRIDE>(tris9, prim, tri_out, slot);
                    tri_local++;
                } else { stack[sp++] = node_right(b.hi[x]); stack[sp++] = node_left(xl); }
            }
        }
    }
    nb[15] = (uint8_t)imask;
    uint4* dst = reinterpret_cast<uint4*>(nodes + (uint64_t)(level_base + i) * 80ull);
#pragma unroll
    for (int q = 0; q < 5; q++) dst[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}

// Device scratch of one build: ONE cudaMalloc (reserve) carved up by a bump allocator — a two-level build makes ~80 allocations,
// and in a process that already holds a lot of device memory each cudaMalloc / cudaFree costs up to a millisecond.  Requests
// that do not fit the arena fall back to their own cudaMalloc.  Everything is freed on scope exit, except an arena borrowed from
// its owner (a TLAS rebuild works in one the scene keeps: no allocation and no device-wide cudaFree per call).
struct Scratch {
    void* p[128]; int n = 0;
    char* arena = nullptr; size_t cap = 0, used = 0;
    bool owned = true;
    Scratch() = default;
    Scratch(void* borrowed, size_t bytes) : arena(static_cast<char*>(borrowed)), cap(bytes), owned(false) {}
    cudaError_t reserve(size_t bytes) {
        if (cudaMalloc((void**)&arena, bytes) != cudaSuccess) { arena = nullptr; cap = 0; cudaGetLastError(); }   // fall back to per-array allocations
        else cap = bytes;
        return cudaSuccess;
    }
    template <typename T> cudaError_t alloc(T** out, size_t bytes) {
        const size_t need = ((bytes ? bytes : 16) + 255) & ~(size_t)255;
        if (arena && used + need <= cap) { *out = (T*)(arena + used); used += need; return cudaSuccess; }
        if (n >= 128) return cudaErrorMemoryAllocation;
        void* q = nullptr; cudaError_t e = cudaMalloc(&q, need);
        if (e == cudaSuccess) { p[n++] = q; *out = (T*)q; }
        return e;
    }
    ~Scratch() { for (int i = 0; i < n; i++) cudaFree(p[i]); if (arena && owned) cudaFree(arena); }
};

// Exclusive sums of the flag arrays a and b over m + 1 entries, entry m zeroed first so that the sum there is the total.
// `consume` enqueues the work that reads the sums; then tot = the two totals, read back once the stream has drained.
template <typename F>
int scan_totals(void* d_tmp, size_t tmp_bytes, uint32_t* a, uint32_t* a_pos, uint32_t* b, uint32_t* b_pos, uint32_t m, cudaStream_t st,
                F consume, uint32_t tot[2], char* err, size_t errlen) {
    BCU(cudaMemsetAsync(a + m, 0, 4, st)); BCU(cudaMemsetAsync(b + m, 0, 4, st));
    BCU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, a, a_pos, (int)m + 1, st));
    BCU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, b, b_pos, (int)m + 1, st));
    consume();
    BCU(cudaMemcpyAsync(&tot[0], a_pos + m, 4, cudaMemcpyDeviceToHost, st));
    BCU(cudaMemcpyAsync(&tot[1], b_pos + m, 4, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    BCU(cudaGetLastError());
    return 0;
}

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// one PLOC run over `n` boxes already on the device; leaves are nodes [0, n), inner nodes follow.  With `prim_seg`
// clusters only merge inside their segment and the run ends with one root per segment, in segment order.
struct PlocOut { Bvh2 b; int* roots; uint32_t n_roots; uint32_t iters; void* d_tmp; size_t tmp_bytes; uint32_t n_nodes; };

int ploc_run(Scratch& sc, const float4* plo, const float4* phi, uint32_t n, const uint32_t* prim_seg, int r, cudaStream_t st,
             PlocOut* out, char* err, size_t errlen) {
    int* d_scene; unsigned long long *keys, *keys2; uint32_t *vals, *vals2;
    Bvh2 b; int *cl_a, *cl_b, *nn; uint32_t *keep, *keep_pos, *lead, *lead_pos, *node_seg = nullptr;
    BCU(sc.alloc(&d_scene, 6 * 4));
    BCU(sc.alloc(&keys, (size_t)n * 8)); BCU(sc.alloc(&keys2, (size_t)n * 8));
    BCU(sc.alloc(&vals, (size_t)n * 4)); BCU(sc.alloc(&vals2, (size_t)n * 4));
    BCU(sc.alloc(&b.lo, (size_t)2 * n * 16)); BCU(sc.alloc(&b.hi, (size_t)2 * n * 16)); BCU(sc.alloc(&b.count, (size_t)2 * n * 4));
    BCU(sc.alloc(&cl_a, (size_t)n * 4)); BCU(sc.alloc(&cl_b, (size_t)n * 4)); BCU(sc.alloc(&nn, (size_t)n * 4));
    BCU(sc.alloc(&keep, (size_t)(n + 1) * 4)); BCU(sc.alloc(&keep_pos, (size_t)(n + 1) * 4));
    BCU(sc.alloc(&lead, (size_t)(n + 1) * 4)); BCU(sc.alloc(&lead_pos, (size_t)(n + 1) * 4));
    if (prim_seg) BCU(sc.alloc(&node_seg, (size_t)2 * n * 4));
    BCU(cudaMemcpyAsync(d_scene, EMPTY_BOUNDS, sizeof EMPTY_BOUNDS, cudaMemcpyHostToDevice, st));
    box_bounds_kernel<<<blocks(n), TPB, 0, st>>>(plo, phi, n, d_scene);
    morton_kernel<<<blocks(n), TPB, 0, st>>>(plo, phi, n, d_scene, prim_seg, keys, vals);
    size_t tmp_bytes = 0, tmp2 = 0;
    BCU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys2, vals, vals2, (int)n, 0, 63, st));
    BCU(cub::DeviceScan::ExclusiveSum(nullptr, tmp2, keep, keep_pos, (int)n + 1, st));
    if (tmp2 > tmp_bytes) tmp_bytes = tmp2;
    void* d_tmp; BCU(sc.alloc(&d_tmp, tmp_bytes));
    BCU(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, keys, keys2, vals, vals2, (int)n, 0, 63, st));
    leaf_init_kernel<<<blocks(n), TPB, 0, st>>>(plo, phi, vals2, n, prim_seg, node_seg, b, cl_a);
    BCU(cudaGetLastError());
    uint32_t m = n, next_node = n, iters = 0;
    int* cl_in = cl_a; int* cl_out = cl_b;
    const char* tail_env = getenv("TRAY_BUILD_PLOC_TAIL");       // 0: keep the multi-kernel loop to the end (tests compare the two)
    const bool use_tail = !(tail_env && tail_env[0] == '0');
    PlocTailOut* d_tail = nullptr;
    BCU(sc.alloc(&d_tail, sizeof(PlocTailOut)));
    while (m > 1) {
        if (use_tail && m <= (uint32_t)PLOC_TAIL) {       // the rest of the run in one block, one synchronisation
            ploc_tail_kernel<<<1, PLOC_TAIL, 0, st>>>(cl_in, m, r, b, node_seg, next_node, d_tail);
            PlocTailOut t;
            BCU(cudaMemcpyAsync(&t, d_tail, sizeof t, cudaMemcpyDeviceToHost, st));
            BCU(cudaStreamSynchronize(st));
            BCU(cudaGetLastError());
            if (t.stalled && !prim_seg) { snprintf(err, errlen, "PLOC made no progress at %u clusters", t.m); return -3; }
            m = t.m; next_node = t.next_node; iters += t.iters;
            break;
        }
        ploc_nn_kernel<<<blocks(m), TPB, (size_t)(TPB + 2 * r) * 36, st>>>(cl_in, m, r, b, node_seg, nn);
        ploc_flag_kernel<<<blocks(m), TPB, 0, st>>>(nn, m, keep, lead);
        uint32_t tot[2];
        const int rc = scan_totals(d_tmp, tmp_bytes, keep, keep_pos, lead, lead_pos, m, st, [&] {
            ploc_merge_kernel<<<blocks(m), TPB, 0, st>>>(cl_in, nn, m, keep, keep_pos, lead, lead_pos, next_node, b, node_seg, cl_out);
        }, tot, err, errlen);
        if (rc) return rc;
        if (tot[1] == 0) {
            if (prim_seg) break;                      // every segment is down to one cluster
            snprintf(err, errlen, "PLOC made no progress at %u clusters", m); return -3;
        }
        next_node += tot[1]; m = tot[0]; iters++;
        int* t = cl_in; cl_in = cl_out; cl_out = t;
    }
    out->b = b; out->roots = cl_in; out->n_roots = m; out->iters = iters; out->d_tmp = d_tmp; out->tmp_bytes = tmp_bytes;
    out->n_nodes = next_node;
    return 0;
}

// reinsertion passes over the BVH2 of a PLOC run (3b above); `stats` (optional) receives the SAH cost before / after and the moves
struct OptStats { double cost_before, cost_after; uint32_t moves, passes; };
int optimize_run(Scratch& sc, const PlocOut& pl, uint32_t n_leaves, uint32_t passes, uint32_t max_visits, uint32_t rounds, cudaStream_t st,
                 OptStats* stats, char* err, size_t errlen) {
    const uint32_t nn = pl.n_nodes;
    if (stats) memset(stats, 0, sizeof *stats);
    if (passes == 0 || nn <= n_leaves + 2) return 0;
    OptArrays o; o.visits = nullptr;
    uint32_t* arrived; uint32_t* d_count; double* d_cost; uint8_t* drop; uint8_t* dirty;
    BCU(sc.alloc(&o.parent, (size_t)nn * 4)); BCU(sc.alloc(&o.gain, (size_t)nn * 4)); BCU(sc.alloc(&o.target, (size_t)nn * 4));
    BCU(sc.alloc(&o.lock, (size_t)nn * 8)); BCU(sc.alloc(&arrived, (size_t)nn * 4));
    BCU(sc.alloc(&d_count, 4)); BCU(sc.alloc(&d_cost, 16)); BCU(sc.alloc(&drop, (size_t)nn)); BCU(sc.alloc(&dirty, (size_t)nn)); BCU(sc.alloc(&o.win, (size_t)nn));
    BCU(cudaMemsetAsync(o.parent, 0xff, (size_t)nn * 4, st));
    opt_parent_kernel<<<blocks(nn - n_leaves), TPB, 0, st>>>(pl.b, n_leaves, nn, o.parent);
    BCU(cudaMemsetAsync(d_cost, 0, 16, st));
    BCU(cudaMemsetAsync(d_count, 0, 4, st));
    opt_cost_kernel<<<blocks(nn - n_leaves), TPB, 0, st>>>(pl.b, n_leaves, nn, d_cost);
    for (uint32_t pass = 0; pass < passes; pass++) {
        opt_find_kernel<<<(nn + 127) / 128, 128, 0, st>>>(pl.b, nn, o, max_visits);
        BCU(cudaMemsetAsync(dirty, 0, (size_t)nn, st));
        for (uint32_t round = 0; round < rounds; round++) {     // several claim / apply rounds over the moves one search found
            BCU(cudaMemsetAsync(o.lock, 0, (size_t)nn * 8, st));
            opt_lock_kernel<<<blocks(nn), TPB, 0, st>>>(pl.b, nn, o, dirty, (int)round);
            opt_check_kernel<<<blocks(nn), TPB, 0, st>>>(pl.b, nn, o);
            opt_cycle_kernel<<<blocks(nn), TPB, 0, st>>>(nn, o, drop);
            opt_apply_kernel<<<blocks(nn), TPB, 0, st>>>(pl.b, nn, o, drop, dirty, d_count);
        }
        BCU(cudaMemsetAsync(arrived, 0, (size_t)nn * 4, st));
        opt_refit_kernel<<<blocks(n_leaves), TPB, 0, st>>>(pl.b, n_leaves, o.parent, arrived);
    }
    opt_cost_kernel<<<blocks(nn - n_leaves), TPB, 0, st>>>(pl.b, n_leaves, nn, d_cost + 1);
    BCU(cudaGetLastError());
    if (stats) {
        double c[2]; uint32_t moves;
        BCU(cudaMemcpyAsync(c, d_cost, 16, cudaMemcpyDeviceToHost, st));
        BCU(cudaMemcpyAsync(&moves, d_count, 4, cudaMemcpyDeviceToHost, st));
        BCU(cudaStreamSynchronize(st));
        stats->cost_before = c[0]; stats->cost_after = c[1]; stats->moves = moves; stats->passes = passes;
    }
    return 0;
}

// the reinsertion knobs: TRAY_CUDA_BUILD_REINSERT passes (0 = off), _VISITS node visits per move search, _ROUNDS claim / apply
// rounds per pass (obvhs: `reinsertion_batch_ratio`, reference src/main.rs:563-587)
struct Reinsert { uint32_t passes, visits, rounds; };
Reinsert reinsert_knobs() {
    const auto env_u32 = [](const char* name, uint32_t dflt) { const char* v = getenv(name); return v && *v ? (uint32_t)atoi(v) : dflt; };
    return { env_u32("TRAY_CUDA_BUILD_REINSERT", 4u), env_u32("TRAY_CUDA_BUILD_REINSERT_VISITS", 192u), env_u32("TRAY_CUDA_BUILD_REINSERT_ROUNDS", 3u) };
}

// level-synchronous collapse of the BVH2 subtrees `roots` (one wide root node each, stored at node indices 0..n_roots-1 of
// `nodes`, i.e. at `nodes` itself — pass the destination already offset).  forest = child indices relative to each root.
// level_end[L] = the node index (relative to `nodes`) one past level L.
struct CollapseOut { uint32_t n_nodes, n_prims, levels; bool force_exact; std::vector<uint32_t> level_end; };

int collapse_run(Scratch& sc, const PlocOut& pl, uint32_t n_prims, bool forest, uint32_t max_leaf, uint32_t tri_stride,
                 const float* d_tris9, uint8_t* nodes, uint64_t node_cap, uint8_t* tri_out, uint32_t* prim_idx, uint32_t prim_base0,
                 cudaStream_t st, CollapseOut* out, char* err, size_t errlen) {
    const uint32_t n = n_prims;
    int *items_a, *items_b; uint32_t *n_inner, *n_tri, *inner_off, *tri_off, *d_flags, *root_a = nullptr, *root_b = nullptr;
    BCU(sc.alloc(&items_a, (size_t)(n + 1) * 4)); BCU(sc.alloc(&items_b, (size_t)(n + 1) * 4));
    BCU(sc.alloc(&n_inner, (size_t)(n + 2) * 4)); BCU(sc.alloc(&n_tri, (size_t)(n + 2) * 4));
    BCU(sc.alloc(&inner_off, (size_t)(n + 2) * 4)); BCU(sc.alloc(&tri_off, (size_t)(n + 2) * 4));
    BCU(sc.alloc(&d_flags, 4));
    if (forest) { BCU(sc.alloc(&root_a, (size_t)(n + 1) * 4)); BCU(sc.alloc(&root_b, (size_t)(n + 1) * 4)); }
    BCU(cudaMemsetAsync(d_flags, 0, 4, st));
    BCU(cudaMemcpyAsync(items_a, pl.roots, (size_t)pl.n_roots * 4, cudaMemcpyDeviceToDevice, st));
    uint32_t n_items = pl.n_roots, level_base = 0, prim_base = prim_base0, levels = 0;
    out->level_end.clear();
    int* it_in = items_a; int* it_out = items_b; uint32_t* rt_in = root_a; uint32_t* rt_out = root_b;
    while (n_items) {
        if ((uint64_t)level_base + n_items > node_cap) { snprintf(err, errlen, "node count exceeds its bound"); return -3; }
        collapse_count_kernel<<<blocks(n_items), TPB, 0, st>>>(it_in, n_items, pl.b, max_leaf, n_inner, n_tri);
        const uint32_t next_base = level_base + n_items;
        uint32_t tot[2];
        const int rc = scan_totals(pl.d_tmp, pl.tmp_bytes, n_inner, inner_off, n_tri, tri_off, n_items, st, [&] {
#define EMIT(S) collapse_emit_kernel<S><<<blocks(n_items), TPB, 0, st>>>(it_in, n_items, pl.b, max_leaf, inner_off, tri_off, level_base, next_base, \
                    prim_base, d_tris9, nodes, tri_out, prim_idx, it_out, d_flags, forest ? rt_in : nullptr, forest ? rt_out : nullptr)
            if (tri_stride == 64) EMIT(64); else if (tri_stride == 24) EMIT(24); else if (tri_stride == 48) EMIT(48); else EMIT(0);
#undef EMIT
        }, tot, err, errlen);
        if (rc) return rc;
        level_base = next_base; prim_base += tot[1]; n_items = tot[0]; levels++;
        out->level_end.push_back(level_base);
        int* t = it_in; it_in = it_out; it_out = t;
        uint32_t* u = rt_in; rt_in = rt_out; rt_out = u;
    }
    if (prim_base - prim_base0 != n) { snprintf(err, errlen, "collapse placed %u of %u primitives", prim_base - prim_base0, n); return -3; }
    uint32_t flags = 0;
    BCU(cudaMemcpyAsync(&flags, d_flags, 4, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    out->n_nodes = level_base; out->n_prims = n; out->levels = levels; out->force_exact = (flags & 1u) != 0;
    return 0;
}

__global__ void seg_of_prims_kernel(const uint64_t* __restrict__ offsets, uint32_t n_obj, uint32_t n, uint32_t* __restrict__ prim_seg) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t lo = 0, hi = n_obj;                      // last k with offsets[k] <= i
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (offsets[mid] <= i) lo = mid; else hi = mid; }
    prim_seg[i] = lo;
}

// boxes of the BLAS roots (TLAS primitives)
__global__ void blas_boxes_kernel(const int* __restrict__ roots, uint32_t n_obj, Bvh2 b, float4* __restrict__ plo, float4* __restrict__ phi) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_obj) return;
    plo[i] = b.lo[roots[i]]; phi[i] = b.hi[roots[i]];
}

// The TLAS leg of a two-level build, over n instance boxes (xyz of tlo / thi): PLOC, reinsertion, collapse.  Writes the wide
// nodes at `nodes` (child indices relative to it) and perm[j] = the instance of TLAS leaf j.
struct TlasOut { uint32_t n_nodes, iters; CollapseOut co; };
int tlas_run(Scratch& sc, const float4* tlo, const float4* thi, uint32_t n, uint32_t max_leaf, int r, const Reinsert& re, uint8_t* nodes,
             uint32_t* perm, cudaStream_t st, TlasOut* out, char* err, size_t errlen) {
    PlocOut tp;
    int rc = ploc_run(sc, tlo, thi, n, nullptr, r, st, &tp, err, errlen);
    if (rc) return rc;
    rc = optimize_run(sc, tp, n, re.passes, re.visits, re.rounds, st, nullptr, err, errlen);
    if (rc) return rc;
    rc = collapse_run(sc, tp, n, false, max_leaf, 0, nullptr, nodes, (uint64_t)n + 1, nullptr, perm, 0, st, &out->co, err, errlen);
    if (rc) return rc;
    out->n_nodes = out->co.n_nodes; out->iters = tp.iters;
    return 0;
}

// TLAS primitives of a rebuild: the exact box of the BLAS root of canonical instance i (ordered ints of the refit)
__global__ void tlas_boxes_kernel(const uint32_t* __restrict__ canon, uint32_t n, const int4* __restrict__ node_box, float4* __restrict__ plo,
                                  float4* __restrict__ phi) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int4 l = node_box[2ull * canon[i]], h = node_box[2ull * canon[i] + 1];
    plo[i] = make_float4(o2f(l.x), o2f(l.y), o2f(l.z), 0.f);
    phi[i] = make_float4(o2f(h.x), o2f(h.y), o2f(h.z), 0.f);
}

// blas_offsets of the rebuilt TLAS: leaf j holds canonical instance perm[j], whose BLAS root is canon[perm[j]]
__global__ void blas_compose_kernel(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ canon, uint32_t n, uint32_t* __restrict__ blas) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) blas[j] = canon[perm[j]];
}

// an instanced TLAS: leaf j holds instance perm[j], whose record (with its BLAS root) is in[perm[j]]
__global__ void instance_compose_kernel(const uint32_t* __restrict__ perm, const uint4* __restrict__ in, uint32_t n, uint32_t* __restrict__ blas,
                                        uint4* __restrict__ rec) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint4* src = in + 4ull * perm[j];
#pragma unroll
    for (int q = 0; q < 4; q++) rec[4ull * j + q] = src[q];
    blas[j] = src[3].x;
}

__global__ void gather_nodes_kernel(const uint4* __restrict__ nodes, const uint32_t* __restrict__ idx, uint32_t n, uint4* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
#pragma unroll
    for (int q = 0; q < 5; q++) out[5ull * i + q] = nodes[5ull * idx[i] + q];
}

__global__ void exact_scan_kernel(const uint4* __restrict__ nodes, uint32_t n, uint32_t* __restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && tray::node_needs_exact(nodes[5ull * i].w)) atomicOr(flag, 1u);
}

// the topology's TLAS part after a rebuild: every one of the m new nodes, in collapse order (which is level order)
__global__ void tlas_items_kernel(uint2* __restrict__ items, uint32_t m, uint32_t tlas_start) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) items[k] = make_uint2(tlas_start + k, tlas_start);
}

// ---- 5. refit: the same trees, re-encoded tight over moved triangles (tray_cuda_scene_refit) ---------------------------------
// A topology walk, once per scene, lists the nodes reachable from the roots level by level as (node, tree base) pairs: a
// child's index is its tree base + child_base_idx + rank (the BLAS root, or tlas_start in the TLAS).  A refit then runs one
// pass over the triangle slots (records + slot boxes) and one launch per level, deepest first, in which every node takes the
// union of its slots' boxes and re-encodes p, exponents and the q bytes of its used slots.  Boxes are ordered ints (f2o),
// min / max are exact, and no two threads write one node: the bytes are the same on every run.
enum : uint32_t { WALK_LEAF_RANGE = 1u, WALK_CHILD_RANGE = 2u, WALK_TWICE = 4u };

__device__ __forceinline__ uint32_t leaf_count(uint32_t meta) {   // unary triangle count of a leaf slot's meta byte
    const uint32_t u = meta >> 5;
    return u == 1u ? 1u : u == 3u ? 2u : u == 7u ? 3u : 0u;
}
__device__ __forceinline__ uint32_t node_meta(const uint4& n1, int s) { return ((s < 4 ? n1.z : n1.w) >> (8 * (s & 3))) & 0xffu; }

// the coordinate check of a refit: scan[0] != 0 when a coordinate is not finite; scan[1 + a] / scan[4 + a] the minimum / maximum
// of axis a over all vertices as ordered ints (their difference tells whether every box extent stays finite)
__global__ void refit_scan_kernel(const float* __restrict__ tris9, uint64_t n9, int* __restrict__ scan) {
    bool bad = false;
    float mn[3] = { 3.4e38f, 3.4e38f, 3.4e38f }, mx[3] = { -3.4e38f, -3.4e38f, -3.4e38f };
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n9; i += (uint64_t)gridDim.x * blockDim.x) {
        const float v = tris9[i];
        bad |= !isfinite(v);
        const int a = (int)(i % 3);
#pragma unroll
        for (int b = 0; b < 3; b++)
            if (a == b) { mn[b] = fminf(mn[b], v); mx[b] = fmaxf(mx[b], v); }
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(scan, 1);
    warp_bounds(mn, mx, scan + 1, scan + 4);
}

__global__ void refit_roots_kernel(const uint2* __restrict__ items, uint32_t begin, uint32_t n, uint32_t* __restrict__ visited,
                                   uint32_t* __restrict__ err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && atomicExch(visited + items[begin + i].x, 1u) != 0u) atomicOr(err, WALK_TWICE);
}

// one level of the walk: checks every leaf range against `leaf_limit` and appends the inner children at `tail`.  A node with a
// leaf entry sets bit 1 of its tree root's visited word: that tree reaches a primitive.
__global__ void refit_walk_kernel(const uint4* __restrict__ nodes, uint2* __restrict__ items, uint32_t begin, uint32_t n, uint32_t cap,
                                  uint64_t child_lo, uint64_t child_hi, uint64_t leaf_limit, uint32_t* __restrict__ tail,
                                  uint32_t* __restrict__ visited, uint32_t* __restrict__ err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 it = items[begin + i];
    const uint4 n0 = nodes[5ull * it.x], n1 = nodes[5ull * it.x + 1];
    const uint32_t imask = n0.w >> 24;
    bool leaf = false;
    for (int s = 0; s < 8; s++) {
        const uint32_t meta = node_meta(n1, s);
        if (((imask >> s) & 1u) || meta == 0u) continue;
        if ((uint64_t)n1.y + (meta & 31u) + leaf_count(meta) > leaf_limit) atomicOr(err, WALK_LEAF_RANGE);
        leaf |= leaf_count(meta) > 0u;
    }
    if (leaf) atomicOr(visited + it.y, 2u);
    const uint32_t k = __popc(imask);
    if (!k) return;
    const uint32_t pos = atomicAdd(tail, k);
    for (uint32_t r = 0; r < k; r++) {
        const uint64_t c = (uint64_t)it.y + n1.x + r;
        if (c < child_lo || c >= child_hi) { atomicOr(err, WALK_CHILD_RANGE); continue; }
        if (atomicExch(visited + c, 1u) != 0u) { atomicOr(err, WALK_TWICE); continue; }
        if (pos + r < cap) items[pos + r] = make_uint2((uint32_t)c, it.y);
        else atomicOr(err, WALK_TWICE);                  // more nodes than the array holds: some node came twice
    }
}

// a node that no root reaches keeps its bytes through every refit: whether one of them asks for the exact node test is fixed.
// Bit 0: such a node below `split` (tlas_start), bit 1: at or above it (nodes a TLAS rebuild overwrites or leaves past n_nodes).
__global__ void refit_unreached_exact_kernel(const uint4* __restrict__ nodes, uint64_t n_nodes, uint64_t split, const uint32_t* __restrict__ visited,
                                             uint32_t* __restrict__ flag) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes || visited[i]) return;
    if (tray::node_needs_exact(nodes[5 * i].w)) atomicOr(flag, i < split ? 1u : 2u);
}

// what a TLAS rebuild needs of the BLAS part, over its n walk items (the first n_roots of them its roots): bit 0 = some node
// has an index >= tlas_start (the TLAS is not the tail of the node array), bit 1 = some BLAS reaches no primitive
__global__ void refit_blas_check_kernel(const uint2* __restrict__ items, uint32_t n, uint32_t n_roots, const uint32_t* __restrict__ visited,
                                        uint32_t tlas_start, uint32_t* __restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t x = items[i].x;
    if (x >= tlas_start) atomicOr(flag, 1u);
    if (i < n_roots && !(visited[x] & 2u)) atomicOr(flag, 2u);
}

// records of slot k from triangle prim_indices[k] (k without the map), and the slot's box from the f32 vertices
template <int STRIDE>
__global__ void refit_tris_kernel(const float* __restrict__ tris9, uint32_t n, const uint32_t* __restrict__ prim_indices,
                                  uint8_t* __restrict__ tri_out, int4* __restrict__ slot_box) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t prim = prim_indices ? prim_indices[k] : k;
    write_tri_record<STRIDE>(tris9, prim, tri_out, k);
    float mn[3], mx[3];
    tri_box(tris9 + 9ull * prim, mn, mx);
    int lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; a++) { lo[a] = f2o(mn[a]); hi[a] = f2o(mx[a]); }
    slot_box[2ull * k] = make_int4(lo[0], lo[1], lo[2], 0);
    slot_box[2ull * k + 1] = make_int4(hi[0], hi[1], hi[2], 0);
}

// one level: a node's slots are its inner children (boxes of the level below) and its leaves (slot boxes of triangles, or, in
// the TLAS, the boxes of the BLAS roots behind the instances).  A node with no box under it keeps its bytes.
template <bool TLAS>
__global__ void __launch_bounds__(TPB) refit_node_kernel(const uint2* __restrict__ items, uint32_t n, uint4* __restrict__ nodes,
                                                         int4* __restrict__ node_box, const int4* __restrict__ slot_box,
                                                         const uint32_t* __restrict__ blas, uint32_t* __restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 it = items[i];
    uint4* nd = nodes + 5ull * it.x;
    uint32_t w[20];
#pragma unroll
    for (int q = 0; q < 5; q++) { const uint4 v = nd[q]; w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w; }
    const uint4 n1 = make_uint4(w[4], w[5], w[6], w[7]);
    const uint32_t imask = w[3] >> 24;
    int blo[8][3], bhi[8][3];
    int nlo[3] = { INT_MAX, INT_MAX, INT_MAX }, nhi[3] = { INT_MIN, INT_MIN, INT_MIN };
    uint32_t used = 0;
#pragma unroll
    for (int s = 0; s < 8; s++) {
        const uint32_t meta = node_meta(n1, s);
#pragma unroll
        for (int a = 0; a < 3; a++) { blo[s][a] = INT_MAX; bhi[s][a] = INT_MIN; }
        if ((imask >> s) & 1u) {
            const uint64_t c = (uint64_t)it.y + n1.x + __popc(imask & ((1u << s) - 1u));
            const int4 l = node_box[2 * c], h = node_box[2 * c + 1];
            blo[s][0] = l.x; blo[s][1] = l.y; blo[s][2] = l.z; bhi[s][0] = h.x; bhi[s][1] = h.y; bhi[s][2] = h.z;
        } else if (meta != 0u) {
            const uint32_t first = n1.y + (meta & 31u), cnt = leaf_count(meta);
            for (uint32_t j = 0; j < cnt; j++) {
                const uint64_t b = TLAS ? 2ull * blas[first + j] : 2ull * (first + j);
                const int4 l = TLAS ? node_box[b] : slot_box[b], h = TLAS ? node_box[b + 1] : slot_box[b + 1];
                blo[s][0] = min(blo[s][0], l.x); blo[s][1] = min(blo[s][1], l.y); blo[s][2] = min(blo[s][2], l.z);
                bhi[s][0] = max(bhi[s][0], h.x); bhi[s][1] = max(bhi[s][1], h.y); bhi[s][2] = max(bhi[s][2], h.z);
            }
        }
        if (meta != 0u) used |= 1u << s;
#pragma unroll
        for (int a = 0; a < 3; a++) { nlo[a] = min(nlo[a], blo[s][a]); nhi[a] = max(nhi[a], bhi[s][a]); }
    }
    node_box[2ull * it.x] = make_int4(nlo[0], nlo[1], nlo[2], 0);
    node_box[2ull * it.x + 1] = make_int4(nhi[0], nhi[1], nhi[2], 0);
    if (nlo[0] > nhi[0]) return;
    const float nmn[3] = { o2f(nlo[0]), o2f(nlo[1]), o2f(nlo[2]) }, nmx[3] = { o2f(nhi[0]), o2f(nhi[1]), o2f(nhi[2]) };
    const bool exact = encode_bounds(w, nmn, nmx, used, [&](int s, float cmn[3], float cmx[3]) {
#pragma unroll
        for (int a = 0; a < 3; a++) { cmn[a] = o2f(blo[s][a]); cmx[a] = o2f(bhi[s][a]); }
    });
    if (exact) atomicOr(flag, 1u);
#pragma unroll
    for (int q = 0; q < 5; q++) nd[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}

}  // namespace

// object_offsets == NULL: one flat BVH.  Otherwise (n_objects + 1 offsets into the triangle array): one BLAS per object —
// built together, as a forest, by a PLOC run that never merges across objects — plus a TLAS over the BLAS boxes, laid out
// as cwbvh_gpu_runner lays them out (src/rt_gpu/mod.rs:53-100): BLAS nodes | TLAS nodes, tlas_start, blas_offsets in
// TLAS-leaf order, triangle indices global.
int build_tlas(const float* tris9_host, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects, uint32_t tri_stride,
               uint32_t max_leaf, uint32_t radius, cudaStream_t st, Result* out, char* err, size_t errlen) {
    *out = Result{};
    if (n_tris == 0) return 0;
    if (n_tris >= 0x7fffffffull) { snprintf(err, errlen, "too many triangles"); return -1; }
    const bool tlas = object_offsets != nullptr;
    if (tlas) {
        if (n_objects == 0 || n_objects >= (1u << 21)) { snprintf(err, errlen, "object count must be 1 .. 2^21 - 1"); return -1; }
        if (object_offsets[0] != 0 || object_offsets[n_objects] != n_tris) { snprintf(err, errlen, "object_offsets must run from 0 to n_tris"); return -1; }
        for (uint32_t k = 0; k < n_objects; k++)
            if (object_offsets[k + 1] <= object_offsets[k]) { snprintf(err, errlen, "object %u is empty", k); return -1; }
    }
    const uint32_t n = (uint32_t)n_tris;
    const int r = (int)(radius < 1 ? 1 : (radius > 64 ? 64 : radius));
    const double t_begin = now_ms();
    Scratch sc;
    // every array of the run (~320 B per triangle) + slack, then those of the TLAS
    sc.reserve((size_t)n * 344 + (size_t)(tlas ? n_objects : 0) * 16 + (64u << 20) + (tlas ? (size_t)n_objects * 344 + (16u << 20) : 0));
    float* d_tris9; float4 *plo, *phi; uint32_t* prim_seg = nullptr; uint64_t* d_off = nullptr;
    BCU(sc.alloc(&d_tris9, (size_t)n * 36));
    BCU(sc.alloc(&plo, (size_t)n * 16)); BCU(sc.alloc(&phi, (size_t)n * 16));
    BCU(tray::upload_pipelined(d_tris9, tris9_host, (size_t)n * 36, st));
    if (tlas) {
        BCU(sc.alloc(&prim_seg, (size_t)n * 4)); BCU(sc.alloc(&d_off, (size_t)(n_objects + 1) * 8));
        BCU(cudaMemcpyAsync(d_off, object_offsets, (size_t)(n_objects + 1) * 8, cudaMemcpyHostToDevice, st));
        seg_of_prims_kernel<<<blocks(n), TPB, 0, st>>>(d_off, n_objects, n, prim_seg);
    }
    BCU(cudaStreamSynchronize(st));
    const double t_upload = now_ms();
    tri_boxes_kernel<<<blocks(n), TPB, 0, st>>>(d_tris9, n, plo, phi);
    PlocOut pl;
    int rc = ploc_run(sc, plo, phi, n, prim_seg, r, st, &pl, err, errlen);
    if (rc) return rc;
    if (tlas && pl.n_roots != n_objects) { snprintf(err, errlen, "PLOC left %u roots for %u objects", pl.n_roots, n_objects); return -3; }
    BCU(cudaStreamSynchronize(st));
    const double t_ploc = now_ms();
    const Reinsert re = reinsert_knobs();
    OptStats os;
    rc = optimize_run(sc, pl, n, re.passes, re.visits, re.rounds, st, &os, err, errlen);
    if (rc) return rc;
    BCU(cudaStreamSynchronize(st));
    const double t_opt = now_ms();

    // node count of a BLAS is bounded by its triangle count (>= 1 node); the TLAS by the object count
    const uint64_t blas_cap = (uint64_t)n + (tlas ? n_objects : 1), tlas_cap = tlas ? (uint64_t)n_objects + 1 : 0;
    // the outputs: handed to `out` on success, freed on every other return
    DevPtr<uint8_t> d_nodes, d_tri_out; DevPtr<uint32_t> d_prim_idx, d_blas;
    BCU(dev_alloc(d_nodes, (blas_cap + tlas_cap) * 80));
    BCU(dev_alloc(d_tri_out, (size_t)n * tri_stride));
    BCU(dev_alloc(d_prim_idx, (size_t)n * 4));
    if (tlas) BCU(dev_alloc(d_blas, (size_t)n_objects * 4));
    CollapseOut co;
    rc = collapse_run(sc, pl, n, tlas, max_leaf, tri_stride, d_tris9, d_nodes.get(), blas_cap, d_tri_out.get(), d_prim_idx.get(), 0, st, &co,
                      err, errlen);
    if (rc) return rc;
    uint32_t tlas_start = 0, n_nodes = co.n_nodes, tl_iters = 0, tl_levels = 0;
    bool force_exact = co.force_exact;
    if (tlas) {
        // TLAS: the same pipeline over the BLAS boxes; its "triangles" are instance slots.  blas_offsets in TLAS-leaf order are its
        // leaf permutation, as object k's BLAS has its root wide node at node index k (forest level 0).
        float4 *tlo, *thi;
        BCU(sc.alloc(&tlo, (size_t)n_objects * 16)); BCU(sc.alloc(&thi, (size_t)n_objects * 16));
        blas_boxes_kernel<<<blocks(n_objects), TPB, 0, st>>>(pl.roots, n_objects, pl.b, tlo, thi);
        tlas_start = co.n_nodes;
        TlasOut to;
        rc = tlas_run(sc, tlo, thi, n_objects, max_leaf, r, re, d_nodes.get() + (uint64_t)tlas_start * 80, d_blas.get(), st, &to, err, errlen);
        if (rc) return rc;
        n_nodes += to.n_nodes; tl_iters = to.iters; tl_levels = to.co.levels; force_exact = force_exact || to.co.force_exact;
    }
    const double t_end = now_ms();
    out->d_nodes = std::move(d_nodes); out->n_nodes = n_nodes; out->node_cap = blas_cap + tlas_cap; out->d_tris = std::move(d_tri_out);
    out->d_prim_indices = std::move(d_prim_idx); out->d_blas_offsets = std::move(d_blas); out->n_instances = tlas ? n_objects : 0; out->tlas_start = tlas_start;
    out->force_exact = force_exact;
    out->stats.n_tris = n; out->stats.n_nodes = n_nodes; out->stats.ploc_iterations = pl.iters + tl_iters; out->stats.levels = co.levels + tl_levels;
    out->stats.ms_upload = (float)(t_upload - t_begin); out->stats.ms_sort = 0.f;
    out->stats.ms_ploc = (float)(t_ploc - t_upload); out->stats.ms_collapse = (float)(t_end - t_opt); out->stats.ms_total = (float)(t_end - t_begin);
    out->stats.ms_reinsert = (float)(t_opt - t_ploc); out->stats.reinsert_passes = os.passes; out->stats.reinsert_moves = os.moves;
    out->stats.sah_before = (float)os.cost_before; out->stats.sah_after = (float)os.cost_after;
    return 0;
}

int refit_walk(const void* d_nodes, uint64_t n_nodes, uint64_t n_tris, const uint32_t* d_blas, uint32_t n_instances, uint32_t tlas_start,
               cudaStream_t st, RefitTopology* out, char* err, size_t errlen) {
    RefitTopology t;
    // roots: node 0, or the distinct blas_offsets (a BLAS shared by two instances is one tree) and then the TLAS
    std::vector<uint32_t> roots;
    if (n_instances) {
        roots.resize(n_instances);
        if (cudaMemcpy(roots.data(), d_blas, (size_t)n_instances * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
            snprintf(err, errlen, "blas_offsets download failed"); cudaGetLastError(); return -2;
        }
        std::sort(roots.begin(), roots.end());
        // the instances' roots in canonical order (a TLAS rebuild permutes blas_offsets, so this stays what it is)
        BCU(dev_alloc(t.d_canon, (size_t)n_instances * 4));
        BCU(cudaMemcpyAsync(t.d_canon.get(), roots.data(), (size_t)n_instances * 4, cudaMemcpyHostToDevice, st));
        roots.erase(std::unique(roots.begin(), roots.end()), roots.end());
        if (roots.back() >= n_nodes) { snprintf(err, errlen, "blas_offsets entry %u outside %llu nodes", roots.back(), (unsigned long long)n_nodes); return -1; }
        t.roots = roots;
        BCU(dev_alloc(t.d_roots, roots.size() * 4));
        BCU(dev_alloc(t.d_root_nodes, roots.size() * 80));
        BCU(cudaMemcpyAsync(t.d_roots.get(), roots.data(), roots.size() * 4, cudaMemcpyHostToDevice, st));
    } else if (n_nodes) {
        roots.push_back(0u);
    }
    DevPtr<uint32_t> visited_buf, walk_buf;
    const uint64_t cap = n_nodes ? n_nodes : 1;
    BCU(dev_alloc(t.d_items, cap * sizeof(uint2)));
    BCU(dev_alloc(t.d_node_box, cap * 2 * sizeof(int4)));
    BCU(dev_alloc(t.d_slot_box, (n_tris ? n_tris : 1) * 2 * sizeof(int4)));
    BCU(dev_alloc(t.d_flag, 7 * 4));                  // the level flag; the coordinate check's 7 words
    BCU(dev_alloc(visited_buf, cap * 4));
    BCU(dev_alloc(walk_buf, 8));
    uint32_t *visited = visited_buf.get(), *d_walk = walk_buf.get();      // d_walk: [0] tail, [1] error bits
    uint2* items = t.d_items.get();
    BCU(cudaMemsetAsync(visited, 0, cap * 4, st));
    BCU(cudaMemsetAsync(d_walk, 0, 8, st));
    const uint4* nodes = static_cast<const uint4*>(d_nodes);
    uint32_t tail = 0;
    t.level_off.push_back(0);
    // one tree part: its roots become a level, then level after level until one adds no node
    auto walk = [&](const std::vector<uint2>& part_roots, uint64_t child_lo, uint64_t leaf_limit) -> int {
        if (part_roots.empty()) return 0;
        // the `tail` nodes listed so far are distinct: a part whose roots do not fit next to them repeats one (e.g. a
        // blas_offsets entry equal to tlas_start).  Refused here, before its roots are written to the list.
        if ((uint64_t)tail + part_roots.size() > cap) {
            snprintf(err, errlen, "the tree cannot be refit: a node is reached twice");
            return -1;
        }
        BCU(cudaMemcpyAsync(items + tail, part_roots.data(), part_roots.size() * sizeof(uint2), cudaMemcpyHostToDevice, st));
        refit_roots_kernel<<<blocks(part_roots.size()), TPB, 0, st>>>(items, tail, (uint32_t)part_roots.size(), visited, d_walk + 1);
        tail += (uint32_t)part_roots.size();
        BCU(cudaMemcpyAsync(d_walk, &tail, 4, cudaMemcpyHostToDevice, st));
        t.level_off.push_back(tail);
        for (;;) {
            const uint32_t begin = t.level_off[t.level_off.size() - 2], n = tail - begin;
            refit_walk_kernel<<<blocks(n), TPB, 0, st>>>(nodes, items, begin, n, (uint32_t)cap, child_lo, n_nodes, leaf_limit, d_walk,
                                                         visited, d_walk + 1);
            uint32_t w[2];
            BCU(cudaMemcpyAsync(w, d_walk, 8, cudaMemcpyDeviceToHost, st));
            BCU(cudaStreamSynchronize(st));
            BCU(cudaGetLastError());
            if (w[1]) {
                snprintf(err, errlen, "the tree cannot be refit: %s", (w[1] & WALK_TWICE) ? "a node is reached twice"
                         : (w[1] & WALK_CHILD_RANGE) ? "a child index is outside the node array" : "a leaf range is outside its array");
                return -1;
            }
            if (w[0] == tail) return 0;
            tail = w[0];
            t.level_off.push_back(tail);
        }
    };
    std::vector<uint2> part;
    for (uint32_t r : roots) part.push_back(make_uint2(r, r));
    if (const int rc = walk(part, 0, n_tris)) return rc;
    t.n_blas_levels = (uint32_t)t.level_off.size() - 1;
    BCU(cudaMemsetAsync(t.d_flag.get(), 0, 8, st));
    if (n_instances) {
        const uint32_t n_blas = t.level_off.back();
        refit_blas_check_kernel<<<blocks(n_blas), TPB, 0, st>>>(items, n_blas, (uint32_t)roots.size(), visited, tlas_start, t.d_flag.get() + 1);
        part.assign(1, make_uint2(tlas_start, tlas_start));
        if (const int rc = walk(part, tlas_start, n_instances)) return rc;
    }
    if (n_nodes) refit_unreached_exact_kernel<<<blocks(n_nodes), TPB, 0, st>>>(nodes, n_nodes, tlas_start, visited, t.d_flag.get());
    uint32_t f[2] = { 0, 0 };
    BCU(cudaMemcpyAsync(f, t.d_flag.get(), 8, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    BCU(cudaGetLastError());
    t.unreached_exact = f[0] != 0; t.unreached_exact_blas = (f[0] & 1u) != 0;
    t.blas_past_tlas = (f[1] & 1u) != 0; t.blas_empty = (f[1] & 2u) != 0;
    t.cap = cap;
    t.bytes = cap * (sizeof(uint2) + 2 * sizeof(int4)) + (n_tris ? n_tris : 1) * 2 * sizeof(int4) + 7 * 4 + (uint64_t)n_instances * 4
            + (uint64_t)t.roots.size() * 84;
    *out = std::move(t);
    return 0;
}

int refit_check(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, cudaStream_t st, bool* bad, char* err, size_t errlen) {
    int init[7] = { 0 }, scan[7];                     // flag 0, then the empty bounds
    memcpy(init + 1, EMPTY_BOUNDS, sizeof EMPTY_BOUNDS);
    int* d_scan = reinterpret_cast<int*>(t.d_flag.get());
    BCU(cudaMemcpyAsync(d_scan, init, sizeof init, cudaMemcpyHostToDevice, st));
    if (n_tris) refit_scan_kernel<<<blocks(n_tris * 9 < (1ull << 24) ? n_tris * 9 : (1ull << 24)), TPB, 0, st>>>(d_tris9, n_tris * 9, d_scan);
    BCU(cudaMemcpyAsync(scan, d_scan, sizeof scan, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    BCU(cudaGetLastError());
    *bad = scan[0] != 0;
    // every node box lies inside the vertices' bounds: if their extent is finite on every axis, so is every extent the encoder sees
    for (int a = 0; a < 3 && n_tris && !*bad; a++) {
        const float ext = o2f(scan[4 + a]) - o2f(scan[1 + a]);
        *bad = !std::isfinite(ext);
    }
    return 0;
}

int refit_run(const RefitTopology& t, const float* d_tris9, uint64_t n_tris, const uint32_t* d_prim_indices, uint32_t tri_stride,
              void* d_nodes, void* d_tris, const uint32_t* d_blas, bool blas_only, cudaStream_t st, bool* exact, char* err, size_t errlen) {
    const uint32_t n = (uint32_t)n_tris;
    uint8_t* tri_out = static_cast<uint8_t*>(d_tris);
    uint32_t* flag = t.d_flag.get();
    BCU(cudaMemsetAsync(flag, 0, 4, st));
    if (n) {
#define TRIS(S) refit_tris_kernel<S><<<blocks(n), TPB, 0, st>>>(d_tris9, n, d_prim_indices, tri_out, t.d_slot_box.get())
        if (tri_stride == 64) TRIS(64); else if (tri_stride == 24) TRIS(24); else TRIS(48);
#undef TRIS
    }
    uint4* nodes = static_cast<uint4*>(d_nodes);
    const uint32_t n_levels = (uint32_t)t.level_off.size() - 1;
    const uint2* items = t.d_items.get();
    int4 *node_box = t.d_node_box.get(), *slot_box = t.d_slot_box.get();
    // BLAS (or flat) levels deepest first, then the TLAS over the BLAS roots' boxes
    for (uint32_t part = 0; part < (blas_only ? 1u : 2u); part++) {
        const uint32_t first = part == 0 ? 0 : t.n_blas_levels, last = part == 0 ? t.n_blas_levels : n_levels;
        for (uint32_t L = last; L-- > first;) {
            const uint32_t begin = t.level_off[L], cnt = t.level_off[L + 1] - begin;
            if (part == 0) refit_node_kernel<false><<<blocks(cnt), TPB, 0, st>>>(items + begin, cnt, nodes, node_box, slot_box, d_blas, flag);
            else refit_node_kernel<true><<<blocks(cnt), TPB, 0, st>>>(items + begin, cnt, nodes, node_box, slot_box, d_blas, flag);
        }
    }
    BCU(cudaGetLastError());
    uint32_t f = 0;
    BCU(cudaMemcpyAsync(&f, flag, 4, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    BCU(cudaGetLastError());
    *exact = f != 0 || (blas_only ? t.unreached_exact_blas : t.unreached_exact);
    return 0;
}

size_t tlas_arena_bytes(uint32_t n_instances) { return (size_t)n_instances * 384 + (16u << 20); }

int refit_reserve(RefitTopology& t, uint64_t cap, uint32_t n_instances, cudaStream_t st, char* err, size_t errlen) {
    if (tlas_arena_bytes(n_instances) > t.tlas_arena_bytes) {
        const size_t bytes = tlas_arena_bytes(n_instances);
        t.d_tlas_arena.reset();
        t.bytes -= t.tlas_arena_bytes;
        t.tlas_arena_bytes = 0;
        BCU(dev_alloc(t.d_tlas_arena, bytes));
        t.tlas_arena_bytes = bytes;
        t.bytes += bytes;
    }
    if (cap <= t.cap) return 0;
    DevPtr<uint2> items; DevPtr<int4> box;
    BCU(dev_alloc(items, cap * sizeof(uint2)));
    BCU(dev_alloc(box, cap * 2 * sizeof(int4)));
    BCU(cudaMemcpyAsync(items.get(), t.d_items.get(), (size_t)t.level_off.back() * sizeof(uint2), cudaMemcpyDeviceToDevice, st));
    BCU(cudaStreamSynchronize(st));
    t.d_items = std::move(items); t.d_node_box = std::move(box);
    t.bytes += (cap - t.cap) * (sizeof(uint2) + 2 * sizeof(int4));
    t.cap = cap;
    return 0;
}

int rebuild_tlas(RefitTopology& t, void* d_nodes, uint32_t tlas_start, uint32_t n, uint32_t* d_blas, uint32_t max_leaf, uint32_t radius,
                 cudaStream_t st, cudaEvent_t written, uint32_t* n_tlas_nodes, bool* exact, char* err, size_t errlen,
                 const InstanceTlas* inst) {
    if ((uint64_t)tlas_start + n + 1 > t.cap) { snprintf(err, errlen, "the topology holds %llu nodes", (unsigned long long)t.cap); return -3; }
    const int r = (int)(radius < 1 ? 1 : (radius > 64 ? 64 : radius));
    if (!t.d_tlas_arena) { snprintf(err, errlen, "no TLAS build arena (refit_reserve first)"); return -3; }
    Scratch sc(t.d_tlas_arena.get(), t.tlas_arena_bytes);
    float4 *tlo, *thi; uint32_t* perm;
    BCU(sc.alloc(&tlo, (size_t)n * 16)); BCU(sc.alloc(&thi, (size_t)n * 16)); BCU(sc.alloc(&perm, (size_t)n * 4));
    if (inst) {
        BCU(cudaMemcpyAsync(tlo, inst->h_lo, (size_t)n * 16, cudaMemcpyHostToDevice, st));
        BCU(cudaMemcpyAsync(thi, inst->h_hi, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    } else {
        tlas_boxes_kernel<<<blocks(n), TPB, 0, st>>>(t.d_canon.get(), n, t.d_node_box.get(), tlo, thi);
    }
    TlasOut to;
    if (const int rc = tlas_run(sc, tlo, thi, n, max_leaf, r, reinsert_knobs(), static_cast<uint8_t*>(d_nodes) + (uint64_t)tlas_start * 80, perm,
                                st, &to, err, errlen)) return rc;
    if (inst) instance_compose_kernel<<<blocks(n), TPB, 0, st>>>(perm, inst->d_in, n, d_blas, inst->d_rec);
    else blas_compose_kernel<<<blocks(n), TPB, 0, st>>>(perm, t.d_canon.get(), n, d_blas);
    BCU(cudaGetLastError());
    if (written) BCU(cudaEventRecord(written, st));
    // the BLAS levels stay; the TLAS levels become those of the new tree, every node of which is reached
    t.level_off.resize(t.n_blas_levels + 1);
    const uint32_t base = t.level_off.back();
    tlas_items_kernel<<<blocks(to.n_nodes), TPB, 0, st>>>(t.d_items.get() + base, to.n_nodes, tlas_start);
    for (uint32_t e : to.co.level_end) t.level_off.push_back(base + e);
    t.unreached_exact = t.unreached_exact_blas;
    BCU(cudaStreamSynchronize(st));
    BCU(cudaGetLastError());
    *n_tlas_nodes = to.n_nodes; *exact = to.co.force_exact;
    return 0;
}

int root_nodes(const RefitTopology& t, const void* d_nodes, cudaStream_t st, std::vector<uint4>* out, char* err, size_t errlen) {
    const uint32_t n = (uint32_t)t.roots.size();
    out->assign((size_t)n * 5, make_uint4(0, 0, 0, 0));
    if (!n) return 0;
    gather_nodes_kernel<<<blocks(n), TPB, 0, st>>>(static_cast<const uint4*>(d_nodes), t.d_roots.get(), n, t.d_root_nodes.get());
    BCU(cudaGetLastError());
    BCU(cudaMemcpyAsync(out->data(), t.d_root_nodes.get(), (size_t)n * 80, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    return 0;
}

int blas_exact(const RefitTopology& t, const void* d_nodes, uint32_t tlas_start, cudaStream_t st, bool* exact, char* err, size_t errlen) {
    uint32_t* flag = t.d_flag.get();
    BCU(cudaMemsetAsync(flag, 0, 4, st));
    if (tlas_start) exact_scan_kernel<<<blocks(tlas_start), TPB, 0, st>>>(static_cast<const uint4*>(d_nodes), tlas_start, flag);
    BCU(cudaGetLastError());
    uint32_t f = 0;
    BCU(cudaMemcpyAsync(&f, flag, 4, cudaMemcpyDeviceToHost, st));
    BCU(cudaStreamSynchronize(st));
    *exact = f != 0;
    return 0;
}

}  // namespace tray_build
