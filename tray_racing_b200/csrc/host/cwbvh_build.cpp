// cwbvh_build.cpp — host-side CWBVH producer for the tray_cuda backend (CPU, C++17, OpenMP).
//
// Role: the reference gets its CwBvh from obvhs' PLOC builder (`cwbvh_from_tris` src/cwbvh.rs:24-105,
// `tlas_from_blas` src/cwbvh.rs:108-137), an external crate that cannot be built here.  This file is NOT a
// port of PLOC: it is an independent binned-SAH BVH2 -> greedy 8-wide collapse that EMITS THE SAME
// FORMAT — the 80-byte CwBvhNode contract pinned in-tree by the traversal shader
// (src/rt_gpu/rt_gpu_software_query.hlsl:213-303,370-387) and by the in-tree encoder
// (embree/src/bvh_embree_to_cwbvh.rs:85-186: p / exponent / floor-ceil quantisation / child_meta
// encoding / contiguous inner children; embree/src/bvh_embree.rs:284-349: children placed by octant).
// It exists so that the traversal kernel has valid inputs at every BASELINE.json scene size; a real obvhs
// dump can replace its output byte for byte (INTEGRATION.md).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "tray_host.h"

namespace {

// min / max that order -0.0 below +0.0 whichever argument comes first, as the device builder's fminf / fmaxf do: a node's
// p is the minimum of its primitives bit for bit, sign of zero included (std::min keeps its first argument on a tie)
inline float min_z(float a, float b) { return (b < a || (b == a && std::signbit(b))) ? b : a; }
inline float max_z(float a, float b) { return (b > a || (b == a && !std::signbit(b))) ? b : a; }

struct Box {
    float mn[3], mx[3];
    void reset() {
        for (int a = 0; a < 3; a++) { mn[a] = std::numeric_limits<float>::max(); mx[a] = -std::numeric_limits<float>::max(); }
    }
    void grow(const Box& o) {
        for (int a = 0; a < 3; a++) { mn[a] = min_z(mn[a], o.mn[a]); mx[a] = max_z(mx[a], o.mx[a]); }
    }
    void grow(const float p[3]) {
        for (int a = 0; a < 3; a++) { mn[a] = min_z(mn[a], p[a]); mx[a] = max_z(mx[a], p[a]); }
    }
    float half_area() const {
        float dx = mx[0] - mn[0], dy = mx[1] - mn[1], dz = mx[2] - mn[2];
        if (dx < 0 || dy < 0 || dz < 0) return 0.f;
        return dx * dy + dy * dz + dz * dx;
    }
};

struct Node2 {            // binary BVH node over a contiguous range of `order`
    Box box;
    uint32_t left, right; // children (inner) — valid when count > leaf threshold and !is_leaf
    uint32_t first, count;
    uint32_t is_leaf;
};

constexpr int kBins = 16;

struct Builder2 {
    const Box* prim;          // primitive boxes
    std::vector<float> cen;   // centroids, 3 per primitive
    std::vector<uint32_t> order;
    std::vector<Node2> nodes;
    std::atomic<uint32_t> next{0};

    uint32_t alloc() { return next.fetch_add(1, std::memory_order_relaxed); }

    void build(uint32_t ni) {
        Node2& n = nodes[ni];
        const uint32_t first = n.first, count = n.count;
        if (count == 1) { n.is_leaf = 1; return; }
        // centroid bounds
        float cmn[3] = { 1e38f, 1e38f, 1e38f }, cmx[3] = { -1e38f, -1e38f, -1e38f };
        for (uint32_t i = first; i < first + count; i++) {
            const float* c = &cen[3 * (size_t)order[i]];
            for (int a = 0; a < 3; a++) { cmn[a] = std::min(cmn[a], c[a]); cmx[a] = std::max(cmx[a], c[a]); }
        }
        float ext[3] = { cmx[0] - cmn[0], cmx[1] - cmn[1], cmx[2] - cmn[2] };
        uint32_t mid = 0;
        bool have_split = false;
        if (ext[0] > 0 || ext[1] > 0 || ext[2] > 0) {
            // binned SAH on all three axes in one pass
            Box bbox[3][kBins]; uint32_t bcnt[3][kBins];
            for (int a = 0; a < 3; a++) for (int b = 0; b < kBins; b++) { bbox[a][b].reset(); bcnt[a][b] = 0; }
            float scale[3];
            for (int a = 0; a < 3; a++) scale[a] = ext[a] > 0 ? (float)kBins * (1.f - 1e-6f) / ext[a] : 0.f;
            for (uint32_t i = first; i < first + count; i++) {
                const uint32_t p = order[i];
                const float* c = &cen[3 * (size_t)p];
                for (int a = 0; a < 3; a++) {
                    if (ext[a] <= 0) continue;
                    int b = std::min(kBins - 1, std::max(0, (int)((c[a] - cmn[a]) * scale[a])));
                    bbox[a][b].grow(prim[p]); bcnt[a][b]++;
                }
            }
            float best = std::numeric_limits<float>::max(); int best_axis = -1, best_bin = -1;
            for (int a = 0; a < 3; a++) {
                if (ext[a] <= 0) continue;
                float right_area[kBins]; uint32_t right_cnt[kBins];
                Box acc; acc.reset(); uint32_t c = 0;
                for (int b = kBins - 1; b > 0; b--) {
                    if (bcnt[a][b]) acc.grow(bbox[a][b]);
                    c += bcnt[a][b]; right_area[b] = acc.half_area(); right_cnt[b] = c;
                }
                acc.reset(); c = 0;
                for (int b = 0; b < kBins - 1; b++) {
                    if (bcnt[a][b]) acc.grow(bbox[a][b]);
                    c += bcnt[a][b];
                    if (c == 0 || right_cnt[b + 1] == 0) continue;
                    float cost = acc.half_area() * (float)c + right_area[b + 1] * (float)right_cnt[b + 1];
                    if (cost < best) { best = cost; best_axis = a; best_bin = b; }
                }
            }
            if (best_axis >= 0) {
                const int a = best_axis; const float s = scale[a], lo = cmn[a];
                uint32_t* beg = &order[first];
                uint32_t* m = std::partition(beg, beg + count, [&](uint32_t p) {
                    int b = std::min(kBins - 1, std::max(0, (int)((cen[3 * (size_t)p + a] - lo) * s)));
                    return b <= best_bin;
                });
                mid = (uint32_t)(m - beg);
                have_split = mid > 0 && mid < count;
            }
        }
        if (!have_split) {
            // coincident centroids (or a degenerate binning): object-median split, or a multi-primitive leaf
            if (count <= 3 && !(ext[0] > 0 || ext[1] > 0 || ext[2] > 0)) { n.is_leaf = 1; return; }
            int a = ext[0] >= ext[1] ? (ext[0] >= ext[2] ? 0 : 2) : (ext[1] >= ext[2] ? 1 : 2);
            mid = count / 2;
            uint32_t* beg = &order[first];
            std::nth_element(beg, beg + mid, beg + count, [&](uint32_t x, uint32_t y) {
                return cen[3 * (size_t)x + a] < cen[3 * (size_t)y + a];
            });
        }
        const uint32_t l = alloc(), r = alloc();
        Node2& nn = nodes[ni];
        nn.left = l; nn.right = r; nn.is_leaf = 0;
        Node2& ln = nodes[l]; Node2& rn = nodes[r];
        ln.first = first; ln.count = mid; rn.first = first + mid; rn.count = count - mid;
        ln.box.reset(); rn.box.reset();
        for (uint32_t i = first; i < first + mid; i++) ln.box.grow(prim[order[i]]);
        for (uint32_t i = first + mid; i < first + count; i++) rn.box.grow(prim[order[i]]);
        ln.left = ln.right = rn.left = rn.right = 0; ln.is_leaf = rn.is_leaf = 0;
        if (count > 8192) {
#pragma omp task default(shared) firstprivate(l)
            build(l);
#pragma omp task default(shared) firstprivate(r)
            build(r);
#pragma omp taskwait
        } else {
            build(l); build(r);
        }
    }
};

// smallest power of two 2^k with 255 * 2^k >= extent  (bvh_embree_to_cwbvh.rs:97-110: exp2(ceil(log2(extent/255))))
int quant_exponent(float extent) {
    extent = std::max(extent, 1e-20f);
    int k = (int)std::ceil(std::log2((double)extent / 255.0));
    while (std::ldexp(255.0, k) < (double)extent) k++;
    while (std::ldexp(255.0, k - 1) >= (double)extent) k--;
    return k;
}

struct Collapser {
    const Builder2& b2;
    uint32_t max_leaf;
    std::vector<tray_cwbvh_node> out;
    std::vector<uint32_t> prim_out;
    uint32_t max_depth = 0;

    Collapser(const Builder2& b, uint32_t ml) : b2(b), max_leaf(ml) {}

    void run(uint32_t root2) {
        struct Item { uint32_t out_idx, n2, depth; };
        std::vector<Item> stack;
        out.emplace_back(); std::memset(&out[0], 0, sizeof(tray_cwbvh_node));
        stack.push_back({ 0, root2, 1 });
        while (!stack.empty()) {
            Item it = stack.back(); stack.pop_back();
            max_depth = std::max(max_depth, it.depth);
            uint32_t kids[8]; int nk = 0;
            const Node2& n = b2.nodes[it.n2];
            if (n.count <= max_leaf || n.is_leaf) { kids[nk++] = it.n2; }   // tiny scene: root is one leaf child
            else { kids[nk++] = n.left; kids[nk++] = n.right; }
            // phase 1: open the largest-area subtree that MUST be an inner child (more than max_leaf prims)
            // phase 2: use free slots to split small subtrees into tighter leaves
            for (int phase = 0; phase < 2; phase++) {
                while (nk < 8) {
                    int best = -1; float best_a = -1.f;
                    for (int i = 0; i < nk; i++) {
                        const Node2& c = b2.nodes[kids[i]];
                        if (c.is_leaf) continue;
                        bool big = c.count > max_leaf;
                        if ((phase == 0) != big) continue;
                        float a = c.box.half_area() * (phase == 0 ? 1.f : (float)c.count);
                        if (a > best_a) { best_a = a; best = i; }
                    }
                    if (best < 0) break;
                    const Node2& c = b2.nodes[kids[best]];
                    kids[best] = c.left; kids[nk++] = c.right;
                }
            }
            // place children into slots by octant (bvh_embree.rs:284-349: greedy min-cost assignment of
            // (child centre - node centre) . (+-1,+-1,+-1); slot bit 4 = -x, 2 = -y, 1 = -z)
            float ctr[3]; for (int a = 0; a < 3; a++) ctr[a] = 0.5f * (n.box.mn[a] + n.box.mx[a]);
            float cost[8][8];
            for (int c = 0; c < nk; c++) {
                const Box& cb = b2.nodes[kids[c]].box;
                float d[3]; for (int a = 0; a < 3; a++) d[a] = 0.5f * (cb.mn[a] + cb.mx[a]) - ctr[a];
                for (int s = 0; s < 8; s++)
                    cost[c][s] = d[0] * ((s & 4) ? -1.f : 1.f) + d[1] * ((s & 2) ? -1.f : 1.f) + d[2] * ((s & 1) ? -1.f : 1.f);
            }
            int slot_of[8]; bool child_done[8] = {}, slot_used[8] = {};
            int slot_child[8]; for (int s = 0; s < 8; s++) slot_child[s] = -1;
            for (int k = 0; k < nk; k++) {
                float bc = std::numeric_limits<float>::max(); int bi = -1, bs = -1;
                for (int c = 0; c < nk; c++) if (!child_done[c])
                    for (int s = 0; s < 8; s++) if (!slot_used[s] && cost[c][s] < bc) { bc = cost[c][s]; bi = c; bs = s; }
                child_done[bi] = true; slot_used[bs] = true; slot_of[bi] = bs; slot_child[bs] = bi;
            }
            (void)slot_of;
            // encode (bvh_embree_to_cwbvh.rs:85-186)
            tray_cwbvh_node node; std::memset(&node, 0, sizeof(node));
            int ke[3]; double scale[3];
            for (int a = 0; a < 3; a++) {
                node.p[a] = n.box.mn[a];
                ke[a] = quant_exponent(n.box.mx[a] - n.box.mn[a]);
                node.e[a] = (uint8_t)(ke[a] + 127);
                scale[a] = std::ldexp(1.0, ke[a]);
            }
            node.child_base_idx = (uint32_t)out.size();
            node.primitive_base_idx = (uint32_t)prim_out.size();
            uint32_t tri_off = 0; uint32_t n_inner = 0;
            uint8_t* qlo[3] = { node.child_min_x, node.child_min_y, node.child_min_z };
            uint8_t* qhi[3] = { node.child_max_x, node.child_max_y, node.child_max_z };
            uint32_t inner_n2[8];
            for (int s = 0; s < 8; s++) {
                if (slot_child[s] < 0) continue;
                const Node2& c = b2.nodes[kids[slot_child[s]]];
                for (int a = 0; a < 3; a++) {
                    double lo = std::floor(((double)c.box.mn[a] - (double)node.p[a]) / scale[a]);
                    double hi = std::ceil(((double)c.box.mx[a] - (double)node.p[a]) / scale[a]);
                    lo = std::min(255.0, std::max(0.0, lo)); hi = std::min(255.0, std::max(0.0, hi));
                    qlo[a][s] = (uint8_t)lo; qhi[a][s] = (uint8_t)hi;
                }
                if (c.count > max_leaf && !c.is_leaf) {
                    node.imask |= (uint8_t)(1u << s);
                    node.child_meta[s] = (uint8_t)((24 + s) | 0x20);
                    inner_n2[n_inner++] = kids[slot_child[s]];
                } else {
                    static const uint8_t unary[4] = { 0, 0x20, 0x60, 0xE0 };
                    node.child_meta[s] = (uint8_t)(unary[c.count] | tri_off);
                    for (uint32_t i = 0; i < c.count; i++) prim_out.push_back(b2.order[c.first + i]);
                    tri_off += c.count;
                }
            }
            out[it.out_idx] = node;
            const uint32_t base = (uint32_t)out.size();
            out.resize(out.size() + n_inner);
            for (uint32_t i = n_inner; i-- > 0;) stack.push_back({ base + i, inner_n2[i], it.depth + 1 });
        }
    }
};

}  // namespace

struct tray_cwbvh {
    std::vector<tray_cwbvh_node> nodes;
    std::vector<uint32_t> prim_indices;
    float aabb_min[3], aabb_max[3];
    uint32_t max_depth;
};

extern "C" {

int tray_host_build_cwbvh_from_aabbs(const float* bmin, const float* bmax, uint64_t n,
                                     uint32_t max_prims_per_leaf, int nthreads, tray_cwbvh** out) {
    if (!out || (n && (!bmin || !bmax)) || max_prims_per_leaf < 1 || max_prims_per_leaf > 3 || n >= 0x7fffffffull)
        return -1;
    tray_cwbvh* h = new tray_cwbvh();
    h->max_depth = 0;
    for (int a = 0; a < 3; a++) { h->aabb_min[a] = 0; h->aabb_max[a] = 0; }
    *out = h;
    if (n == 0) return 0;
    std::vector<Box> prim(n);
    Builder2 b; b.prim = prim.data();
    b.cen.resize(3 * n); b.order.resize(n);
    Box all; all.reset();
    for (uint64_t i = 0; i < n; i++) {
        for (int a = 0; a < 3; a++) {
            prim[i].mn[a] = bmin[3 * i + a]; prim[i].mx[a] = bmax[3 * i + a];
            b.cen[3 * i + a] = 0.5f * (prim[i].mn[a] + prim[i].mx[a]);
        }
        b.order[i] = (uint32_t)i;
        all.grow(prim[i]);
    }
    b.nodes.resize(2 * n);
    uint32_t root = b.alloc();
    b.nodes[root].box = all; b.nodes[root].first = 0; b.nodes[root].count = (uint32_t)n;
    b.nodes[root].left = b.nodes[root].right = 0; b.nodes[root].is_leaf = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
#pragma omp single nowait
#endif
    b.build(root);
    Collapser c(b, max_prims_per_leaf);
    c.out.reserve(n / 2 + 16); c.prim_out.reserve(n);
    c.run(root);
    h->nodes.swap(c.out); h->prim_indices.swap(c.prim_out);
    h->max_depth = c.max_depth;
    for (int a = 0; a < 3; a++) { h->aabb_min[a] = all.mn[a]; h->aabb_max[a] = all.mx[a]; }
    return 0;
}

int tray_host_build_cwbvh_from_tris(const float* tris9, uint64_t n, uint32_t max_prims_per_leaf,
                                    int nthreads, tray_cwbvh** out) {
    if (n && !tris9) return -1;
    std::vector<float> mn(3 * n), mx(3 * n);
    for (uint64_t i = 0; i < n; i++) {
        const float* t = tris9 + 9 * i;
        for (int a = 0; a < 3; a++) {
            mn[3 * i + a] = min_z(t[a], min_z(t[3 + a], t[6 + a]));
            mx[3 * i + a] = max_z(t[a], max_z(t[3 + a], t[6 + a]));
        }
    }
    return tray_host_build_cwbvh_from_aabbs(mn.data(), mx.data(), n, max_prims_per_leaf, nthreads, out);
}

uint64_t tray_host_cwbvh_node_count(const tray_cwbvh* h) { return h ? h->nodes.size() : 0; }
uint64_t tray_host_cwbvh_prim_count(const tray_cwbvh* h) { return h ? h->prim_indices.size() : 0; }
uint32_t tray_host_cwbvh_max_depth(const tray_cwbvh* h) { return h ? h->max_depth : 0; }
const tray_cwbvh_node* tray_host_cwbvh_nodes(const tray_cwbvh* h) { return h ? h->nodes.data() : nullptr; }
const uint32_t* tray_host_cwbvh_prim_indices(const tray_cwbvh* h) { return h ? h->prim_indices.data() : nullptr; }
void tray_host_cwbvh_aabb(const tray_cwbvh* h, float mn[3], float mx[3]) {
    for (int a = 0; a < 3; a++) { mn[a] = h->aabb_min[a]; mx[a] = h->aabb_max[a]; }
}
void tray_host_cwbvh_free(tray_cwbvh* h) { delete h; }

// Structural check in the spirit of obvhs `bvh.validate` (called at src/cwbvh.rs:102-104): every primitive
// is referenced exactly once, every decoded child box contains the primitives below it (conservative
// quantisation, bvh_embree_to_cwbvh.rs:135-148), <= 24 triangles per node (:167), meta encodings are
// well-formed, and the group-stack depth needed by the traversal stays within `stack_limit`.
int tray_host_cwbvh_validate(const tray_cwbvh_node* nodes, uint64_t n_nodes, const uint32_t* prim_indices,
                             uint64_t n_prims, const float* prim_min, const float* prim_max,
                             uint32_t stack_limit, tray_validate_report* rep) {
    tray_validate_report r; std::memset(&r, 0, sizeof(r));
    if (n_nodes == 0) { if (rep) *rep = r; return n_prims == 0 ? 0 : -1; }
    std::vector<uint8_t> seen(n_prims, 0), node_seen(n_nodes, 0);
    struct Item { uint32_t idx; uint32_t depth; float mn[3], mx[3]; bool has_box; uint32_t stack_need; };
    std::vector<Item> st; Item root{}; root.idx = 0; root.depth = 1; root.has_box = false; root.stack_need = 0;
    st.push_back(root);
    int rc = 0;
    while (!st.empty()) {
        Item it = st.back(); st.pop_back();
        if (it.idx >= n_nodes) { r.bad_child_index++; rc = -1; continue; }
        if (node_seen[it.idx]++) { r.node_visited_twice++; rc = -1; continue; }
        r.nodes_reached++;
        r.max_depth = std::max(r.max_depth, it.depth);
        r.max_stack = std::max(r.max_stack, it.stack_need);
        const tray_cwbvh_node& n = nodes[it.idx];
        double sc[3];
        for (int a = 0; a < 3; a++) { uint32_t bits = (uint32_t)n.e[a] << 23; float f; std::memcpy(&f, &bits, 4); sc[a] = f; }
        const uint8_t* qlo[3] = { n.child_min_x, n.child_min_y, n.child_min_z };
        const uint8_t* qhi[3] = { n.child_max_x, n.child_max_y, n.child_max_z };
        uint32_t tri_total = 0, inner_rank = 0, n_children = 0;
        uint32_t n_inner = (uint32_t)__builtin_popcount(n.imask);
        for (int s = 0; s < 8; s++) {
            uint8_t m = n.child_meta[s];
            bool inner = (n.imask >> s) & 1;
            if (m == 0) { if (inner) { r.bad_meta++; rc = -1; } continue; }
            n_children++;
            float cmn[3], cmx[3];
            for (int a = 0; a < 3; a++) {
                if (qlo[a][s] > qhi[a][s]) { r.bad_quant++; rc = -1; }
                cmn[a] = (float)((double)n.p[a] + qlo[a][s] * sc[a]);
                cmx[a] = (float)((double)n.p[a] + qhi[a][s] * sc[a]);
            }
            if (inner) {
                if (m != (uint8_t)(0x20 | (24 + s))) { r.bad_meta++; rc = -1; }
                Item c{}; c.idx = n.child_base_idx + inner_rank; c.depth = it.depth + 1; c.has_box = true;
                // group-stack need: one entry is pushed per level whenever siblings remain
                c.stack_need = it.stack_need + (n_inner > 1 ? 1u : 0u);
                // culling happens against every ancestor's decoded box: carry the intersection down
                for (int a = 0; a < 3; a++) {
                    c.mn[a] = it.has_box ? std::max(it.mn[a], cmn[a]) : cmn[a];
                    c.mx[a] = it.has_box ? std::min(it.mx[a], cmx[a]) : cmx[a];
                }
                st.push_back(c); inner_rank++;
            } else {
                uint32_t cnt = (m >> 5) == 1 ? 1 : (m >> 5) == 3 ? 2 : (m >> 5) == 7 ? 3 : 0;
                uint32_t off = m & 0x1f;
                if (cnt == 0 || off + cnt > 24) { r.bad_meta++; rc = -1; continue; }
                tri_total += cnt;
                for (uint32_t k = 0; k < cnt; k++) {
                    uint64_t slot = (uint64_t)n.primitive_base_idx + off + k;
                    if (slot >= n_prims) { r.bad_prim_index++; rc = -1; continue; }
                    uint32_t p = prim_indices ? prim_indices[slot] : (uint32_t)slot;
                    if (p >= n_prims) { r.bad_prim_index++; rc = -1; continue; }
                    if (seen[p]++) { r.prim_seen_twice++; rc = -1; }
                    r.prims_reached++;
                    if (prim_min && prim_max) {
                        for (int a = 0; a < 3; a++) {
                            if (prim_min[3 * (size_t)p + a] < cmn[a] || prim_max[3 * (size_t)p + a] > cmx[a]) { r.box_violations++; rc = -1; break; }
                            // and, transitively, inside every ancestor's decoded box
                            if (it.has_box && (prim_min[3 * (size_t)p + a] < it.mn[a] || prim_max[3 * (size_t)p + a] > it.mx[a])) { r.box_violations++; rc = -1; break; }
                        }
                    }
                }
            }
        }
        if (tri_total > 24) { r.bad_meta++; rc = -1; }
        r.children_total += n_children; r.leaf_children += n_children - n_inner;
    }
    for (uint64_t i = 0; i < n_prims; i++) if (!seen[i]) { r.prims_missing++; rc = -1; }
    if (r.nodes_reached != n_nodes) { r.nodes_unreached = n_nodes - r.nodes_reached; rc = -1; }
    if (stack_limit && r.max_stack + 2 > stack_limit) { r.stack_too_deep = 1; rc = -1; }
    if (rep) *rep = r;
    return rc;
}

}  // extern "C"
