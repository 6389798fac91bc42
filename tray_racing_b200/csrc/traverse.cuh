// traverse.cuh — sm_100a device code: 8-wide CWBVH closest-hit traversal + ray/triangle intersection.
//
// Three kernels make a frame (src/rt_cpu/rt_cpu.rs:35-91, rt_gpu_software.hlsl:47-144):
//   raygen_primary_kernel  pixel -> ray, one thread per pixel, fully coalesced   — rt_cpu.rs:38-55
//   trace_kernel           closest hit for a buffer of rays (the hot kernel)     — Traversable::traverse, batch grain
//   raygen_bounce_kernel   hit -> 1-spp cosine bounce ray, COMPACTED to hit pixels — rt_cpu.rs:61-80
// Ray generation is full-width SIMD work with IEEE divisions; keeping it out of the traversal kernel makes the
// per-lane refill of that kernel two 16-byte loads, so idle lanes can be refilled eagerly.
//
// Execution model (B200: 148 SMs, 4 schedulers each; no tensor cores — this is pointer chasing + FP32/ALU):
//   * persistent warps: the grid is sized to the resident-CTA capacity of the chip; idle lanes pull new rays
//     through one warp-aggregated atomicAdd on a global cursor (ray replacement keeps warps full on incoherent rays)
//   * each lane runs the reference's per-ray state machine UNCHANGED (same node order, same triangle order, same
//     shrinking tmax), so (prim, t) is bit-identical to the oracle by construction; only the WARP-level schedule
//     is new: every iteration the warp votes (__ballot_sync/__popc) whether to run a node step or a triangle
//     step, and only lanes whose next action is of that kind take part — no per-lane while-while divergence
//   * 80-byte nodes are fetched as 5 x 16-byte ld.global.nc; 48/64-byte triangles as 3 x 16-byte
//   * the traversal stack lives in shared memory, [entry][thread] so that a warp's accesses are conflict-free;
//     entries past STACK_SMEM spill to a per-thread local array (checked; overflow raises a flag)
//   * all parity-relevant float math uses round-to-nearest intrinsics without FMA contraction, because the
//     reference CPU path (Rust/glam) never fuses (SURVEY.md §7 "bit-level float parity").
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tray_cuda.h"

namespace tray {

#ifndef TRAY_BLOCK_THREADS
#define TRAY_BLOCK_THREADS 128
#endif
constexpr int BLOCK_THREADS = TRAY_BLOCK_THREADS;
#ifndef TRAY_MIN_BLOCKS
#define TRAY_MIN_BLOCKS (1024 / TRAY_BLOCK_THREADS)
#endif
#ifndef TRAY_STACK_SMEM
#define TRAY_STACK_SMEM 12
#endif
constexpr int STACK_SMEM = TRAY_STACK_SMEM;      // entries per thread in shared memory
constexpr int STACK_SPILL = 48 - STACK_SMEM;     // further entries per thread in local memory (total 48 > obvhs' 32, cwbvh.rs:88)
constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t INVALID = 0xffffffffu;
// rows are LUT_ROW = 260 bytes apart: the same hit byte under different octants then falls into different banks (lanes of an
// incoherent warp mostly hold one-bit hit bytes; at a 256-byte pitch they would all collide in banks 0, 1, 2, 4, ...)
constexpr uint32_t LUT_ROW = 260u, LUT_BYTES = 8u * LUT_ROW;
// trace_kernel's ray index: the ray's place in its launch (the host keeps launches below 2^30 rays) and two tag bits
constexpr uint32_t BOUNCE_BIT = 0x80000000u;     // FRAME kernel: a bounce ray, its index is the work item
constexpr uint32_t WIDE_BIT = 0x40000000u;       // RayConst::wide
constexpr uint32_t INDEX_MASK = 0x3fffffffu;
// bits of the device error word (TraceParams::overflow)
constexpr uint32_t ERR_STACK_OVERFLOW = 1u;      // a push past the last of the STACK_SMEM + STACK_SPILL entries
constexpr uint32_t ERR_WATCHDOG = 4u;            // FRAME kernel: the primary hits of a group never arrived
// a launch's cursor block, CURSOR_WORDS 64-bit words: [0] the work cursor (u32), [CURSOR_COUNTERS + N_COUNTERS * k ..] counter slot k
// (rays, nodes, tris, instances, hits; slot 1: the bounce rays of a frame), [CURSOR_N_BOUNCE] the bounce-ray count of a frame (u32)
constexpr uint32_t CURSOR_COUNTERS = 1, N_COUNTERS = 5, CURSOR_N_BOUNCE = 11, CURSOR_WORDS = 16;
constexpr float F32_MAX_ = 3.402823466e+38f;
constexpr float F32_EPS_ = 1.1920929e-7f;     // sampling.hlsl:3
constexpr float BOX_EPS_ = 0.0001f;           // query.hlsl:274

struct FrameParams {
    tray_view view;
    uint32_t width, height, frame_count;
    uint32_t shard_index, shard_count, tiles_x;   // tiles_x = ceil(width / 32)
    uint32_t n_items;                             // padded local pixel count of this shard (multiple of 256)
};

enum ShadeMode { SHADE_NONE = 0, SHADE_PRIMARY = 1, SHADE_BOUNCE = 2, SHADE_OCCLUSION = 3 };

struct TraceParams {
    const uint4* __restrict__ nodes;          // 5 x uint4 per node
    const uint4* __restrict__ tris;           // 3 or 4 x uint4 per triangle
    const uint32_t* __restrict__ blas_offsets;
    uint32_t tlas_start;
    const tray_ray* __restrict__ rays;        // n_work rays
    const uint32_t* __restrict__ ray_item;    // optional: output slot of ray i (compacted bounce rays); NULL = i
    uint32_t n_work;
    const uint32_t* __restrict__ n_work_dev;  // optional: ray count produced on the device (overrides n_work)
    tray_hit* __restrict__ hits_out;
    uchar4* __restrict__ rgba_out;            // optional: compact (item order), or the row-major frame of `frame` when row_major
    uint32_t row_major;
    uint32_t shade_mode;
    uint32_t* __restrict__ cursor;            // work cursor
    unsigned long long* __restrict__ counters;// counter slot (N_COUNTERS; FRAME: two slots) of the cursor block (COUNT builds)
    uint32_t* __restrict__ overflow;          // device error word (ERR_*)
    // optional, COUNT builds: one cost record per ray at its output item (tray_cuda_trace_cost, tray_cuda_scene_set_ray_cost).
    // FRAME kernel: the bounce records follow the n_work primary ones.  An 8-byte member in this slot keeps the 16-byte
    // alignment of the members after it, and with it the generated code of every kernel.
    tray_ray_cost* __restrict__ ray_cost;
    uint32_t k4b;                             // 0x4B000000, passed at run time (see byte_f32)
    uint32_t force_exact;                     // scene has node scales >= 2^40: always take the unfused node test
    float zero;                               // 0.0f, passed at run time (see child_test_fast)
    uint32_t one;                             // 1, passed at run time: keeps the hit-mask accumulation an IMAD on the FMA pipe (see child_test_fast)
    uint32_t refill_min;                      // idle lanes needed before a partial warp refills
    uint32_t tri_weight;                      // vote: triangle phase when n_tri * tri_weight >= n_node
    uint32_t variant;                         // MODE 1 kernels only: TRAY_VARIANT_* switches (tray_cuda_scene_set_variant)
    FrameParams frame;                        // frame launches: camera, frame geometry, frame_count (item -> pixel)
    // FRAME kernel only (one launch per frame: bounce rays of finished 32-item groups start while the primary pass drains)
    tray_hit* __restrict__ bounce_out;        // bounce hits by item
    tray_ray* __restrict__ rays_by_item;      // optional: the generated bounce rays by item (checkers)
    tray_ray* gen_rays;                       // bounce rays by item: written full-width when a group is claimed, read back lane by lane
    uint32_t* __restrict__ unit_cursor;       // next tile whose bounce rays have not been claimed (zeroed by the host)
    uint32_t n_units;                         // n_work / 32: bounce work is claimed in groups of 32 items
    uint32_t gen_min;                         // idle lanes needed before the warp generates bounce rays into them
    // INST kernels only (instanced scenes, tray_cuda_scene_set_instances).  Appended, so that the members above keep their offsets.
    const uint4* __restrict__ inst_rec;       // per TLAS leaf, an InstanceRecord
    uint32_t* __restrict__ inst_out;          // optional: the instance of each hit by output item (INVALID for a miss)
};

// One instance as the device reads it, 64 bytes: rows 0..2 of world_to_object ([W | -W t], 4 floats each), then {BLAS root,
// instance id, 0, 0}.  The TLAS holds one per leaf in leaf order; the scene keeps the same records by instance id for the bounce
// normals.
constexpr uint32_t INST_RECORD_U4 = 4;

// ---- exact float helpers (no contraction, IEEE rounding) --------------------------------------
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    return add(add(mul(ax, bx), mul(ay, by)), mul(az, bz));       // glam: (x*x' + y*y') + z*z'
}
__device__ __forceinline__ void cross3(float ax, float ay, float az, float bx, float by, float bz,
                                       float& ox, float& oy, float& oz) {
    ox = sub(mul(ay, bz), mul(az, by));
    oy = sub(mul(az, bx), mul(ax, bz));
    oz = sub(mul(ax, by), mul(ay, bx));
}
__device__ __forceinline__ void normalize3(float& x, float& y, float& z) {   // glam Vec3A: v / sqrt(dot)
    float len = __fsqrt_rn(dot3(x, y, z, x, y, z));
    x = __fdiv_rn(x, len); y = __fdiv_rn(y, len); z = __fdiv_rn(z, len);
}
// byte J of w as an exact float: PRMT builds 0x4B0000bb = 2^23 + byte, FADD removes 2^23 (no I2F: the
// conversion pipe is quarter-rate).
// `k4b` must be a RUNTIME register holding 0x4B000000 (it comes in through the kernel parameters): SASS PRMT
// takes one immediate, and with the selector as that immediate no per-use MOV of the selector is needed.
template <int J> __device__ __forceinline__ float byte_f32(uint32_t w, uint32_t k4b) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(k4b), "n"(0x7440 + J));
    return __fsub_rn(__uint_as_float(r), 8388608.0f);
}
template <int J> __device__ __forceinline__ uint32_t byte_u32(uint32_t w) {
    uint32_t r;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(r) : "r"(w), "n"(0x4440 + J));
    return r;
}

// ---- per-ray constants ---------------------------------------------------------------------------
struct RayConst {
    float ox, oy, oz, dx, dy, dz, ix, iy, iz, tmin;
    uint32_t oct_inv4;
    uint32_t lut_off;   // shared-memory address of this ray's row of the child-order table: s_lut + (oct_inv & 7) * LUT_ROW
    bool wide;      // |1/d| >= 2^64 on some axis: 2^23 * adj_inv could overflow, use the unfused node test
    // MODE 1 (semantic variants, tray_cuda_scene_set_variant) only — dead registers in every other kernel:
    float tdx, tdy, tdz;    // the direction the TRIANGLE test sees (the caller's, when the zero patch feeds the box test only)
    float box_tmin;         // lower clamp of the slab test: 1e-4 (query.hlsl:274) or ray.tmin
};

__device__ __forceinline__ void prepare_ray(RayConst& r, float ox, float oy, float oz, float dx, float dy, float dz, float tmin,
                                            uint32_t variant = 0u, uint32_t lut_base = 0u) {
    r.ox = ox; r.oy = oy; r.oz = oz; r.tmin = tmin;
    r.dx = dx == 0.0f ? F32_EPS_ : dx;           // query.hlsl:334
    r.dy = dy == 0.0f ? F32_EPS_ : dy;
    r.dz = dz == 0.0f ? F32_EPS_ : dz;
    const bool raw = (variant & TRAY_VARIANT_ZERODIR_BOX_ONLY) != 0u;
    r.tdx = raw ? dx : r.dx; r.tdy = raw ? dy : r.dy; r.tdz = raw ? dz : r.dz;
    r.box_tmin = (variant & TRAY_VARIANT_BOX_TMIN_RAY) ? tmin : BOX_EPS_;
    r.ix = __fdiv_rn(1.0f, r.dx); r.iy = __fdiv_rn(1.0f, r.dy); r.iz = __fdiv_rn(1.0f, r.dz);   // Ray::inv_direction
    r.oct_inv4 = (r.dx < 0.0f ? 0u : 0x04040404u) | (r.dy < 0.0f ? 0u : 0x02020202u) |
                 (r.dz < 0.0f ? 0u : 0x01010101u);                                              // query.hlsl:314-326
    r.lut_off = lut_base + (r.oct_inv4 & 7u) * LUT_ROW;
    r.wide = !(fmaxf(fmaxf(fabsf(r.ix), fabsf(r.iy)), fabsf(r.iz)) < 1.8446744e19f);
}

// ---- packed f32x2 helpers (Blackwell FFMA2 / FADD2: two IEEE-rounded results per issue slot) --------
__device__ __forceinline__ unsigned long long pack2(uint32_t lo, uint32_t hi) {
    unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r;
}
__device__ __forceinline__ unsigned long long pack2f(float lo, float hi) { return pack2(__float_as_uint(lo), __float_as_uint(hi)); }
__device__ __forceinline__ void unpack2f(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r;
}
__device__ __forceinline__ unsigned long long fadd2(unsigned long long a, unsigned long long b) {
    unsigned long long r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r;
}
template <int J> __device__ __forceinline__ uint32_t byte_biased(uint32_t w, uint32_t k4b) {   // 0x4B0000bb = 2^23 + byte
    uint32_t r; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(k4b), "n"(0x7440 + J)); return r;
}
// byte J of w as an exact float on the conversion (XU) pipe: I2F.U8 with a byte selector.  Quarter-rate, but
// that pipe is otherwise idle here, so a few conversions per child run there concurrently with the ALU pipe.
template <int J> __device__ __forceinline__ float byte_i2f(uint32_t w) { return (float)((w >> (8 * J)) & 0xffu); }

// ---- node test: CwBvhNode::intersect_ray, twin query.hlsl:213-303, in slot space ------------------------------
// The lane kernel keeps the top byte of the hit mask / node group word in SLOT space: an inner child (bit_index = 24 + slot,
// query.hlsl:251-262) sets bit 24 + slot, WITHOUT the octant XOR.  That XOR exists so that firstbithigh (query.hlsl:358) finds
// the hit child nearest along the ray, and `slot = bit ^ oct_inv` (:370) undoes it; here the pair becomes ONE lookup when the
// next child is chosen: child_order[oct_inv][hit byte] = the hit slot whose (slot ^ oct_inv) is largest (2 KB table in shared
// memory, built at kernel start).  Same child, same order, same `rel` (query.hlsl:371 counts imask bits below `slot`: slot space
// already).  The node test drops is_inner4 / inner_mask4 / the XOR (query.hlsl:251-257): child_bits << bit_index is the whole
// contribution of a hit child (:291-298), for leaves (bit_index = triangle offset) and inner children alike.
// (A fully pre-decoded 128-byte node, one 32-bit word per child, was built and measured — profiles/experiments/r2_tnode_*: node
// test 215 -> 172 instructions, but 60 % more L1 traffic; the L1 serves scattered 16-byte accesses at ~32 B/clk/SM, it went from
// 42 % to 75 % busy and the incoherent bounce rays of C3 got 5 % slower.  The node stays the caller's 80 bytes.)

// child_order[oi][t]: of the slots set in the hit byte t, the one whose (slot ^ oi) is largest (t = 0: unused)
__device__ __forceinline__ void child_order_fill(uint8_t* lut, unsigned tid, unsigned n_threads) {
    for (unsigned k = tid; k < 2048u; k += n_threads) {
        const unsigned oi = k >> 8, t = k & 255u;
        unsigned best = 0, best_key = 0;
        for (unsigned j = 0; j < 8u; j++)
            if (((t >> j) & 1u) && ((j ^ oi) >= best_key)) { best_key = j ^ oi; best = j; }
        lut[oi * LUT_ROW + t] = (uint8_t)best;
    }
}

// exact (unfused) form (wide rays, huge node scales, MODE 1)
template <int J>
__device__ __forceinline__ uint32_t child_test(uint32_t nx, uint32_t fx, uint32_t ny, uint32_t fy, uint32_t nz, uint32_t fz,
                                               float ax, float ay, float az, float bx, float by, float bz, float tmax,
                                               uint32_t child_bits4, uint32_t meta4, uint32_t k4b, float box_tmin) {
    const float tnx = add(mul(byte_f32<J>(nx, k4b), ax), bx), tfx = add(mul(byte_f32<J>(fx, k4b), ax), bx);
    const float tny = add(mul(byte_f32<J>(ny, k4b), ay), by), tfy = add(mul(byte_f32<J>(fy, k4b), ay), by);
    const float tnz = add(mul(byte_f32<J>(nz, k4b), az), bz), tfz = add(mul(byte_f32<J>(fz, k4b), az), bz);
    const float tmin = fmaxf(fmaxf(fmaxf(tnx, tny), tnz), box_tmin);      // query.hlsl:288
    const float tfar = fminf(fminf(fminf(tfx, tfy), tfz), tmax);          // query.hlsl:289
    const uint32_t contrib = byte_u32<J>(child_bits4) << ((meta4 >> (8 * J)) & 31u);       // query.hlsl:291-298, slot space
    return tmin <= tfar ? contrib : 0u;
}
// `box_tmin` / `divide`: the slab test's lower clamp and the HLSL's divide-by-direction form (query.hlsl:237-242) — MODE 1 only
__device__ __forceinline__ uint32_t node_test(const RayConst& r, float tmax, const uint4& n0, const uint4& n1, const uint4& n2,
                                              const uint4& n3, const uint4& n4, uint32_t k4b, float box_tmin = BOX_EPS_, bool divide = false) {
    const uint32_t e = n0.w;
    const float sx_ = __uint_as_float((e & 0xffu) << 23), sy_ = __uint_as_float(((e >> 8) & 0xffu) << 23), sz_ = __uint_as_float(((e >> 16) & 0xffu) << 23);
    const float px_ = sub(__uint_as_float(n0.x), r.ox), py_ = sub(__uint_as_float(n0.y), r.oy), pz_ = sub(__uint_as_float(n0.z), r.oz);
    const float ax = divide ? __fdiv_rn(sx_, r.dx) : mul(sx_, r.ix);
    const float ay = divide ? __fdiv_rn(sy_, r.dy) : mul(sy_, r.iy);
    const float az = divide ? __fdiv_rn(sz_, r.dz) : mul(sz_, r.iz);
    const float bx = divide ? __fdiv_rn(px_, r.dx) : mul(px_, r.ix);
    const float by = divide ? __fdiv_rn(py_, r.dy) : mul(py_, r.iy);
    const float bz = divide ? __fdiv_rn(pz_, r.dz) : mul(pz_, r.iz);
    const bool sx = r.dx < 0.0f, sy = r.dy < 0.0f, sz = r.dz < 0.0f;
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const uint32_t meta4 = i == 0 ? n1.z : n1.w;
        const uint32_t child_bits4 = (meta4 >> 5) & 0x07070707u;
        const uint32_t lox = i == 0 ? n2.x : n2.y, hix = i == 0 ? n2.z : n2.w;
        const uint32_t loy = i == 0 ? n3.x : n3.y, hiy = i == 0 ? n3.z : n3.w;
        const uint32_t loz = i == 0 ? n4.x : n4.y, hiz = i == 0 ? n4.z : n4.w;
        const uint32_t nx = sx ? hix : lox, fx = sx ? lox : hix;                   // query.hlsl:266-273
        const uint32_t ny = sy ? hiy : loy, fy = sy ? loy : hiy;
        const uint32_t nz = sz ? hiz : loz, fz = sz ? loz : hiz;
        mask |= child_test<0>(nx, fx, ny, fy, nz, fz, ax, ay, az, bx, by, bz, tmax, child_bits4, meta4, k4b, box_tmin);
        mask |= child_test<1>(nx, fx, ny, fy, nz, fz, ax, ay, az, bx, by, bz, tmax, child_bits4, meta4, k4b, box_tmin);
        mask |= child_test<2>(nx, fx, ny, fy, nz, fz, ax, ay, az, bx, by, bz, tmax, child_bits4, meta4, k4b, box_tmin);
        mask |= child_test<3>(nx, fx, ny, fy, nz, fz, ax, ay, az, bx, by, bz, tmax, child_bits4, meta4, k4b, box_tmin);
    }
    return mask;
}

// Fused form, BIT-IDENTICAL to node_test: with f = 2^23 + q (exact, straight out of PRMT) and C = 2^23 * A (exact: a
// power-of-two scaling),  fma(f, A, -C) rounds the exact real value (f - 2^23) * A = q * A once, i.e. it IS fl(q * A) — the
// conversion FADD and the FMUL collapse into one FFMA with no change of rounding.  The following "+ adj_org" stays a separate,
// separately rounded add (query.hlsl:285-286).  (near, far) of one child and axis travel as an f32x2 pair: FFMA2 + FADD2 = 2
// issue slots for what took 6.
// Requires 2^23 * A finite: rays with |1/d| >= 2^64 take node_test instead (RayConst::wide).
// Pipe balance: the ALU pipe is the node test's bottleneck, so the y- and z-plane bytes go through I2F.U8 on the XU pipe instead
// of PRMT (32 conversions per node is the balance point: 24 -> +1.6 %, 32 -> +3.1 %, 40 -> -1.5 %; the x-plane bytes as well is
// slower, the XU pipe saturates).  There q is already the plain float and fma(q, A, 0) = fl(q * A)  (Z0 is a run-time zero so
// that the assembler cannot turn fma+add back into one fused op).
struct NodeConsts { unsigned long long AX, AY, AZ, CX, BX, BY, BZ, Z0; };

template <int J>
__device__ __forceinline__ void child_test_fast(uint32_t& mask, uint32_t nx, uint32_t fx, uint32_t ny, uint32_t fy, uint32_t nz, uint32_t fz,
                                                const NodeConsts& c, float tmax, uint32_t child_bits4, uint32_t meta4, uint32_t k4b, uint32_t one) {
    float tnx, tfx, tny, tfy, tnz, tfz;
    unpack2f(fadd2(ffma2(pack2(byte_biased<J>(nx, k4b), byte_biased<J>(fx, k4b)), c.AX, c.CX), c.BX), tnx, tfx);
    unpack2f(fadd2(ffma2(pack2f(byte_i2f<J>(ny), byte_i2f<J>(fy)), c.AY, c.Z0), c.BY), tny, tfy);
    unpack2f(fadd2(ffma2(pack2f(byte_i2f<J>(nz), byte_i2f<J>(fz)), c.AZ, c.Z0), c.BZ), tnz, tfz);
    const float tmin = fmaxf(fmaxf(fmaxf(tnx, tny), tnz), BOX_EPS_);
    const float tfar = fminf(fminf(fminf(tfx, tfy), tfz), tmax);
    const uint32_t contrib = byte_u32<J>(child_bits4) << ((meta4 >> (8 * J)) & 31u);
    // if (tmin <= tfar) mask |= contrib.  The children's bits are disjoint, so OR = ADD = contrib * 1 + mask: a predicated IMAD on
    // the FMA pipe instead of a LOP3 on the ALU pipe, +1.1 % (profiles/experiments/r2_pipe_balance_ab.log)
    asm("{.reg .pred p; setp.le.f32 p, %1, %2; @p mad.lo.u32 %0, %3, %4, %0;}" : "+r"(mask) : "f"(tmin), "f"(tfar), "r"(contrib), "r"(one));
}
__device__ __forceinline__ void node_half_fast(uint32_t& mask, const RayConst& r, float tmax, const NodeConsts& c, uint32_t meta4,
                                               uint32_t lox, uint32_t hix, uint32_t loy, uint32_t hiy, uint32_t loz, uint32_t hiz, uint32_t k4b, uint32_t one) {
    const uint32_t child_bits4 = (meta4 >> 5) & 0x07070707u;
    const bool sx = r.dx < 0.0f, sy = r.dy < 0.0f, sz = r.dz < 0.0f;
    const uint32_t nx = sx ? hix : lox, fx = sx ? lox : hix;                          // query.hlsl:266-273
    const uint32_t ny = sy ? hiy : loy, fy = sy ? loy : hiy;
    const uint32_t nz = sz ? hiz : loz, fz = sz ? loz : hiz;
    child_test_fast<0>(mask, nx, fx, ny, fy, nz, fz, c, tmax, child_bits4, meta4, k4b, one);
    child_test_fast<1>(mask, nx, fx, ny, fy, nz, fz, c, tmax, child_bits4, meta4, k4b, one);
    child_test_fast<2>(mask, nx, fx, ny, fy, nz, fz, c, tmax, child_bits4, meta4, k4b, one);
    child_test_fast<3>(mask, nx, fx, ny, fy, nz, fz, c, tmax, child_bits4, meta4, k4b, one);
}
__device__ __forceinline__ uint32_t node_test_fast(const RayConst& r, float tmax, const uint4& n0, const uint4& n1, const uint4& n2,
                                                   const uint4& n3, const uint4& n4, uint32_t k4b, float zero, uint32_t one) {
    const uint32_t e = n0.w;
    const float ax = mul(__uint_as_float((e & 0xffu) << 23), r.ix);
    const float ay = mul(__uint_as_float(((e >> 8) & 0xffu) << 23), r.iy);
    const float az = mul(__uint_as_float(((e >> 16) & 0xffu) << 23), r.iz);
    const float bx = mul(sub(__uint_as_float(n0.x), r.ox), r.ix);
    const float by = mul(sub(__uint_as_float(n0.y), r.oy), r.iy);
    const float bz = mul(sub(__uint_as_float(n0.z), r.oz), r.iz);
    const float cx = mul(ax, -8388608.0f);                                                          // -2^23 * A, exact
    NodeConsts c;
    c.AX = pack2f(ax, ax); c.AY = pack2f(ay, ay); c.AZ = pack2f(az, az); c.CX = pack2f(cx, cx);
    c.BX = pack2f(bx, bx); c.BY = pack2f(by, by); c.BZ = pack2f(bz, bz); c.Z0 = pack2f(zero, zero);
    uint32_t mask = 0;
    node_half_fast(mask, r, tmax, c, n1.z, n2.x, n2.z, n3.x, n3.z, n4.x, n4.z, k4b, one);
    node_half_fast(mask, r, tmax, c, n1.w, n2.y, n2.w, n3.y, n3.w, n4.y, n4.w, k4b, one);
    return mask;
}

// ---- triangle records ---------------------------------------------------------------------------
// stride 48 / 64: the CPU path's f32 RtTriangle {v0, e1 = v0 - v1, e2 = v2 - v0 [, ng]} as 3 / 4 x 16-byte loads.
// stride 24: the wgpu path's RtCompressedTriangle {v0: f32 x 3, e[k] = half(v2 - v0)[k] | half(v1 - v0)[k] << 16}
//            (src/rt_gpu/mod.rs:39-43; unpack query.hlsl:75-85, e1 negated at :91) as 3 x 8-byte loads — half the
//            triangle bytes per test, NOT the parity path against rt_cpu (checked against the oracle on the same records).
__device__ __forceinline__ float half_lo(uint32_t w) { return __half2float(__ushort_as_half((unsigned short)(w & 0xffffu))); }
__device__ __forceinline__ float half_hi(uint32_t w) { return __half2float(__ushort_as_half((unsigned short)(w >> 16))); }

template <int TRI_STRIDE>
__device__ __forceinline__ void tri_load(const uint4* __restrict__ tris, uint32_t prim, float& v0x, float& v0y, float& v0z,
                                         float& e1x, float& e1y, float& e1z, float& e2x, float& e2y, float& e2z) {
    if (TRI_STRIDE == 24) {
        const uint2* rec = reinterpret_cast<const uint2*>(tris) + (size_t)prim * 3u;
        const uint2 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
        v0x = __uint_as_float(a.x); v0y = __uint_as_float(a.y); v0z = __uint_as_float(b.x);
        e2x = half_lo(b.y); e2y = half_lo(c.x); e2z = half_lo(c.y);
        e1x = -half_hi(b.y); e1y = -half_hi(c.x); e1z = -half_hi(c.y);
    } else {
        const uint4* rec = tris + (size_t)prim * (TRI_STRIDE / 16);
        const uint4 a = __ldg(rec), b = __ldg(rec + 1), c4 = __ldg(rec + 2);
        v0x = __uint_as_float(a.x); v0y = __uint_as_float(a.y); v0z = __uint_as_float(a.z);
        e1x = __uint_as_float(b.x); e1y = __uint_as_float(b.y); e1z = __uint_as_float(b.z);
        e2x = __uint_as_float(c4.x); e2y = __uint_as_float(c4.y); e2z = __uint_as_float(c4.z);
    }
}

// ---- triangle test: RtTriangle::intersect, twin query.hlsl:89-129; returns t or +inf -------------
// The test's geometric normal (not normalised): the record's for stride 64, cross(e1, e2) otherwise (query.hlsl:93)
template <int TRI_STRIDE>
__device__ __forceinline__ void tri_normal(const uint4* __restrict__ tris, uint32_t prim, float e1x, float e1y, float e1z,
                                           float e2x, float e2y, float e2z, float& ngx, float& ngy, float& ngz) {
    if (TRI_STRIDE == 64) {
        const uint4 g = __ldg(tris + (size_t)prim * 4u + 3);
        ngx = __uint_as_float(g.x); ngy = __uint_as_float(g.y); ngz = __uint_as_float(g.z);
    } else {
        cross3(e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz);                       // :93
    }
}
// The test's barycentrics for the ray (o, dd), query.hlsl:96-101: c = v0 - o, inv_det, u (the weight of v1) and v (of v2).
// tri_test and the attribute pass (hit_attr) both take them from here, so a hit's reported u, v are the test's own bits.
__device__ __forceinline__ void tri_uv(float ox, float oy, float oz, float ddx, float ddy, float ddz, float v0x, float v0y, float v0z,
                                       float e1x, float e1y, float e1z, float e2x, float e2y, float e2z, float ngx, float ngy, float ngz,
                                       float& cx, float& cy, float& cz, float& inv_det, float& u, float& v) {
    cx = sub(v0x, ox); cy = sub(v0y, oy); cz = sub(v0z, oz);                       // :96
    float rx, ry, rz; cross3(ddx, ddy, ddz, cx, cy, cz, rx, ry, rz);               // :97
    inv_det = __fdiv_rn(1.0f, dot3(ngx, ngy, ngz, ddx, ddy, ddz));                 // :98
    u = mul(dot3(rx, ry, rz, e2x, e2y, e2z), inv_det);                             // :100
    v = mul(dot3(rx, ry, rz, e1x, e1y, e1z), inv_det);                             // :101
}
// VARIANT_DIR: the test reads its direction from r.tdx/tdy/tdz (MODE 1) instead of the box test's r.dx/dy/dz
template <int TRI_STRIDE, bool VARIANT_DIR = false>
__device__ __forceinline__ float tri_test(const RayConst& r, float tmax, const uint4* __restrict__ tris, uint32_t prim) {
    const float ddx = VARIANT_DIR ? r.tdx : r.dx, ddy = VARIANT_DIR ? r.tdy : r.dy, ddz = VARIANT_DIR ? r.tdz : r.dz;
    float v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z;
    tri_load<TRI_STRIDE>(tris, prim, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z);
    float ngx, ngy, ngz;
    tri_normal<TRI_STRIDE>(tris, prim, e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz);
    float cx, cy, cz, inv_det, u, v;
    tri_uv(r.ox, r.oy, r.oz, ddx, ddy, ddz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz, cx, cy, cz, inv_det, u, v);
    const float w = sub(sub(1.0f, u), v);                                          // :102
    const uint32_t hit = __float_as_uint(u) | __float_as_uint(v) | __float_as_uint(w);   // :112
    float t = __int_as_float(0x7f800000);
    // :116 tests the sign bit.  An accepted triangle has u, v, w in [+0, 1], whose bits are all below 0x40000000 (2.0f), and u or
    // v > 1 forces w < 0, so `hit < 0x40000000` accepts exactly what the sign test accepts on non-NaN values — and also rejects a
    // NaN in any position, as the reference's x86 CPU path does (its invalid operations give the default NaN 0xFFC00000, sign
    // set; CUDA's canonical NaN 0x7FFFFFFF has the sign clear).  u or v is NaN when dot(r, e2) or dot(r, e1) overflows with
    // opposite signs, and tt can still be finite then.
    if (inv_det != 0.0f && hit < 0x40000000u) {
        const float tt = mul(dot3(ngx, ngy, ngz, cx, cy, cz), inv_det);            // :118
        if (tt >= r.tmin && tt <= tmax) t = tt;                                    // :119
    }
    return t;
}

// ---- work item -> pixel ------------------------------------------------------------------------
// Local work item j of shard s: 256 consecutive items form one 32x8-pixel tile (tile k = s + (j/256)*S in
// row-major tile order), 32 consecutive items form one 8x4 sub-tile — the footprint of one warp fetch.
__device__ __forceinline__ bool item_to_pixel(const FrameParams& P, uint32_t j, uint32_t& px, uint32_t& py) {
    const uint32_t local_tile = j >> 8, w = j & 255u;
    const uint32_t k = P.shard_index + local_tile * P.shard_count;
    const uint32_t sub = w >> 5, l = w & 31u;
    px = (k % P.tiles_x) * 32u + (sub & 3u) * 8u + (l & 7u);
    py = (k / P.tiles_x) * 8u + (sub >> 2) * 4u + (l >> 3);
    return px < P.width && py < P.height;
}

// where the RGBA of work item `item` goes: slot `item` of the compact buffer, or its pixel of a row-major frame target
// (possibly peer memory: the store then travels over NVLink while the warp keeps tracing); -1 = pixel outside the frame
__device__ __forceinline__ long long rgba_slot(const FrameParams& F, uint32_t item, bool row_major) {
    if (!row_major) return (long long)item;
    uint32_t px, py;
    if (!item_to_pixel(F, item, px, py)) return -1;
    return (long long)py * F.width + px;
}

// glam Mat4 * Vec4 (column-major): ((c0*x + c1*y) + c2*z) + c3*w
__device__ __forceinline__ void mat4_mul(const float* m, float x, float y, float z, float w, float o[4]) {
#pragma unroll
    for (int k = 0; k < 4; k++) o[k] = add(add(add(mul(m[k], x), mul(m[4 + k], y)), mul(m[8 + k], z)), mul(m[12 + k], w));
}

// pixel -> primary ray direction (src/rt_cpu/rt_cpu.rs:38-55)
__device__ __forceinline__ void primary_dir(const FrameParams& P, uint32_t px, uint32_t py, float& dx, float& dy, float& dz) {
    const float uvx = __fdiv_rn((float)px, (float)P.width);
    const float uvy = sub(1.0f, __fdiv_rn((float)py, (float)P.height));
    const float ndcx = sub(mul(uvx, 2.0f), 1.0f), ndcy = sub(mul(uvy, 2.0f), 1.0f);
    float vs[4]; mat4_mul(P.view.proj_inv, ndcx, ndcy, 1.0f, 1.0f, vs);
    const float ww = vs[3];
    vs[0] = __fdiv_rn(vs[0], ww); vs[1] = __fdiv_rn(vs[1], ww); vs[2] = __fdiv_rn(vs[2], ww); vs[3] = __fdiv_rn(vs[3], ww);
    float wp[4]; mat4_mul(P.view.view_inv, vs[0], vs[1], vs[2], vs[3], wp);
    dx = sub(wp[0], P.view.eye[0]); dy = sub(wp[1], P.view.eye[1]); dz = sub(wp[2], P.view.eye[2]);
    normalize3(dx, dy, dz);
}

// sampling.hlsl:5-27
__device__ __forceinline__ uint32_t uhash(uint32_t a, uint32_t b) {
    uint32_t x = (a * 1597334673u) ^ (b * 3812015801u);
    x = x ^ (x >> 16); x *= 0x7feb352du;
    x = x ^ (x >> 15); x *= 0x846ca68bu;
    x = x ^ (x >> 16);
    return x;
}
__device__ __forceinline__ float hash_noise(uint32_t x, uint32_t y, uint32_t frame) {
    return mul(__uint2float_rn(uhash(x, (y << 11) + frame)), 2.3283064365386963e-10f);   // 1 / float(0xffffffff) = 2^-32
}
// sin/cos(2*pi*u): fixed quadrant reduction + fmaf Horner, bit-reproducible on any IEEE machine (the platform
// sin/cos the reference calls, sampling.hlsl:30-36, is not; the bounce direction is an input distribution).
__device__ __forceinline__ void sincos_tau(float u, float& s, float& c) {
    const float q4 = mul(u, 4.0f), qf = rintf(q4), r = sub(q4, qf);
    const float x = mul(r, 1.57079632679489661923f), x2 = mul(x, x);
    float sp = __fmaf_rn(x2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = __fmaf_rn(sp, x2, -1.6666654611e-1f);
    const float sn = __fmaf_rn(mul(x, x2), sp, x);
    float cp = __fmaf_rn(x2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = __fmaf_rn(cp, x2, 4.166664568298827e-2f);
    const float cs = __fmaf_rn(mul(x2, x2), cp, __fmaf_rn(x2, -0.5f, 1.0f));
    const int q = (int)qf & 3;
    s = q == 0 ? sn : q == 1 ? cs : q == 2 ? -sn : -cs;
    c = q == 0 ? cs : q == 1 ? -sn : q == 2 ? -cs : sn;
}

// ---- instance transforms: `xf` is an InstanceRecord, rows 0..2 of world_to_object W ([W | -W t]) -------------------------
// The ray of a TLAS leaf in object space: o' = ((W_i0 o_x + W_i1 o_y) + W_i2 o_z) + W_i3 and d' = dot(W_i, d) for row i
__device__ __forceinline__ void xform_row(const uint4& w, float ox, float oy, float oz, float dx, float dy, float dz, float& o, float& d) {
    const float m0 = __uint_as_float(w.x), m1 = __uint_as_float(w.y), m2 = __uint_as_float(w.z);
    o = add(add(add(mul(m0, ox), mul(m1, oy)), mul(m2, oz)), __uint_as_float(w.w));
    d = dot3(m0, m1, m2, dx, dy, dz);
}
// An object-space normal to world space through the transpose of W, n'_i = W_0i n_0 + W_1i n_1 + W_2i n_2 (the inverse
// transpose of object_to_world), not normalised
__device__ __forceinline__ void normal_to_world(const uint4* __restrict__ xf, float& nx, float& ny, float& nz) {
    const uint4 w0 = __ldg(xf), w1 = __ldg(xf + 1), w2 = __ldg(xf + 2);
    const float wx = dot3(__uint_as_float(w0.x), __uint_as_float(w1.x), __uint_as_float(w2.x), nx, ny, nz);
    const float wy = dot3(__uint_as_float(w0.y), __uint_as_float(w1.y), __uint_as_float(w2.y), nx, ny, nz);
    const float wz = dot3(__uint_as_float(w0.z), __uint_as_float(w1.z), __uint_as_float(w2.z), nx, ny, nz);
    nx = wx; ny = wy; nz = wz;
}

// bounce ray from a primary hit (src/rt_cpu/rt_cpu.rs:61-76; basis sampling.hlsl:39-51)
// INST: `xf` is the InstanceRecord of the hit's instance; the object-space normal goes to world space through the transpose of
// world_to_object, n'_i = W_0i n_0 + W_1i n_1 + W_2i n_2 (the inverse transpose of object_to_world), before it is normalised.
template <int TRI_STRIDE, bool INST = false>
__device__ __forceinline__ void bounce_ray(const FrameParams& P, const uint4* __restrict__ tris, uint32_t px, uint32_t py,
                                           float pdx, float pdy, float pdz, float t, uint32_t prim,
                                           float& ox, float& oy, float& oz, float& dx, float& dy, float& dz,
                                           const uint4* __restrict__ xf = nullptr) {
    float nx, ny, nz;
    if (TRI_STRIDE == 64) {
        const uint4 g = __ldg(tris + (size_t)prim * 4u + 3);
        nx = __uint_as_float(g.x); ny = __uint_as_float(g.y); nz = __uint_as_float(g.z);
    } else {
        float v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z;
        tri_load<TRI_STRIDE>(tris, prim, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z);
        cross3(e1x, e1y, e1z, e2x, e2y, e2z, nx, ny, nz);
    }
    if constexpr (INST) normal_to_world(xf, nx, ny, nz);
    normalize3(nx, ny, nz);                                                    // RtTriangle::compute_normal
    const float sgn = copysignf(1.0f, dot3(nx, ny, nz, -pdx, -pdy, -pdz));     // f32::signum (rt_cpu.rs:65)
    nx = mul(nx, sgn); ny = mul(ny, sgn); nz = mul(nz, sgn);
    ox = sub(add(P.view.eye[0], mul(pdx, t)), mul(pdx, 0.01f));                // rt_cpu.rs:67
    oy = sub(add(P.view.eye[1], mul(pdy, t)), mul(pdy, 0.01f));
    oz = sub(add(P.view.eye[2], mul(pdz, t)), mul(pdz, 0.01f));
    const float u0 = hash_noise(px, py, P.frame_count), u1 = hash_noise(px, py, P.frame_count + 1024u);   // rt_cpu.rs:70-73
    const float rr = __fsqrt_rn(u0);
    float sn, cs; sincos_tau(u1, sn, cs);
    const float lx = mul(rr, cs), ly = mul(rr, sn), lz = __fsqrt_rn(fmaxf(0.0f, sub(1.0f, u0)));
    const float sign = nz >= 0.0f ? 1.0f : -1.0f;                              // sampling.hlsl:40-50
    const float a = __fdiv_rn(-1.0f, add(sign, nz));
    const float b = mul(mul(nx, ny), a);
    const float b1x = add(1.0f, mul(mul(mul(sign, nx), nx), a)), b1y = mul(sign, b), b1z = mul(-sign, nx);
    const float b2x = b, b2y = add(sign, mul(mul(ny, ny), a)), b2z = -ny;
    dx = add(add(mul(b1x, lx), mul(b2x, ly)), mul(nx, lz));                    // Mat3::from_cols(b1, b2, n) * l
    dy = add(add(mul(b1y, lx), mul(b2y, ly)), mul(ny, lz));
    dz = add(add(mul(b1z, lx), mul(b2z, ly)), mul(nz, lz));
    normalize3(dx, dy, dz);
}

// the colour of a result of kind `mode` (ShadeMode), gamma-encoded as rt_cpu.rs:104-106
__device__ __forceinline__ uchar4 shade(uint32_t mode, float t) {
    float col;
    if (mode == SHADE_PRIMARY) col = __fdiv_rn(1.0f, t);                                   // rt_cpu.rs:59 (1/inf = 0)
    else if (mode == SHADE_OCCLUSION) col = t < F32_MAX_ ? 0.0f : 1.0f;                   // any-hit AO: visibility only
    else col = t < F32_MAX_ ? __fdiv_rn(t, add(1.0f, t)) : 1.0f;                          // rt_cpu.rs:82-87
    float g = powf(col, 2.2f) * 255.0f;
    g = g < 0.0f ? 0.0f : (g > 255.0f ? 255.0f : g);
    const unsigned char v = (unsigned char)g;
    return make_uchar4(v, v, v, 255);
}
__device__ __forceinline__ void store_rgba(uchar4* rgba_out, const FrameParams& F, bool row_major, uint32_t item, uint32_t mode, float t) {
    if (!rgba_out) return;
    const long long o = rgba_slot(F, item, row_major);
    if (o >= 0) rgba_out[o] = shade(mode, t);
}

// a tray_ray as two 16-byte stores: {origin, tmin}, {direction, tmax}
__device__ __forceinline__ void store_ray(tray_ray* dst, const float4& a, const float4& b) {
    float4* o = reinterpret_cast<float4*>(dst);
    o[0] = a; o[1] = b;
}
// the bounce ray of work item `item` as generated, for checkers (optional buffer, TRAY_RENDER_KEEP_RAYS)
__device__ __forceinline__ void keep_ray(tray_ray* rays_by_item, uint32_t item, const float4& a, const float4& b) {
    if (rays_by_item) store_ray(rays_by_item + item, a, b);
}
// a pixel that shoots no bounce ray (primary miss, or outside the frame) gets its final results at once: a bounce miss, the
// primary shade, a zero ray
__device__ __forceinline__ void finish_no_bounce(const FrameParams& F, bool row_major, uint32_t item, float t_primary, tray_hit* bounce_out,
                                                 uchar4* rgba_out, tray_ray* rays_by_item) {
    tray_hit miss; miss.t = __int_as_float(0x7f800000); miss.prim = INVALID;
    bounce_out[item] = miss;
    store_rgba(rgba_out, F, row_major, item, SHADE_PRIMARY, t_primary);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    keep_ray(rays_by_item, item, z, z);
}

// ---- ray generation ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) raygen_primary_kernel(const __grid_constant__ FrameParams F, tray_ray* __restrict__ rays) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= F.n_items) return;
    uint32_t px, py;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = make_float4(0.f, 0.f, 0.f, 0.f);   // pixel outside the frame: tmax = 0
    if (item_to_pixel(F, j, px, py)) {
        float dx, dy, dz; primary_dir(F, px, py, dx, dy, dz);
        a = make_float4(F.view.eye[0], F.view.eye[1], F.view.eye[2], 0.0f);            // Ray::new(eye, dir, 0.0, f32::MAX)
        b = make_float4(dx, dy, dz, F32_MAX_);
    }
    store_ray(rays + j, a, b);
}

// One thread per pixel of the shard.  Hit pixels append their bounce ray to a compact list (one atomicAdd per block;
// `ray_item` remembers the pixel); missed pixels get their final results here.
constexpr int BOUNCE_BLOCK = 1024;    // pixels per block of raygen_bounce_kernel = the group its rays are sorted in
// INST (instanced scenes): `primary_inst` holds the instance of each primary hit, `inst_xf` the InstanceRecords by instance id.
template <int TRI_STRIDE, bool INST = false>
__global__ void __launch_bounds__(BOUNCE_BLOCK) raygen_bounce_kernel(const __grid_constant__ FrameParams F, const uint4* __restrict__ tris,
                                                            const tray_hit* __restrict__ primary, tray_ray* __restrict__ rays,
                                                            uint32_t* __restrict__ ray_item, uint32_t* __restrict__ n_rays,
                                                            tray_hit* __restrict__ bounce_out, uchar4* __restrict__ rgba_out,
                                                            tray_ray* __restrict__ rays_by_item, uint32_t row_major,
                                                            const uint32_t* __restrict__ primary_inst, const uint4* __restrict__ inst_xf) {
    __shared__ uint32_t s_cnt[8], s_base[8];
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t px = 0, py = 0;
    bool shoot = false;
    tray_hit ph; ph.t = __int_as_float(0x7f800000); ph.prim = INVALID;
    if (j < F.n_items && item_to_pixel(F, j, px, py)) {
        ph = primary[j];
        shoot = ph.t < F32_MAX_;                                                      // rt_cpu.rs:61
    }
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (shoot) {
        float pdx, pdy, pdz; primary_dir(F, px, py, pdx, pdy, pdz);
        float ox, oy, oz, dx, dy, dz;
        if constexpr (INST)
            bounce_ray<TRI_STRIDE, true>(F, tris, px, py, pdx, pdy, pdz, ph.t, ph.prim, ox, oy, oz, dx, dy, dz,
                                         inst_xf + (size_t)primary_inst[j] * INST_RECORD_U4);
        else
            bounce_ray<TRI_STRIDE>(F, tris, px, py, pdx, pdy, pdz, ph.t, ph.prim, ox, oy, oz, dx, dy, dz);
        a = make_float4(ox, oy, oz, 0.0f); b = make_float4(dx, dy, dz, F32_MAX_);
    }
    // The rays of the block's 1024 pixels (4 tiles: close origins) are appended grouped by direction octant, so that the
    // 32 rays a traversal warp fetches together share the order in which they visit a node's children.
    if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    const uint32_t oct = (b.x < 0.f ? 4u : 0u) | (b.y < 0.f ? 2u : 0u) | (b.z < 0.f ? 1u : 0u);
    uint32_t pos = 0;
    if (shoot) pos = atomicAdd(&s_cnt[oct], 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t acc = 0;
        for (uint32_t o = 0; o < 8; o++) { const uint32_t c = s_cnt[o]; s_base[o] = acc; acc += c; }
        const uint32_t g = acc ? atomicAdd(n_rays, acc) : 0u;
        for (uint32_t o = 0; o < 8; o++) s_base[o] += g;
    }
    __syncthreads();
    if (shoot) {
        const uint32_t slot = s_base[oct] + pos;
        store_ray(rays + slot, a, b);
        ray_item[slot] = j;
    }
    if (j < F.n_items) {
        if (!shoot) finish_no_bounce(F, row_major, j, ph.t, bounce_out, rgba_out, rays_by_item);
        else keep_ray(rays_by_item, j, a, b);
    }
}

// FRAME kernel hand-shake: a primary hit record is published and polled as ONE 64-bit scalar access ({t, prim} packed),
// which the PTX memory model makes single-copy atomic (a .v2.u32 pair is two accesses in unspecified order).
__device__ __forceinline__ void publish_hit(tray_hit* dst, const tray_hit& h) {
    const unsigned long long v = (unsigned long long)__float_as_uint(h.t) | ((unsigned long long)h.prim << 32);
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(dst), "l"(v) : "memory");
}
__device__ __forceinline__ bool poll_hit(const tray_hit* src, float2& ph) {       // false: still the host's 0xFF fill pattern
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
    ph.x = __uint_as_float((uint32_t)v); ph.y = __uint_as_float((uint32_t)(v >> 32));
    return v != 0xffffffffffffffffull;
}

// one counter slot += the warp's counts (COUNT builds)
__device__ __forceinline__ void flush_counters(unsigned long long* dst, unsigned lane, unsigned long long rays, unsigned long long nodes,
                                               unsigned long long tris, unsigned long long insts, unsigned long long hits) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        rays += __shfl_xor_sync(FULL, rays, o); nodes += __shfl_xor_sync(FULL, nodes, o);
        tris += __shfl_xor_sync(FULL, tris, o); insts += __shfl_xor_sync(FULL, insts, o);
        hits += __shfl_xor_sync(FULL, hits, o);
    }
    if (lane == 0) {
        atomicAdd(dst + 0, rays); atomicAdd(dst + 1, nodes); atomicAdd(dst + 2, tris);
        atomicAdd(dst + 3, insts); atomicAdd(dst + 4, hits);
    }
}

// ---- the traversal kernel ---------------------------------------------------------------------------
// Per-lane state is kept NORMALISED between steps: a lane is exactly one of
//   TRI   tri_y != 0                         next action: test one triangle (or enter one TLAS instance)
//   NODE  tri_y == 0, cur_y has node bits    next action: fetch + test one node
//   IDLE  tri_y == 0, cur_y == 0             no ray; waits for the next refill
// so one pair of ballots per iteration drives everything (refill, phase vote, exit).
// ANYHIT: a ray retires at its FIRST accepted triangle (the "faster anyhit query" rt_cpu.rs:78-79 asks for AO rays);
// the sequence of tests up to that point is the closest-hit one, so "found a hit" is the same predicate.
// FRAME: ONE launch traces a whole frame (TRAY_RENDER_OVERLAP).  Phase 1 is the primary pass as ever.  Once the primary cursor
// has run dry, a warp with idle lanes claims the next group of 32 items (one atomicAdd per group, in item order), waits until
// the group's 32 primary hits are THERE, generates the group's bounce rays full-width (bounce_ray, the code of
// raygen_bounce_kernel), parks them in the bounce-ray buffer and hands them to its idle lanes one by one — so the drain phase of
// the primary pass is filled with bounce work instead of idle SMs, and the frame has one drain phase instead of two.
// The hand-shake needs neither counters nor fences: the host fills the primary-hit buffer with 0xFFFFFFFF'FFFFFFFF before the
// launch, no hit record looks like that (its t would be a NaN), and a lane publishes its record with ONE aligned 8-byte store;
// a reader that sees something else than the fill pattern sees the whole record.  A warp with nothing else in hand polls with
// __nanosleep and a watchdog (the device is never hung: after ~2 s it sets ERR_WATCHDOG in the error word and leaves).
// Per ray nothing changes: same node order, same triangle order, same (prim, t).
// MODE 1: the three semantics of the reference's CPU path that are sourced from memory of the un-vendored obvhs crate (tie
// rule, slab-test lower clamp, reach of the zero-direction patch) and the HLSL's divide-form box test become RUN-TIME switches
// (P.variant, TRAY_VARIANT_*), so that the day a real obvhs dump arrives the answer is a flag.  Slower (unfused node test);
// MODE 0, the default, compiles them away.
// (A MODE 2 — relaxed order: triangle postponing, tolerance parity — was built and measured in round 2 and is NOT in the
// product: on CWBVHs of this shape 81 % of the nodes hold only leaves, so a lane almost never has triangles and child nodes in
// hand at once; nothing was postponed, nothing mismatched, and the extra vote cost 3 %.  profiles/experiments/r2_relaxed_*.)
// INST (instanced scenes; TLAS, MODE 0, not FRAME): a TLAS leaf places its BLAS by a transform.  Entering it, the lane maps its
// ray into object space with the leaf's world_to_object (origin o' = W o + t, direction d' = W d, not normalised, so tmin, tmax
// and the t of a hit keep their world meaning) and prepares that ray; back at the TLAS it prepares the world ray again, re-read
// from P.rays at its index (both callers, batch traces and the two-launch frame, hold every ray there) instead of holding six
// more registers.  best_inst follows best_prim.
template <bool TLAS, bool COUNT, int TRI_STRIDE, bool ANYHIT = false, bool FRAME = false, int MODE = 0, bool INST = false>
__global__ void __launch_bounds__(BLOCK_THREADS, TRAY_MIN_BLOCKS) trace_kernel(const __grid_constant__ TraceParams P) {
    static_assert(!INST || (TLAS && !FRAME && MODE == 0), "instance transforms exist in the two-level MODE 0 batch kernels only");
    __shared__ uint8_t s_lut[LUT_BYTES];          // child_order[oct_inv][hit byte] (see node_test)
    uint2 spill[STACK_SPILL];
    child_order_fill(s_lut, threadIdx.x, BLOCK_THREADS);
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t k4b = P.k4b;
    const uint32_t n_work = P.n_work_dev ? *P.n_work_dev : P.n_work;

    RayConst r;
    float best_t = 0.f;
    uint32_t best_prim = INVALID;
    uint32_t cur_x = 0, cur_y = 0, tri_x = 0, tri_y = 0;
    // the stack pointer IS the byte offset of the lane's next free entry in tray_stack_mem ([entry][thread]): depth * SP_STEP + thread * 8
    // (one register instead of a depth and a per-thread base address)
    constexpr uint32_t SP_STEP = BLOCK_THREADS * 8u, SP_SMEM_END = STACK_SMEM * SP_STEP, SP_END = (STACK_SMEM + STACK_SPILL) * SP_STEP;
    uint32_t sp = threadIdx.x * 8u;
    // the stack lives in a shared-memory array declared in PTX, so that its address is a plain CTA-local offset that ptxas keeps in a
    // uniform register (STS.64 [R + UR]) — the address of a C++ __shared__ array goes through the generic->shared conversion, which
    // on sm_90+ reads SR_CgaCtaId and rebuilds the shared window base (S2R + MOV + LEA + IADD) at EVERY push and pop: +2.3 % on C3,
    // +1.2 % on C1 together with the late push of the node step (profiles/experiments/r2_push_late_ab.log)
    uint32_t stk_base;
    asm volatile(".shared .align 16 .b8 tray_stack_mem[%1];\n\tmov.u32 %0, tray_stack_mem;" : "=r"(stk_base) : "n"(STACK_SMEM * BLOCK_THREADS * 8));
    auto stk_store = [&](uint32_t off, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(stk_base + off), "r"(x), "r"(y) : "memory"); };
    auto stk_load = [&](uint32_t off) { uint2 e; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(stk_base + off) : "memory"); return e; };
    uint32_t tlas_sp = INVALID, bvh_off = 0;
    uint32_t cur_inst = 0, best_inst = INVALID;  // INST: the instance the lane is in, the instance of best_prim
    uint32_t ray_idx = 0;
    bool exhausted = false;                      // warp-uniform
    // a lane starts fewer than 2^30 rays per launch (INDEX_MASK), so its ray and hit counts fit 32 bits
    uint32_t c_rays = 0, c_hits = 0, b_rays = 0, b_hits = 0;
    unsigned long long c_nodes = 0, c_tris = 0, c_insts = 0;
    unsigned long long b_nodes = 0, b_tris = 0, b_insts = 0;    // FRAME && COUNT: the bounce rays' share
    // COUNT builds: the cost of the lane's ray so far, added to the warp totals above when it retires; r_peak is the highest
    // stack pointer it reached (depth * SP_STEP + thread * 8, so r_peak / SP_STEP is its peak depth in entries)
    uint32_t r_nodes = 0, r_tris = 0, r_insts = 0, r_peak = 0;
    // ray_idx: INDEX_MASK bits of index, BOUNCE_BIT, WIDE_BIT
#define TRAY_CNT(name) do { if constexpr (COUNT) r_##name++; } while (0)
    uint32_t cur_unit = INVALID, cand_unit = INVALID, H = 0, sleeps = 0;   // FRAME, warp-uniform: 32-pixel group being fed from, claimed group, its pixels still to shoot
    bool units_done = false;

    auto push = [&](uint32_t x, uint32_t y) {
        if (sp < SP_SMEM_END) stk_store(sp, x, y);
        else if (sp < SP_END) spill[sp / SP_STEP - STACK_SMEM] = make_uint2(x, y);
        else { atomicOr(P.overflow, ERR_STACK_OVERFLOW); return; }
        sp += SP_STEP;
        if constexpr (COUNT) r_peak = max(r_peak, sp);
    };
    // the lane takes up the ray ray_idx holds, at the root group (query.hlsl:343)
    auto start_ray = [&](float ox, float oy, float oz, float dx, float dy, float dz, float tmin, float tmax, uint32_t variant) {
        prepare_ray(r, ox, oy, oz, dx, dy, dz, tmin, variant, (uint32_t)__cvta_generic_to_shared(s_lut));
        if (r.wide) ray_idx |= WIDE_BIT;
        best_t = tmax; best_prim = INVALID;
        cur_x = 0; cur_y = 0x80000000u; tri_x = 0; tri_y = 0; sp &= SP_STEP - 1u;
        tlas_sp = INVALID; bvh_off = TLAS ? P.tlas_start : 0u;
        if constexpr (COUNT) { r_nodes = 0; r_tris = 0; r_insts = 0; r_peak = 0; }
    };
    // INST: the lane's ray becomes (o, d) with the same tmin: octant row, zero-direction patch and WIDE_BIT follow it
    auto switch_ray = [&](float ox, float oy, float oz, float dx, float dy, float dz) {
        prepare_ray(r, ox, oy, oz, dx, dy, dz, r.tmin, 0u, (uint32_t)__cvta_generic_to_shared(s_lut));
        ray_idx = r.wide ? (ray_idx | WIDE_BIT) : (ray_idx & ~WIDE_BIT);
    };
    // COUNT builds, a ray retires: its counts join the warp totals of its pass, and its record goes to slot `item` of P.ray_cost
    // (`if constexpr` here and at every use of the r_* registers: the kernels that do not count compile to the code they had
    // before these records existed)
    auto retire_cost = [&](uint32_t item, bool hit) {
        if constexpr (COUNT) {
            if (FRAME && (ray_idx & BOUNCE_BIT)) { b_nodes += r_nodes; b_tris += r_tris; b_insts += r_insts; b_hits += hit; }
            else { c_nodes += r_nodes; c_tris += r_tris; c_insts += r_insts; c_hits += hit; }
            if (P.ray_cost) reinterpret_cast<uint4*>(P.ray_cost)[item] = make_uint4(r_nodes, r_tris, r_insts, r_peak / SP_STEP);
        }
    };
    // called when the lane has neither triangles nor nodes left in hand: pop the stack, or retire the ray
    // (query.hlsl:417-427; tlas:480-486; the popped-triangle-group case is query.hlsl:389-393)
    auto pop_or_retire = [&]() {
        if (sp < SP_STEP) {
            tray_hit h;
            h.t = best_prim != INVALID ? best_t : __int_as_float(0x7f800000);   // RayHit::none()
            h.prim = best_prim;
            if (FRAME) {
                const uint32_t it = ray_idx & INDEX_MASK;
                if constexpr (COUNT) retire_cost((ray_idx & BOUNCE_BIT) ? P.n_work + it : it, best_prim != INVALID);
                if (!(ray_idx & BOUNCE_BIT))      // ONE 64-bit scalar store (single-copy atomic, unlike a .v2 pair): the record itself tells a reader that it is there
                    publish_hit(P.hits_out + it, h);
                else {
                    P.bounce_out[it] = h;
                    store_rgba(P.rgba_out, P.frame, P.row_major, it, SHADE_BOUNCE, h.t);
                }
                cur_x = 0; cur_y = 0;
                return;
            }
            const uint32_t ri = ray_idx & INDEX_MASK;
            const uint32_t item = P.ray_item ? __ldg(P.ray_item + ri) : ri;
            P.hits_out[item] = h;
            if constexpr (INST) { if (P.inst_out) P.inst_out[item] = best_prim != INVALID ? best_inst : INVALID; }
            store_rgba(P.rgba_out, P.frame, P.row_major, item, P.shade_mode, h.t);
            if constexpr (COUNT) retire_cost(item, best_prim != INVALID);
            cur_x = 0; cur_y = 0;                                                                    // IDLE
        } else {
            if (TLAS && sp == tlas_sp) {
                tlas_sp = INVALID; bvh_off = P.tlas_start;
                if constexpr (INST) {                                                    // back to the world ray
                    const float4* rp = reinterpret_cast<const float4*>(P.rays + (ray_idx & INDEX_MASK));
                    const float4 a = __ldg(rp), b = __ldg(rp + 1);
                    switch_ray(a.x, a.y, a.z, b.x, b.y, b.z);
                }
            }
            sp -= SP_STEP;
            const uint2 e = sp < SP_SMEM_END ? stk_load(sp) : spill[sp / SP_STEP - STACK_SMEM];
            if (e.y & 0xff000000u) { cur_x = e.x; cur_y = e.y; }
            else { tri_x = e.x; tri_y = e.y; cur_x = 0; cur_y = 0; }
        }
    };

    for (;;) {
        const bool want_tri = tri_y != 0u;
        const bool want_node = !want_tri && cur_y >= 0x01000000u;
        const unsigned m_tri = __ballot_sync(FULL, want_tri), m_node = __ballot_sync(FULL, want_node);
        const unsigned busy = m_tri | m_node;

        // ---- refill idle lanes from the global cursor (persistent warps + ray replacement) ----
        if (busy != FULL) {
            if (!exhausted && ((unsigned)__popc(~busy) >= P.refill_min || busy == 0u)) {
                const unsigned idle = ~busy;
                const uint32_t n_idle = (uint32_t)__popc(idle);
                const int leader = __ffs(idle) - 1;
                uint32_t base = 0;
                if ((int)lane == leader) base = atomicAdd(P.cursor, n_idle);
                base = __shfl_sync(FULL, base, leader);
                if (base + n_idle >= n_work) exhausted = true;
                if ((idle >> lane) & 1u) {
                    ray_idx = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
                    if (base < n_work && ray_idx < n_work) {
                        const float4* rp = reinterpret_cast<const float4*>(P.rays + ray_idx);
                        const float4 a = __ldg(rp), b = __ldg(rp + 1);
                        start_ray(a.x, a.y, a.z, b.x, b.y, b.z, a.w, b.w, MODE == 1 ? P.variant : 0u);
                        if (COUNT) c_rays++;
                    }
                }
                continue;                                    // re-vote with the new rays
            }
            if (!FRAME && busy == 0u) break;                 // cursor exhausted and nothing in flight
        }
        if (FRAME) {
            const unsigned idle = ~busy;
            if (exhausted && idle != 0u) {
                if (H != 0u) {
                    if ((unsigned)__popc(idle) >= P.gen_min || busy == 0u) {
                        // the k-th idle lane shoots the k-th pending pixel of the group (rt_cpu.rs:61-76)
                        const unsigned rank = (unsigned)__popc(idle & ((1u << lane) - 1u));
                        const bool take = ((idle >> lane) & 1u) && rank < (unsigned)__popc(H);
                        if (take) {
                            const uint32_t pix = __fns(H, 0, (int)rank + 1);
                            const uint32_t item = cur_unit * 32u + pix;
                            const float4* gp = reinterpret_cast<const float4*>(P.gen_rays + item);     // written by this warp at the claim
                            const float4 ga = __ldcg(gp), gb = __ldcg(gp + 1);
                            ray_idx = item | BOUNCE_BIT;
                            start_ray(ga.x, ga.y, ga.z, gb.x, gb.y, gb.z, 0.0f, F32_MAX_, 0u);   // Ray::new(o, dir, 0.0, f32::MAX)
                            if (COUNT) b_rays++;
                        }
                        int n_take = min(__popc(idle), __popc(H));
                        while (n_take-- > 0) H &= H - 1u;                                     // the lowest bits are the ones taken
                        continue;
                    }
                } else {
                    // the group in hand is used up: claim the next 32-pixel group (in item order) and wait for its tile
                    if (cand_unit == INVALID && !units_done) {
                        uint32_t u = 0;
                        if (lane == 0) u = atomicAdd(P.unit_cursor, 1u);
                        u = __shfl_sync(FULL, u, 0);
                        if (u >= P.n_units) units_done = true; else cand_unit = u;
                    }
                    if (cand_unit != INVALID) {
                        // the group is ready when the primary hits of its 32 items are all there: the host fills the hit buffer
                        // with the pattern 0xFFFFFFFF'FFFFFFFF before the launch, no hit record looks like that (t would be a NaN),
                        // and a record is one aligned 8-byte store — no counters, no fences in the primary pass
                        const uint32_t item = cand_unit * 32u + lane;
                        float2 ph;
                        const bool there = poll_hit(P.hits_out + item, ph);
                        if (__ballot_sync(FULL, there) == FULL) {
                            cur_unit = cand_unit; cand_unit = INVALID; sleeps = 0;
                            // the group's 32 pixels: who shoots?  Missed pixels get their final results here (rt_cpu.rs:59)
                            uint32_t px, py;
                            const bool inside = item_to_pixel(P.frame, item, px, py);
                            const bool shoot = inside && ph.x < F32_MAX_;                     // rt_cpu.rs:61
                            if (!shoot) finish_no_bounce(P.frame, P.row_major, item, ph.x, P.bounce_out, P.rgba_out, P.rays_by_item);
                            else {
                                const float4 pb = __ldg(reinterpret_cast<const float4*>(P.rays + item) + 1);   // the primary direction as generated
                                float ox, oy, oz, dx, dy, dz;
                                bounce_ray<TRI_STRIDE>(P.frame, P.tris, px, py, pb.x, pb.y, pb.z, ph.x, __float_as_uint(ph.y), ox, oy, oz, dx, dy, dz);
                                const float4 a = make_float4(ox, oy, oz, 0.0f), b = make_float4(dx, dy, dz, F32_MAX_);
                                store_ray(P.gen_rays + item, a, b);
                                keep_ray(P.rays_by_item, item, a, b);
                            }
                            __syncwarp();                      // the group's rays are read back by other lanes of this warp
                            H = __ballot_sync(FULL, shoot);
                            continue;
                        }
                        if (busy == 0u) {                     // nothing else in hand: wait for the tile's last primary rays
                            __nanosleep(500);
                            if (++sleeps > 4000000u) { atomicOr(P.overflow, ERR_WATCHDOG); break; }       // watchdog: never hang the device
                            continue;
                        }
                    } else if (busy == 0u) break;             // no group left, nothing in flight
                }
            }
            if (busy == 0u) { if (exhausted && units_done && cand_unit == INVALID && H == 0u) break; continue; }
        }

        // ---- warp vote: node step or triangle step ----
        const bool tri_phase = m_node == 0u || (unsigned)__popc(m_tri) * P.tri_weight >= (unsigned)__popc(m_node);

        if (!tri_phase) {
            if (want_node) {
                const uint32_t hits_imask = cur_y;
                uint32_t slot;                                                                 // query.hlsl:358 + :370 in one lookup (see node_test)
                asm("ld.shared.u8 %0, [%1];" : "=r"(slot) : "r"(r.lut_off + (hits_imask >> 24)));
                cur_y = hits_imask ^ (0x01000000u << slot);                                    // :362
                const uint32_t rel = (uint32_t)__popc(hits_imask & ((1u << slot) - 1u));       // :371 (slot < 8: imask bits only)
                const uint4* np = P.nodes + (size_t)(bvh_off + cur_x + rel) * 5u;              // :373, tlas:383
                const uint4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
                if (cur_y & 0xff000000u) push(cur_x, cur_y);                                   // :365-368, in the shadow of the node fetch
                TRAY_CNT(nodes);
                uint32_t hitmask;                                                              // slot space (see node_test)
                if (MODE == 1) hitmask = node_test(r, best_t, n0, n1, n2, n3, n4, k4b, r.box_tmin, (P.variant & TRAY_VARIANT_BOX_DIVIDE) != 0u);
                else hitmask = ((ray_idx & WIDE_BIT) || P.force_exact) ? node_test(r, best_t, n0, n1, n2, n3, n4, k4b)
                                                : node_test_fast(r, best_t, n0, n1, n2, n3, n4, k4b, P.zero, P.one);   // :380
                cur_x = n1.x; tri_x = n1.y;                                                    // :383-384
                cur_y = (hitmask & 0xff000000u) | (n0.w >> 24);                                // :386 (top byte: hit inner children, slot space)
                tri_y = hitmask & 0x00ffffffu;                                                 // :387
                if (tri_y == 0u && cur_y < 0x01000000u) pop_or_retire();
            }
        } else {
            if (want_tri) {
                const uint32_t local = 31u - (uint32_t)__clz((int)tri_y);                      // :398
                tri_y &= ~(1u << local);                                                       // :401
                const uint32_t g = tri_x + local;                                              // :403
                if (TLAS && tlas_sp == INVALID) {
                    // TLAS leaf: g is an instance slot (query_tlas.hlsl:410-446)
                    if (tri_y != 0u) push(tri_x, tri_y);
                    if (cur_y & 0xff000000u) push(cur_x, cur_y);
                    tlas_sp = sp;
                    if constexpr (INST) {
                        // into object space: o' = W o + t and d' = W d of the caller's direction (not the zero-patched one)
                        const uint4* rec = P.inst_rec + (size_t)g * INST_RECORD_U4;
                        const uint4 w0 = __ldg(rec), w1 = __ldg(rec + 1), w2 = __ldg(rec + 2), w3 = __ldg(rec + 3);
                        const float4 d = __ldg(reinterpret_cast<const float4*>(P.rays + (ray_idx & INDEX_MASK)) + 1);
                        bvh_off = w3.x; cur_inst = w3.y;
                        float ox, oy, oz, dx, dy, dz;
                        xform_row(w0, r.ox, r.oy, r.oz, d.x, d.y, d.z, ox, dx);
                        xform_row(w1, r.ox, r.oy, r.oz, d.x, d.y, d.z, oy, dy);
                        xform_row(w2, r.ox, r.oy, r.oz, d.x, d.y, d.z, oz, dz);
                        switch_ray(ox, oy, oz, dx, dy, dz);
                    } else {
                        bvh_off = __ldg(P.blas_offsets + g);
                    }
                    TRAY_CNT(insts);
                    cur_x = 0; cur_y = 0x80000000u; tri_y = 0;
                } else {
                    TRAY_CNT(tris);
                    // Two triangles of the lane's pending group per iteration (82 % of the groups hold >= 2): both records are
                    // fetched together and the two tests run side by side.  The second test's only use of tmax is its final
                    // `tt <= tmax` (query.hlsl:119), so running it against the OLD tmax and comparing with the updated best_t
                    // afterwards accepts exactly what the sequential order accepts — bit-exact, ties included.  -2.5 % frame time
                    // (profiles/experiments/r2_ab_tri2_*).
                    const bool two = MODE != 1 && tri_y != 0u;
                    const uint32_t local2 = 31u - (uint32_t)__clz((int)tri_y);                  // read only when `two`
                    const uint32_t g2 = tri_x + local2;
                    if (two) tri_y &= ~(1u << local2);
                    float t2 = __int_as_float(0x7f800000);
                    if (two) t2 = tri_test<TRI_STRIDE, false>(r, best_t, P.tris, g2);
                    const float t = tri_test<TRI_STRIDE, MODE == 1>(r, best_t, P.tris, g);
                    // CPU tie rule: first of equal t wins (§8a a11); TRAY_VARIANT_TIE_LAST: the HLSL's `tt <= t` (query.hlsl:120)
                    const bool closer = (MODE == 1 && (P.variant & TRAY_VARIANT_TIE_LAST)) ? (t <= best_t && t < __int_as_float(0x7f800000)) : (t < best_t);
                    if (closer) { best_t = t; best_prim = g; if constexpr (INST) best_inst = cur_inst; }
                    if (two && !(ANYHIT && best_prim != INVALID)) {      // (any-hit: the reference never runs the second test after a hit)
                        TRAY_CNT(tris);
                        if (t2 < best_t) { best_t = t2; best_prim = g2; if constexpr (INST) best_inst = cur_inst; }
                    }
                    if (ANYHIT && best_prim != INVALID) { sp &= SP_STEP - 1u; tri_y = 0u; cur_y = 0u; }   // drop the rest of the traversal
                    if (tri_y == 0u && cur_y < 0x01000000u) pop_or_retire();
                }
            }
        }
    }

    if (COUNT) {
        flush_counters(P.counters, lane, c_rays, c_nodes, c_tris, c_insts, c_hits);
        if (FRAME) flush_counters(P.counters + N_COUNTERS, lane, b_rays, b_nodes, b_tris, b_insts, b_hits);   // the bounce rays' slot
    }
#undef TRAY_CNT
}

// compact local order -> row-major frame (one thread per local work item)
template <typename T>
__global__ void untile_kernel(const __grid_constant__ FrameParams F, const T* __restrict__ src, T* __restrict__ dst) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= F.n_items) return;
    uint32_t px, py;
    if (item_to_pixel(F, j, px, py)) dst[(size_t)py * F.width + px] = src[j];
}

// all shards' compact RGBA (shard s at src + s * items_per_shard) -> row-major frame: one thread per PIXEL, so the frame is written
// in full 128-byte rows (the inverse of item_to_pixel)
__global__ void untile_shards_kernel(const uchar4* __restrict__ src, uint32_t width, uint32_t height, uint32_t tiles_x, uint32_t shards,
                                     uint64_t items_per_shard, uchar4* __restrict__ dst) {
    const uint32_t px = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y;
    if (px >= width || py >= height) return;
    const uint32_t k = (py >> 3) * tiles_x + (px >> 5);
    const uint32_t shard = k % shards, local_tile = k / shards;
    const uint32_t lx = px & 31u, ly = py & 7u;
    const uint32_t j = local_tile * 256u + (((ly >> 2) * 4u + (lx >> 3)) << 5) + ((ly & 3u) << 3) + (lx & 7u);
    dst[(size_t)py * width + px] = src[(size_t)shard * items_per_shard + j];
}

// ---- hit attributes (tray_cuda_hit_attributes): one thread per hit, after the traversal -------------------------------------
// A pass of its own rather than three more live values in trace_kernel (its INST instantiations sit at 64 registers with spills):
// it re-reads the ray, the hit and the triangle record (and the instance's transform), rebuilds the ray the triangle test saw and
// repeats the test's u, v and Ng through the helpers tri_test uses, so the values are the test's own bits.
struct AttrScene {
    const uint4* __restrict__ tris;
    uint64_t n_tris;
    const uint4* __restrict__ inst_xf;       // INST: InstanceRecords by instance id
    uint32_t n_inst;
    uint32_t variant;                        // TRAY_VARIANT_*: only ZERODIR_BOX_ONLY reaches the triangle test's direction
};

// {u, v, ng} of hit `prim` (of instance `inst`) on the ray {a = origin, tmin; b = direction, tmax}; all bytes 0xFF for a miss, a
// prim past the triangles or an instance past the instances, with nothing read for them
template <int TRI_STRIDE, bool INST>
__device__ __forceinline__ void hit_attr(const AttrScene& S, const float4& a, const float4& b, uint32_t prim, uint32_t inst, tray_hit_attr* out) {
    float* o = reinterpret_cast<float*>(out);
    if (prim == INVALID || prim >= S.n_tris || (INST && inst >= S.n_inst)) {
        const float nan = __uint_as_float(0xffffffffu);
        o[0] = nan; o[1] = nan; o[2] = nan; o[3] = nan; o[4] = nan;
        return;
    }
    RayConst r;
    const uint4* xf = INST ? S.inst_xf + (size_t)inst * INST_RECORD_U4 : nullptr;
    if constexpr (INST) {                    // the TLAS leaf's object-space ray, prepared as switch_ray prepares it
        const uint4 w0 = __ldg(xf), w1 = __ldg(xf + 1), w2 = __ldg(xf + 2);
        float ox, oy, oz, dx, dy, dz;
        xform_row(w0, a.x, a.y, a.z, b.x, b.y, b.z, ox, dx);
        xform_row(w1, a.x, a.y, a.z, b.x, b.y, b.z, oy, dy);
        xform_row(w2, a.x, a.y, a.z, b.x, b.y, b.z, oz, dz);
        prepare_ray(r, ox, oy, oz, dx, dy, dz, a.w, 0u);
    } else {
        prepare_ray(r, a.x, a.y, a.z, b.x, b.y, b.z, a.w, S.variant);
    }
    float v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz;
    tri_load<TRI_STRIDE>(S.tris, prim, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z);
    tri_normal<TRI_STRIDE>(S.tris, prim, e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz);
    float cx, cy, cz, inv_det, u, v;       // (r.tdx: the direction of the test, zero-patched unless ZERODIR_BOX_ONLY)
    tri_uv(r.ox, r.oy, r.oz, r.tdx, r.tdy, r.tdz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, ngx, ngy, ngz, cx, cy, cz, inv_det, u, v);
    if constexpr (INST) normal_to_world(xf, ngx, ngy, ngz);
    o[0] = u; o[1] = v; o[2] = ngx; o[3] = ngy; o[4] = ngz;
}

// n hits of a ray batch; INST: `inst_ids` holds the instance of every hit (tray_cuda_trace_instance)
template <int TRI_STRIDE, bool INST>
__global__ void __launch_bounds__(256) hit_attr_kernel(const AttrScene S, const tray_ray* __restrict__ rays, const tray_hit* __restrict__ hits,
                                                       const uint32_t* __restrict__ inst_ids, uint64_t n, tray_hit_attr* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t prim = __ldg(&hits[i].prim);
    const uint32_t inst = INST ? __ldg(inst_ids + i) : 0u;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (prim != INVALID) {
        const float4* rp = reinterpret_cast<const float4*>(rays + i);
        a = __ldg(rp); b = __ldg(rp + 1);
    }
    hit_attr<TRI_STRIDE, INST>(S, a, b, prim, inst, out + i);
}

// The last frame's attributes by local item (compact, as the frame's hit buffers): the primary ray as generated (`prays`), the
// bounce ray regenerated by bounce_ray from the primary hit and direction, as raygen_bounce_kernel and the FRAME kernel make it.
// Pixels that shot no bounce ray (outside the frame, or a primary miss) get the miss record.  Either output may be NULL.
template <int TRI_STRIDE, bool INST>
__global__ void __launch_bounds__(256) frame_attr_kernel(const __grid_constant__ FrameParams F, const AttrScene S, const tray_ray* __restrict__ prays,
                                                         const tray_hit* __restrict__ primary, const tray_hit* __restrict__ bounce,
                                                         const uint32_t* __restrict__ pinst, const uint32_t* __restrict__ binst,
                                                         tray_hit_attr* __restrict__ out_primary, tray_hit_attr* __restrict__ out_bounce) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= F.n_items) return;
    uint32_t px = 0, py = 0;
    const bool inside = item_to_pixel(F, j, px, py);
    const tray_hit ph = primary[j];
    const uint32_t pk = INST ? pinst[j] : 0u;
    const float4* rp = reinterpret_cast<const float4*>(prays + j);
    const float4 pa = __ldg(rp), pb = __ldg(rp + 1);
    if (out_primary) hit_attr<TRI_STRIDE, INST>(S, pa, pb, ph.prim, pk, out_primary + j);
    if (out_bounce) {
        const bool shoot = inside && ph.t < F32_MAX_ && ph.prim < S.n_tris && (!INST || pk < S.n_inst);   // rt_cpu.rs:61
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        uint32_t prim = INVALID;
        if (shoot) {
            float ox, oy, oz, dx, dy, dz;
            bounce_ray<TRI_STRIDE, INST>(F, S.tris, px, py, pb.x, pb.y, pb.z, ph.t, ph.prim, ox, oy, oz, dx, dy, dz,
                                         INST ? S.inst_xf + (size_t)pk * INST_RECORD_U4 : nullptr);
            a = make_float4(ox, oy, oz, 0.0f); b = make_float4(dx, dy, dz, F32_MAX_);   // Ray::new(o, dir, 0.0, f32::MAX)
            prim = bounce[j].prim;
        }
        hit_attr<TRI_STRIDE, INST>(S, a, b, prim, INST ? binst[j] : 0u, out_bounce + j);
    }
}

}  // namespace tray
