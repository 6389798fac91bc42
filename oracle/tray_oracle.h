/*
 * tray_oracle.h — CPU oracle for the CWBVH closest-hit path.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product (libtray_cuda.so) never links, loads or calls it.
 *
 * PARITY UNPINNED: the arithmetic of the reference's CPU path lives in the un-vendored, un-pinned git
 * dependency `obvhs` (Cargo.toml:26-29) and the reference holds no tests or golden vectors
 * (SURVEY.md §4, §8c), and no Rust toolchain exists here to run it.  This is a restatement of the
 * in-tree spec — see tray_oracle.c for the file:line each function follows.
 *
 * It is also the timed CPU baseline (bench.py cpu_baseline / --impl reference), so it is written to be a fair one: -O3,
 * OpenMP over rays like the reference's rayon loop, and the 8-child node test on AVX2 vectors where the CPU has them
 * (bit-identical to the scalar statement, tests/test_oracle.py).
 */
#ifndef TRAY_ORACLE_H
#define TRAY_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct orc_ray { float o[3]; float tmin; float d[3]; float tmax; } orc_ray;   /* 32 B */
typedef struct orc_hit { float t; uint32_t prim; } orc_hit;                           /*  8 B */
typedef struct orc_count { uint32_t nodes, tris, insts; } orc_count;                  /* per ray */

typedef struct orc_view {          /* ViewUniform, src/main.rs:589-617, 160 B */
    float view_inv[16];
    float proj_inv[16];
    float eye[3];
    float exposure;
    uint32_t tlas_start;
    uint32_t pad[3];
} orc_view;

typedef struct orc_scene {
    const uint8_t* nodes;  uint64_t n_nodes;      /* 80-byte CwBvhNode records */
    const uint8_t* tris;   uint64_t n_tris;  uint32_t tri_stride;   /* 48 or 64 (f32, parity path); 24 = f16 edges (wgpu path) */
    const uint32_t* blas_offsets; uint32_t n_instances; uint32_t tlas_start;
    int use_tlas;
} orc_scene;

typedef struct orc_totals { uint64_t rays, nodes, tris, insts, hits; } orc_totals;

#define ORC_INVALID_PRIM 0xFFFFFFFFu
#define ORC_RENDER_BOUNCE 0x1u
#define ORC_RENDER_RGBA   0x2u

/* variant switches (documented deltas between the CPU path and its HLSL twin, SURVEY.md §8c) */
#define ORC_VARIANT_DEFAULT     0u
#define ORC_VARIANT_BOX_DIVIDE  0x1u  /* box test divides by dir (query.hlsl:237-242) instead of * inv_dir */
#define ORC_VARIANT_TIE_LAST    0x2u  /* equal-t replaces (query.hlsl:120) instead of first-wins            */
#define ORC_VARIANT_BOX_TMIN_RAY 0x4u /* slab test clamps at ray.tmin instead of EPSILON = 1e-4 (query.hlsl:274,288) */
#define ORC_VARIANT_ZERODIR_BOX_ONLY 0x8u /* the zero-direction patch (query.hlsl:334) feeds the box test only; the triangle
                                           * test sees the caller's direction (as if obvhs `Ray::new` only guarded 1/d)  */
void orc_set_variant(uint32_t flags);

unsigned orc_abi_version(void);
/* the node test runs 8 children per AVX2 vector when the CPU has it (bit-identical to the scalar code); 0 forces scalar */
void orc_set_simd(int on);
int orc_simd(void);
int orc_max_threads(void);

/* Traversal stack capacity of orc_trace, orc_trace_any, orc_trace_oplog* and orc_render: 1 .. ORC_STACK_MAX entries, default
 * 32 (obvhs, cwbvh.rs:88); the CUDA kernels hold 48.  Returns 0, or -1 (unchanged) when `entries` is out of range. */
#define ORC_STACK_MAX 64
int orc_set_stack_limit(uint32_t entries);
uint32_t orc_stack_limit(void);

/* Per ray, the most entries its traversal holds on the stack at once, counted as the kernels count them: node groups pushed
 * behind a node's first child, and at a TLAS instance entry the rest of the instance group and the node group.  Closest-hit
 * (any_hit = 0) or any-hit traversal, traversed with ORC_STACK_MAX entries whatever orc_set_stack_limit says.
 * Returns 0, or -4 if a ray needs more than ORC_STACK_MAX (its need is then not meaningful). */
int orc_stack_need(const orc_scene* s, const orc_ray* rays, uint64_t n, uint32_t* need, int any_hit, int nthreads);

/* closest hit for n rays; returns 0, or -4 if any ray overflowed the stack (orc_set_stack_limit) */
int orc_trace(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits, orc_count* counts,
              orc_totals* totals, int nthreads);

/* any hit: the same traversal, stopped at the FIRST accepted triangle (hits[i] = that triangle and its t).
 * hits[i].prim != ORC_INVALID_PRIM  <=>  orc_trace finds a hit for the same ray. */
int orc_trace_any(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits, orc_count* counts,
                  orc_totals* totals, int nthreads);

/* per-ray step log ('N' node, 'T' triangle, 'I' instance entry) for warp-scheduling studies in tests/tools */
int orc_trace_oplog(const orc_scene* s, const orc_ray* rays, uint64_t n, const orc_count* counts,
                    uint8_t* ops, const uint64_t* offsets, int nthreads);
/* same, with triangle groups ('T' first / 'U' later triangle) and tmax updates (lower case) marked */
int orc_trace_oplog_detail(const orc_scene* s, const orc_ray* rays, uint64_t n, const orc_count* counts,
                           uint8_t* ops, const uint64_t* offsets, int nthreads);

/* O(rays x tris) reference: same triangle test, same first-wins rule in ascending index order;
 * also reports how many triangles tie with the winning t (for the tie census). */
int orc_brute_force(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits,
                    uint32_t* n_ties, int nthreads);

/* IEEE binary16 -> binary32 as the f16 triangle records are decoded (query.hlsl:75-85) */
float orc_half_to_float(uint16_t h);

/* ray/triangle test on one record; returns t or +inf */
float orc_intersect_tri(const orc_scene* s, uint32_t prim, const orc_ray* ray);

/* pixel -> primary ray (src/rt_cpu/rt_cpu.rs:38-55) */
void orc_primary_ray(const orc_view* v, uint32_t w, uint32_t h, uint32_t px, uint32_t py, orc_ray* out);
void orc_primary_rays(const orc_view* v, uint32_t w, uint32_t h, orc_ray* out, int nthreads);

/* primary hit -> bounce ray (src/rt_cpu/rt_cpu.rs:61-76); out->tmax = 0 when the primary missed */
void orc_bounce_ray(const orc_scene* s, const orc_view* v, const orc_ray* primary, const orc_hit* hit,
                    uint32_t px, uint32_t py, uint32_t frame_count, orc_ray* out);

/* one frame of rt_cpu::start's loop body (src/rt_cpu/rt_cpu.rs:35-91,102-107) */
int orc_render(const orc_scene* s, const orc_view* v, uint32_t w, uint32_t h, uint32_t frame_count,
               uint32_t flags, orc_hit* primary, orc_hit* bounce, orc_ray* bounce_rays, uint8_t* rgba,
               orc_totals* primary_totals, orc_totals* bounce_totals, int nthreads);

/* shading (src/rt_cpu/rt_cpu.rs:59, 82-88, 104-106): the grey level orc_render writes for a result of kind `mode` —
 * PRIMARY: 1/t; BOUNCE: t/(1+t), 1 for a miss; OCCLUSION: 0 for a hit, 1 for a miss (the kernels' ShadeMode numbering) */
#define ORC_SHADE_PRIMARY   1u
#define ORC_SHADE_BOUNCE    2u
#define ORC_SHADE_OCCLUSION 3u
uint8_t orc_shade(uint32_t mode, float t);

/* sampling utilities (src/rt_gpu/sampling.hlsl:5-51) */
uint32_t orc_uhash(uint32_t a, uint32_t b);
float orc_hash_noise(uint32_t x, uint32_t y, uint32_t frame);
void orc_sincos_tau(float u, float* s, float* c);

/* node box test alone (for known-answer tests): returns the 32-bit hit mask */
uint32_t orc_node_intersect(const uint8_t* node80, const orc_ray* ray, float tmax);

/* ---- build_ref.c: serial reference of the device builder (tray_build::build_tlas in build_gpu.cu) ----------------------
 * Morton sort -> PLOC -> reinsertion -> 8-wide collapse -> encode, single-threaded, byte for byte what the device builds.
 * The device reads the knobs from the environment (TRAY_CUDA_BUILD_REINSERT, _VISITS, _ROUNDS); here they are parameters.
 * Triangle records are not written: they depend only on prim_indices. */
typedef struct orc_build_params {
    uint32_t max_leaf;       /* 1 .. 3 */
    uint32_t radius;         /* PLOC search radius 1 .. 64; 0 means 14 */
    uint32_t passes;         /* reinsertion passes (device default 4) */
    uint32_t visits;         /* node visits per move search (192) */
    uint32_t rounds;         /* lock / apply rounds per pass (3) */
} orc_build_params;

typedef struct orc_build_stats {
    uint64_t n_nodes;
    uint32_t ploc_iterations, levels;         /* two-level builds: forest + TLAS */
    uint32_t reinsert_passes, reinsert_moves; /* the flat / forest run alone; all 0 when it ran no reinsertion */
    double sah_before, sah_after;             /* sum of the inner nodes' half-areas before / after the reinsertion */
} orc_build_stats;

typedef struct orc_bvh2_node {                /* 40 B; leaf: left = -1, right = primitive index */
    float lo[3], hi[3];
    int32_t left, right;
    uint32_t count;
    int32_t parent;                           /* -1 at a root */
} orc_bvh2_node;

typedef struct orc_build_result {
    uint8_t* nodes; uint64_t n_nodes;         /* 80-byte CwBvhNode records: BLAS forest | TLAS */
    uint32_t* prim_indices; uint64_t n_prims; /* BVH slot -> input triangle */
    uint32_t* blas_offsets; uint32_t n_instances, tlas_start;   /* two-level builds, TLAS-leaf order */
    int force_exact;                          /* some node exponent byte >= 167 */
    orc_build_stats stats;
    orc_bvh2_node* bvh2; uint32_t n_bvh2, n_bvh2_leaves;        /* final BVH2 of the flat / forest run */
} orc_build_result;

/* object_offsets == NULL: one flat BVH; otherwise n_objects + 1 offsets, one BLAS per object plus a TLAS.
 * Returns 0, -1 on bad arguments, -2 out of memory, -3 when the build fails as the device build would (a stalled PLOC). */
int orc_build_ref(const float* tris9, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects,
                  const orc_build_params* params, orc_build_result* out);
void orc_build_free(orc_build_result* r);

#ifdef __cplusplus
}
#endif
#endif
