/*
 * tray_cuda.h — C ABI of the B200-native CWBVH closest-hit traversal backend for tray_racing.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point is what a Rust `tray_cuda`
 * crate would bind with `extern "C"`; the slot it fills is the reference's software-GPU entry point
 *
 *     rt_gpu_software::start(event_loop, options, scene, bvh_bytes, instance_bytes, tri_bytes,
 *                            tlas_start) -> f32                  (src/rt_gpu/rt_gpu_software.rs:24-32)
 *
 * called from `cwbvh_gpu_runner` (src/rt_gpu/mod.rs:92-100,108-110), and — at ray-batch grain — the
 * CPU operator `Traversable::traverse(&self, ray: Ray) -> RayHit` (traversable/src/lib.rs:13-28,
 * src/cwbvh.rs:144-182).
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions return 0 on success and a
 * negative tray_status on failure; `tray_cuda_last_error()` returns a thread-local message.
 * Host buffers are borrowed for the duration of a call.  A `tray_scene` owns all device memory of
 * ONE device (the BVH is replicated: one scene per GPU, rays sharded by image tile); a `tray_group` is the
 * one-process form of that (devices[], n_devices — the SURVEY.md §8b proposal).
 * Not re-entrant per scene; distinct scenes may be driven from distinct host threads.
 */
#ifndef TRAY_CUDA_H
#define TRAY_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRAY_CUDA_ABI_VERSION 3u

/* ---- status codes -------------------------------------------------------------------------- */
typedef enum tray_status {
    TRAY_OK = 0,
    TRAY_ERR_ARG = -1,      /* bad pointer / size / stride / alignment                          */
    TRAY_ERR_CUDA = -2,     /* a CUDA runtime call failed (message has the cudaError string)     */
    TRAY_ERR_NO_DEVICE = -3,/* no CUDA device: there is NO CPU fallback by design                */
    TRAY_ERR_OVERFLOW = -4  /* traversal stack overflow was detected (BVH deeper than supported) */
} tray_status;

/* ---- POD records (layouts pinned by static asserts in the implementation) --------------------
 *
 * CWBVH node: obvhs `CwBvhNode`, #[repr(C)], 80 bytes, viewed as uint4[5] by the reference shader
 * (src/rt_gpu/rt_gpu_software_query.hlsl:40-43,219-264; encoder embree/src/bvh_embree_to_cwbvh.rs:172-185;
 * stride asserted at src/rt_gpu/mod.rs:70,105).  Passed as raw bytes, index 0 = root.            */
typedef struct tray_cwbvh_node {
    float    p[3];               /*  0: quantisation origin = node AABB min                      */
    uint8_t  e[3];               /* 12: biased f32 exponent per axis, scale = asfloat(e << 23)   */
    uint8_t  imask;              /* 15: bit i set <=> child slot i is an inner node              */
    uint32_t child_base_idx;     /* 16: index of first inner child (contiguous, slot order)      */
    uint32_t primitive_base_idx; /* 20: index of first triangle of this node                     */
    uint8_t  child_meta[8];      /* 24 */
    uint8_t  child_min_x[8];     /* 32 */
    uint8_t  child_max_x[8];     /* 40 */
    uint8_t  child_min_y[8];     /* 48 */
    uint8_t  child_max_y[8];     /* 56 */
    uint8_t  child_min_z[8];     /* 64 */
    uint8_t  child_max_z[8];     /* 72 */
} tray_cwbvh_node;               /* 80 bytes                                                      */

/* Triangle record, BVH order (tris[primitive_indices[i]], src/rt_cpu/mod.rs:38-43).
 * f32 like the CPU path's obvhs `RtTriangle` {v0, e1 = v0 - v1, e2 = v2 - v0, ng = cross(e1, e2)}
 * (SURVEY.md §8a row a10) — NOT the f16 `RtCompressedTriangle` of the wgpu path, which cannot meet
 * the 1e-5 parity bar.  Two strides are accepted for the parity path:
 *   48: {v0.xyz, pad, e1.xyz, pad, e2.xyz, pad}           (ng recomputed in-register, bit-identical)
 *   64: {v0, e1, e2, ng} each padded to 16 B              (byte image of [RtTriangle])
 * and, as the NON-parity variant of SURVEY.md §8 f4 (half the triangle bytes per test),
 *   24: the wgpu path's own `RtCompressedTriangle` byte image {v0: f32 x 3, e: u32 x 3},
 *       e[k] = half(v2 - v0)[k] | half(v1 - v0)[k] << 16  (src/rt_gpu/mod.rs:39-43,86; query.hlsl:75-85) */
typedef struct tray_tri48 {
    float v0[3], pad0;
    float e1[3], pad1;
    float e2[3], pad2;
} tray_tri48;

typedef struct tray_tri64 {
    float v0[3], pad0;
    float e1[3], pad1;
    float e2[3], pad2;
    float ng[3], pad3;
} tray_tri64;

typedef struct tray_tri24 {
    float    v0[3];
    uint32_t e[3];               /* e[k] = half(v2 - v0)[k] | half(v1 - v0)[k] << 16 */
} tray_tri24;

/* Ray = obvhs `Ray::new(origin, direction, tmin, tmax)` (src/rt_cpu/rt_cpu.rs:50-55).  32 bytes. */
typedef struct tray_ray {
    float origin[3];
    float tmin;
    float dir[3];
    float tmax;
} tray_ray;

/* Hit = the (t, primitive_id) pair of obvhs `RayHit` (embree/src/embree_managed.rs:52-57).
 * Miss: t = +inf, prim = 0xFFFFFFFF (RayHit::none()).  `prim` indexes the BVH-ordered triangle
 * array; in TLAS mode it is the GLOBAL triangle index (src/rt_gpu/mod.rs:45-47).                 */
typedef struct tray_hit {
    float    t;
    uint32_t prim;
} tray_hit;

#define TRAY_INVALID_PRIM 0xFFFFFFFFu

/* The surface at a hit (tray_cuda_hit_attributes): what the triangle test computed for the hit's triangle and ray.  20 bytes.
 * Miss record: all 20 bytes 0xFF (a NaN in every field).                                                                   */
typedef struct tray_hit_attr {
    float u, v;     /* barycentric weights of v1 and v2 (v0's is 1 - u - v), exactly as the triangle test computed them */
    float ng[3];    /* geometric normal, NOT normalised, in world space */
} tray_hit_attr;

/* `ViewUniform` (src/main.rs:589-617): column-major glam Mat4s, #[repr(C)], padded to 160 bytes. */
typedef struct tray_view {
    float    view_inv[16];
    float    proj_inv[16];
    float    eye[3];
    float    exposure;
    uint32_t tlas_start;
    uint32_t pad[3];
} tray_view;

/* Per-launch work counters (the reference's PROFILE_RT counters,
 * src/rt_gpu/rt_gpu_software_query.hlsl:377-379,407-409: aabb_hit_count/8 and tri_hit_count).     */
typedef struct tray_counters {
    uint64_t rays;       /* rays traced                                       */
    uint64_t nodes;      /* CWBVH nodes fetched (80 B each)                   */
    uint64_t tris;       /* triangle records tested                           */
    uint64_t instances;  /* blas_offsets lookups (TLAS mode)                  */
    uint64_t hits;       /* rays that ended with a hit                        */
} tray_counters;

/* The cost of ONE ray, as the counting kernels see it (the reference's PROFILE_RT heat map colours each pixel by its own ray's
 * counters, rt_gpu_software.hlsl:93-102).  nodes, tris and instances count exactly what tray_counters counts for that ray, so a
 * batch's or a frame's records sum to the tray_counters of the same call with counting on; the rays of an empty scene report
 * 0 nodes, as the totals do.  16 bytes, one aligned store per ray.                                                        */
typedef struct tray_ray_cost {
    uint32_t nodes;      /* CWBVH nodes fetched (the reference's aabb_hit_count / 8)                                  */
    uint32_t tris;       /* triangle records tested (tri_hit_count)                                                   */
    uint32_t instances;  /* TLAS leaf entries (blas_offsets lookups)                                                  */
    uint32_t stack;      /* most traversal-stack entries the ray held at once: the peak of the kernel's stack pointer, at
                          * most 48; a ray that needed more reports 48 and its call TRAY_ERR_OVERFLOW                    */
} tray_ray_cost;         /* 16 bytes */

typedef struct tray_scene_info {
    uint64_t n_nodes, n_tris;
    uint32_t tri_stride, n_instances, tlas_start, is_tlas;
    int32_t  device;
    uint32_t sm_count;
    uint64_t device_bytes;          /* bytes of device memory owned by the scene                  */
    uint64_t l2_bytes;              /* cudaDevAttrL2CacheSize                                     */
    uint64_t l2_persist_bytes;      /* persisting-L2 window actually applied to the node array    */
} tray_scene_info;

/* render flags */
#define TRAY_RENDER_BOUNCE     0x1u /* trace the 1-spp cosine "AO" bounce ray per hit pixel (rt_cpu.rs:61-88) */
#define TRAY_RENDER_RGBA       0x2u /* write pow(col,2.2)*255 RGBA8 (rt_cpu.rs:102-107)                       */
#define TRAY_RENDER_COUNTERS   0x4u /* run the counting build of the kernels (slower; fills tray_counters)    */
#define TRAY_RENDER_KEEP_RAYS  0x8u /* also store the generated bounce rays (for checkers)                    */
#define TRAY_RENDER_ANYHIT_AO  0x10u /* bounce rays stop at their FIRST hit (rt_cpu.rs:78-79 "a faster anyhit query"):
                                      * the bounce buffer holds that hit, RGBA is visibility (0 / 1) — not the reference image */
#define TRAY_RENDER_OVERLAP    0x20u /* ONE kernel launch for the frame: once the primary rays have all been handed out, warps with idle
                                      * lanes generate and trace the bounce rays of the 256-pixel tiles whose primary rays have all
                                      * retired, so the primary pass's drain phase is filled with bounce work.  Same hits, bounce rays
                                      * and image as the two-launch path; ms_primary is then the whole frame, ms_bounce 0.  Needs
                                      * TRAY_RENDER_BOUNCE; ignored with TRAY_RENDER_ANYHIT_AO. */

typedef struct tray_scene tray_scene;

/* ---- semantic switches (parity hardening) ---------------------------------------------------------------------------
 * Three semantics of the reference's CPU path are not in /root/reference but in the un-vendored obvhs crate, and a fourth
 * differs between that path and its in-tree HLSL twin (SURVEY.md §8c).  The DEFAULT kernels hard-code the CPU-path reading;
 * these flags make a scene run the other reading through a slower kernel with the switches at run time, so that a real
 * obvhs dump (INTEGRATION.md §5) can settle each one with a flag.  tests/ and scripts/variant_census.py count how many rays of
 * every BASELINE config change (prim, t) under each.  Closest-hit tray_cuda_trace* / tray_cuda_render without counters only. */
#define TRAY_VARIANT_BOX_DIVIDE       0x1u /* box test divides by the direction (query.hlsl:237-242) instead of * 1/d        */
#define TRAY_VARIANT_TIE_LAST         0x2u /* an equal-t triangle replaces the hit (query.hlsl:120 `tt <= t`), not first-wins */
#define TRAY_VARIANT_BOX_TMIN_RAY     0x4u /* slab test clamps at ray.tmin instead of EPSILON = 1e-4 (query.hlsl:274,288)     */
#define TRAY_VARIANT_ZERODIR_BOX_ONLY 0x8u /* the zero-direction patch (query.hlsl:334) feeds the box test only; the triangle
                                            * test sees the caller's direction                                               */
int tray_cuda_scene_set_variant(tray_scene* scene, uint32_t variant_flags);

/* ---- device / lifetime ---------------------------------------------------------------------- */

/* Number of CUDA devices visible; 0 (not an error) when there is none. */
int tray_cuda_device_count(void);

unsigned tray_cuda_abi_version(void);

/* Upload a CWBVH to `device`.  Mirrors the one-time storage-buffer upload of
 * rt_gpu_software.rs:177-180 with the argument meaning of `start()` (rt_gpu_software.rs:24-32):
 *   nodes/n_nodes   bvh_bytes as 80-byte nodes: flat BVH with root at 0, or BLAS0|BLAS1|..|TLAS with
 *                   the TLAS root at index `tlas_start` (src/rt_gpu/mod.rs:62-69,88-91,99)
 *   tris/n_tris     tri_bytes, BVH-ordered, stride 48, 64 or 24 (see above)
 *   blas_offsets    instance_bytes as u32: node offset of the BLAS behind TLAS leaf k
 *                   (src/rt_gpu/mod.rs:72-78); NULL / n_instances = 0 selects single-level traversal
 *   tlas_start      node index of the TLAS root; ignored when n_instances == 0                     */
int tray_cuda_scene_create(const void* nodes, uint64_t n_nodes,
                           const void* tris, uint64_t n_tris, uint32_t tri_stride,
                           const uint32_t* blas_offsets, uint32_t n_instances, uint32_t tlas_start,
                           int device, tray_scene** out_scene);

void tray_cuda_scene_destroy(tray_scene* scene);

/* ---- device-side builder (SURVEY.md §8 f3) ----------------------------------------------------------------
 * The step before the path: the reference builds its CwBvh on the CPU (`cwbvh_from_tris`, src/cwbvh.rs:24-105,
 * 0.95-2.9 s for its large scenes) and uploads it.  This builds the same FORMAT on the GPU — Morton sort, PLOC
 * clustering (search radius = obvhs' `search_distance`, default 14, src/main.rs:563-587), parallel reinsertion passes over the
 * binary tree (obvhs' reinsertion step), collapse to 8-wide,
 * octant slot order and quantisation as embree/src/bvh_embree_to_cwbvh.rs:85-186 — straight into the scene's device
 * buffers; only the triangle soup crosses PCIe.  (Two-level scenes: tray_cuda_scene_build_tlas.)  Deterministic: the same
 * triangles give the same bytes on every device, so per-rank replicas agree on every primitive id.
 *   tris9                n_tris x 9 floats (v0, v1, v2), HOST memory, borrowed for the call
 *   max_prims_per_leaf   1..3 (reference default 3, src/main.rs:575)
 *   search_radius        PLOC neighbourhood, 1..64; 0 = 14                                                  */
typedef struct tray_build_stats {
    uint64_t n_tris, n_nodes;
    uint32_t ploc_iterations, levels;
    float    ms_upload, ms_sort, ms_ploc, ms_collapse, ms_total;   /* host wall clock around synchronised phases */
    /* reinsertion passes between PLOC and the collapse (obvhs: reinsertion_batch_ratio, src/main.rs:563-587; environment
     * TRAY_CUDA_BUILD_REINSERT = number of passes, default 4, 0 = off): time, subtrees moved, SAH cost (sum of the inner nodes'
     * half areas) of the BVH2 before and after */
    float    ms_reinsert;
    uint32_t reinsert_passes, reinsert_moves;
    float    sah_before, sah_after;
} tray_build_stats;

int tray_cuda_scene_build(const float* tris9, uint64_t n_tris, uint32_t tri_stride, uint32_t max_prims_per_leaf,
                          uint32_t search_radius, int device, tray_scene** out_scene, tray_build_stats* out_stats);

/* Two-level build: object k = triangles [object_offsets[k], object_offsets[k+1]) (n_objects + 1 offsets, every object
 * non-empty).  One BLAS per object — all of them built together by a PLOC run that never merges across objects — and a
 * TLAS over the BLAS boxes, laid out exactly as `cwbvh_gpu_runner` lays out its `--tlas` buffers
 * (src/rt_gpu/mod.rs:53-100): BLAS nodes | TLAS nodes, TLAS root at tlas_start, blas_offsets in TLAS-leaf order, triangle
 * indices global.  tray_cuda_scene_info reports n_instances and tlas_start.                                       */
int tray_cuda_scene_build_tlas(const float* tris9, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects,
                               uint32_t tri_stride, uint32_t max_prims_per_leaf, uint32_t search_radius, int device,
                               tray_scene** out_scene, tray_build_stats* out_stats);

/* blas_offsets (n_instances x u32) of a two-level scene, to HOST memory */
int tray_cuda_scene_download_instances(tray_scene* scene, uint32_t* blas_offsets);

/* Copy a scene's BVH back to HOST memory (any pointer may be NULL): nodes n_nodes x 80 B, tris n_tris x tri_stride,
 * prim_indices n_tris x u32 (BVH slot -> input triangle; only scenes made by tray_cuda_scene_build have them —
 * others return TRAY_ERR_ARG when prim_indices != NULL).  For checkers and for the dump format of INTEGRATION.md. */
int tray_cuda_scene_download(tray_scene* scene, void* nodes, void* tris, uint32_t* prim_indices);

int tray_cuda_scene_info(const tray_scene* scene, tray_scene_info* out_info);

/* *out_exact = 1 when the scene's traversal takes the unfused (exact) node test at every node — some node has an exponent byte
 * >= 167 (a scale >= 2^40, where the fused test could overflow), or TRAY_CUDA_FORCE_EXACT is set — and 0 when it takes the
 * fused one.  Decided when the scene is made and again by every tray_cuda_scene_refit and tray_cuda_scene_refit_rebuild_tlas. */
int tray_cuda_scene_exact_node_test(const tray_scene* scene, int* out_exact);

/* ---- refit: move the triangles, keep the tree -----------------------------------------------------------------------------
 * Rewrites the triangle records from new vertex positions and re-encodes, for every node reachable from a root (node 0, or
 * every distinct blas_offsets entry and then tlas_start), only p, the exponents and the q bytes of the used slots
 * (child_meta != 0), tight over the new triangles exactly as the builders encode them; imask, child / primitive bases, child_meta,
 * empty slots, unreachable nodes, blas_offsets and prim_indices keep their bytes.  Two-level scenes: every BLAS first (a shared
 * one once), then the TLAS over the BLAS roots' boxes.  Afterwards the scene traces exactly like tray_cuda_scene_create on its
 * downloaded bytes, the exact node test included (on when some node's exponent byte is >= 167, or TRAY_CUDA_FORCE_EXACT).  A
 * refit with the scene's own triangles is the identity on trees of either builder.
 *   tris9     n_tris x 9 floats (v0, v1, v2) in the scene's triangle order: input order for scenes of tray_cuda_scene_build
 *             (slot k takes triangle prim_indices[k]), BVH slot order for scenes of tray_cuda_scene_create
 *   ms_refit  CUDA-event time of the refit launches (coordinate check, record pass, one launch per tree level), without the
 *             host upload and without the topology walk of the first call (NULL ok)
 * Synchronous.  Starts after every frame and batch trace already enqueued on the scene (every frame slot, the scene stream, the
 * copy streams) and returns with the new bytes in place: a frame rendered before keeps its results (download, readback, ray
 * costs), every later render or trace sees the new geometry.  tray_cuda_trace_device work on a caller's own stream is the
 * caller's to order: pass that stream to tray_cuda_scene_refit_device.
 * TRAY_ERR_ARG, with nothing changed: NULL scene or triangles, n_tris != the scene's, a coordinate that is not finite, triangles
 * whose extent on some axis overflows f32 (max - min = inf: no box over them can be encoded; the builders cannot build over them
 * either), or a tree the walk cannot refit (a node reached twice, a child or leaf index outside its array, a
 * blas_offsets entry outside the node array).  The first call walks the topology once and keeps it with the scene
 * (tray_scene_info.device_bytes counts it).  A scene with no triangles refits with n_tris = 0 and nothing happens. */
int tray_cuda_scene_refit(tray_scene* scene, const float* tris9, uint64_t n_tris, float* ms_refit);
/* the same with DEVICE memory; the refit starts after the work enqueued so far on `stream` (NULL: none) */
int tray_cuda_scene_refit_device(tray_scene* scene, const float* d_tris9, uint64_t n_tris, void* stream, float* ms_refit);

/* ---- refit every BLAS, rebuild the TLAS: objects that move as a whole ------------------------------------------------------
 * For two-level scenes whose objects move apart: a refit keeps the TLAS grouping instances that are no longer near each other,
 * a TLAS rebuild regroups them at a fraction of a full build's cost.
 *   1. Every BLAS is refit exactly as tray_cuda_scene_refit refits it: the same triangle records, the same bytes for every node
 *      below tlas_start.
 *   2. The TLAS primitives are the instances, each with its BLAS root's exact box, in canonical order: by blas_offsets value (the
 *      BLAS root node), ties (one BLAS under two instances) by TLAS-leaf position.  For scenes of tray_cuda_scene_build_tlas
 *      object k's root is node k, so the canonical order is object order and the new TLAS and blas_offsets are byte for byte
 *      those tray_cuda_scene_build_tlas builds on the moved triangles.
 *   3. The TLAS is built as tray_cuda_scene_build_tlas builds its TLAS: PLOC with search_radius (0 = 14, 1..64), the
 *      reinsertion passes (TRAY_CUDA_BUILD_REINSERT*), the collapse with max_prims_per_leaf (1..3).
 *   4. It is written over nodes [tlas_start, tlas_start + m); blas_offsets[j] becomes the root of TLAS leaf j; n_nodes becomes
 *      tlas_start + m and tlas_start stays.  A scene made by tray_cuda_scene_create holds exactly n_nodes: the first call that
 *      needs more grows its node array to tlas_start + n_instances + 1 nodes.  The first call also allocates the TLAS build's
 *      device scratch, n_instances x 384 B + 16 MiB, which the scene keeps: later calls allocate and free nothing on the device.
 *      tray_scene_info.device_bytes counts both.
 *   5. The exact node test is decided as the refit decides it, over the BLAS nodes, the new TLAS and the unreached nodes below
 *      tlas_start.  Later refits and rebuilds work on the new TLAS.
 *   ms   CUDA-event time on the scene stream from the coordinate check to the last TLAS write, the TLAS build's host round
 *        trips included, the host upload and the topology walk of a first call not; a first call's also holds its growth and
 *        scratch allocation (NULL ok)
 * Synchronous and ordered as tray_cuda_scene_refit.  TRAY_ERR_ARG, with nothing changed: every refusal of the refit, a scene
 * without a TLAS, max_prims_per_leaf or search_radius out of range, a node reached from a BLAS root at index >= tlas_start (the
 * TLAS is not the tail of the node array), a BLAS that reaches no triangle, or tlas_start + n_instances + 1 beyond 32 bits. */
int tray_cuda_scene_refit_rebuild_tlas(tray_scene* scene, const float* tris9, uint64_t n_tris, uint32_t max_prims_per_leaf,
                                       uint32_t search_radius, float* ms);
/* the same with DEVICE memory; starts after the work enqueued so far on `stream` (NULL: none) */
int tray_cuda_scene_refit_rebuild_tlas_device(tray_scene* scene, const float* d_tris9, uint64_t n_tris, uint32_t max_prims_per_leaf,
                                              uint32_t search_radius, void* stream, float* ms);

/* ---- instances: place BLAS by 3x4 transforms, rebuild only the TLAS -------------------------------------------------------
 * Makes a two-level scene INSTANCED: instance k is the BLAS whose root is blas_roots[k], placed by object_to_world + 12k (row-major
 * 3x4 [R | t]: world = R object + t).  Rigid motion is a new transform and a TLAS build, with no triangle and no BLAS node
 * touched; one BLAS may be placed any number of times.  Goes beyond the reference, whose runner has no instance transforms.
 *   Instance identity  instance k is the caller's index: it stays k across calls, rebuilds and TLAS-leaf permutations.
 *                      hits[i].prim keeps its meaning, the global triangle index; tray_cuda_trace_instance adds k.
 *   Valid roots        the distinct blas_offsets values the scene had when it was made.  Any BLAS may be used by any number of
 *                      instances, or by none.
 *   Inverse            world_to_object is computed on the host in double from object_to_world, as the adjugate over the
 *                      determinant with translation -W t, and rounded to nearest f32.
 *   TLAS primitive of instance k, in double, with no contraction:
 *                      1. the BLAS root's decoded box: the union over its used slots (child_meta != 0) of p + q 2^(e-127);
 *                      2. its 8 corners mapped by object_to_world as ((M_i0 x + M_i1 y) + M_i2 z) + M_i3;
 *                      3. the hull of the mapped corners;
 *                      4. every face moved out by 2^-18 max |coordinate of the hull| (it covers the rounding between the
 *                         world-space test at the TLAS and the object-space tests below it);
 *                      5. rounded outward to f32.
 *   Build              tray_cuda_scene_build_tlas's TLAS leg over those boxes in instance order: PLOC with search_radius (0 = 14,
 *                      1..64), the reinsertion passes, the collapse with max_prims_per_leaf (1..3).  Written at tlas_start;
 *                      blas_offsets[j] becomes blas_roots[leaf_instance[j]], n_nodes tlas_start + m, n_instances n_instances.
 *                      The exact node test is decided as tray_cuda_scene_refit_rebuild_tlas decides it.
 *   Memory             a first call, or a call with more instances than any before it, grows the node array to tlas_start + n + 1
 *                      nodes, blas_offsets, the instance records (64 B per instance, twice) and the TLAS build's scratch, and keeps
 *                      them: a call with no more instances than an earlier one allocates nothing on the device.
 *                      tray_scene_info.device_bytes counts all of it.
 *   ms                 CUDA-event time from the upload of the transforms to the last TLAS write (NULL ok)
 *   Scale              the tests hold objects of size 2^k placed at world size ~1, |k| <= 32 (strides 48 and 64; stride 24 keeps its
 *                      edges in f16, |k| <= 8), under powers of two, rotations, signed axis permutations, diag(2^-12, 1, 2^12),
 *                      strong shear and translations of 1e4, to a float64 world-space evaluation.  The object-space triangle
 *                      test's determinant grows as ~s^3 in the object size s and bounds the range: it leaves f32 near |k| = 42.
 *                      An object-space direction's zero components are patched at the instance's scale: with
 *                      2^r = the largest |W_ij| of row i rounded down to a power of two, component i becomes 2^-23 * 2^r where
 *                      |r| > 3, and 2^-23 (the patch of a plain scene) where |r| <= 3.  A bounce normal is brought to [1, 2) by a power of two before and after the transpose
 *                      of W, so its squared length (~s^6 otherwise) stays in f32.
 * Synchronous and ordered as tray_cuda_scene_refit: a frame rendered before keeps its results.  An instanced scene stays instanced.
 * TRAY_ERR_ARG, with nothing changed: NULL scene or pointers, n_instances == 0, a scene without a TLAS, semantic variants
 * (tray_cuda_scene_set_variant flags), an invalid root, max_prims_per_leaf or search_radius out of range, a coordinate of
 * object_to_world that is not finite, a zero determinant, a rounded inverse or a TLAS box that is not finite in f32, a tree the
 * refit walk refuses, a node reached from a BLAS root at index >= tlas_start, a BLAS that reaches no triangle, or
 * tlas_start + n_instances + 1 beyond 32 bits.
 * On an instanced scene: tray_cuda_scene_refit and tray_cuda_scene_set_variant are refused (its TLAS leaves are transformed boxes);
 * tray_cuda_scene_refit_rebuild_tlas(_device) refits every BLAS and then builds the TLAS as this call would, from the current roots
 * and transforms; tray_cuda_render always takes the two-launch path (TRAY_RENDER_OVERLAP is ignored) and bounce normals go to world
 * space through the transpose of world_to_object; the plain trace, trace_cost and render calls work and report no instances. */
int tray_cuda_scene_set_instances(tray_scene* scene, const uint32_t* blas_roots, const float* object_to_world, uint32_t n_instances,
                                  uint32_t max_prims_per_leaf, uint32_t search_radius, float* ms);
/* leaf_instance[j]: the instance k of TLAS leaf j (n_instances entries); world_to_object: n_instances x 12 floats by instance, as
 * the kernels use them.  Either may be NULL.  TRAY_ERR_ARG on a scene that is not instanced. */
int tray_cuda_scene_download_instance_xforms(tray_scene* scene, uint32_t* leaf_instance, float* world_to_object);
/* tray_cuda_trace / tray_cuda_trace_any (any_hit != 0) with one more output: instance_ids[i] = the instance k of hit i, 0xFFFFFFFF
 * for a miss.  TRAY_ERR_ARG on a scene that is not instanced. */
int tray_cuda_trace_instance(tray_scene* scene, const tray_ray* rays, uint64_t n, int any_hit, tray_hit* hits,
                             uint32_t* instance_ids, float* ms_kernel, float* ms_total);
/* the same with DEVICE buffers, as tray_cuda_trace_device */
int tray_cuda_trace_instance_device(tray_scene* scene, const tray_ray* d_rays, uint64_t n, int any_hit, tray_hit* d_hits,
                                    uint32_t* d_instance_ids, void* stream, float* ms_kernel);
/* The last frame's instance ids, row-major (w * h each, either NULL): 0xFFFFFFFF for misses, for other shards' pixels and for
 * pixels without a bounce ray.  TRAY_ERR_ARG on a scene that is not instanced, or for `bounce` after a frame without
 * TRAY_RENDER_BOUNCE. */
int tray_cuda_frame_download_instance(tray_scene* scene, uint32_t* primary, uint32_t* bounce);

/* ---- hit attributes: barycentrics and geometric normal of each hit ------------------------------------------------------------
 * For hit i of ray i, tray_hit_attr {u, v, ng} as the triangle test computed them for triangle hits[i].prim and that ray, bit for
 * bit (one pass over the hits after the traversal, with the test's own arithmetic):
 *   record     {v0, e1 = v0 - v1, e2 = v2 - v0} (stride 24: e1, e2 unpacked from f16 as the test unpacks them)
 *   direction  d = the ray's direction with zero components replaced by 2^-23 (FLT_EPSILON), as the traversal prepares it;
 *              under TRAY_VARIANT_ZERODIR_BOX_ONLY the caller's d
 *   u, v       det = dot(Ng, d), u = dot(cross(d, v0 - o), e2) / det (the weight of v1), v = dot(cross(d, v0 - o), e1) / det
 *              (the weight of v2), in f32 without contraction.  They depend on neither t nor tmax: closest-hit, any-hit and
 *              tie-variant hits all get their triangle's own values.
 *   ng         stride 64: the record's ng; strides 48 and 24: cross(e1, e2) in f32 (= cross(v0 - v1, v2 - v0)).  Not normalised and
 *              not flipped toward the ray.
 *   instances  (instanced scenes) u, v from the object-space ray of the traversal, o'_i = ((W_i0 o_x + W_i1 o_y) + W_i2 o_z) + W_i3,
 *              d'_i = (W_i0 d_x + W_i1 d_y) + W_i2 d_z then zero-patched at the instance's scale (tray_cuda_scene_set_instances,
 *              Scale) (W = world_to_object of instance instance_ids[i]); ng
 *              taken to world space as the bounce normal is, n'_i = (W_0i n_0 + W_1i n_1) + W_2i n_2, not normalised.  On other
 *              scenes object space is world space.
 *   miss       all 20 bytes 0xFF for prim == 0xFFFFFFFF, prim >= n_tris and, on an instanced scene, instance_ids[i] == 0xFFFFFFFF
 *              or >= n_instances; nothing is read for them.
 * instance_ids is required on an instanced scene (the output of tray_cuda_trace_instance; a plain tray_cuda_trace reports no
 * instance, so its hits on an instanced scene cannot be attributed) and must be NULL on any other scene: TRAY_ERR_ARG otherwise.
 * The scene's CURRENT triangles, transforms and variant flags are used: attributes of hits traced before a refit,
 * tray_cuda_scene_set_instances or tray_cuda_scene_set_variant describe the new geometry.
 * HOST buffers: copies in, one launch, copies out on the scene stream, then returns; n == 0 does nothing.  ms_kernel (NULL ok):
 * CUDA-event time of the launch. */
int tray_cuda_hit_attributes(tray_scene* scene, const tray_ray* rays, const tray_hit* hits, const uint32_t* instance_ids,
                             uint64_t n, tray_hit_attr* attrs, float* ms_kernel);
/* the same with DEVICE buffers, ordered as tray_cuda_trace_device: on `stream` (NULL: the scene stream), after the work enqueued
 * so far on the scene stream (so hits of a tray_cuda_trace_device there are complete); synchronises only when ms_kernel != NULL */
int tray_cuda_hit_attributes_device(tray_scene* scene, const tray_ray* d_rays, const tray_hit* d_hits, const uint32_t* d_instance_ids,
                                    uint64_t n, tray_hit_attr* d_attrs, void* stream, float* ms_kernel);
/* The last frame's attributes, row-major (w * h records each, either NULL): the primary hits' on the frame's primary rays, the
 * bounce hits' on its bounce rays, as tray_cuda_hit_attributes computes them.  The miss record for misses, other shards' pixels
 * and pixels without a bounce ray.  Synchronous.  TRAY_ERR_ARG, with nothing written: no frame rendered, `bounce` after a frame
 * without TRAY_RENDER_BOUNCE, or a scene changed since the frame by tray_cuda_scene_refit(_device),
 * tray_cuda_scene_refit_rebuild_tlas(_device), tray_cuda_scene_set_instances or tray_cuda_scene_set_variant (the attributes would
 * no longer describe that frame's hits; the next frame's call succeeds). */
int tray_cuda_frame_download_attributes(tray_scene* scene, tray_hit_attr* primary, tray_hit_attr* bounce);

/* ---- ray-batch operator: Traversable::traverse at batch grain (traversable/src/lib.rs:20) ----- */

/* Closest hit for `n` rays.  HOST buffers: the copy H2D of rays and D2H of hits are inside the
 * call (and inside *ms_total).  Batches of >= 2^18 rays run as a pipeline over chunks of 2^20 rays —
 * host threads stage the caller's rays into pinned slots, a copy stream uploads chunk i+1 while the
 * traversal kernel runs on chunk i and chunk i-1 is read back — so the caller's (pageable) memory is
 * only borrowed, never registered.  *ms_kernel is the CUDA-event time of the traversal kernel alone
 * for small batches, and the span of the GPU work (uploads it waited for included) for pipelined
 * ones.  Either timing pointer may be NULL.                                                       */
int tray_cuda_trace(tray_scene* scene, const tray_ray* rays, uint64_t n, tray_hit* hits,
                    float* ms_kernel, float* ms_total);

/* Same with DEVICE pointers (rays and hits already resident in HBM); launches on `stream`
 * (a cudaStream_t passed as void*, NULL = the scene's own stream) and does NOT synchronise unless
 * ms_kernel != NULL; when it does, it also reports a stack overflow of the batch (TRAY_ERR_OVERFLOW).  Without
 * ms_kernel the overflow is reported by the next synchronising call on the scene (tray_cuda_sync).   */
int tray_cuda_trace_device(tray_scene* scene, const tray_ray* d_rays, uint64_t n, tray_hit* d_hits,
                           void* stream, float* ms_kernel);

/* Any hit (SURVEY.md §8 f4): the same traversal, each ray stopped at the FIRST accepted triangle — the shadow /
 * occlusion query the reference wishes for at rt_cpu.rs:78-79 (its own intersects_bl_bvh, query.hlsl:440-445, runs
 * the closest-hit loop).  hits[i] = that triangle and its t, or {+inf, 0xFFFFFFFF}; hits[i].prim != 0xFFFFFFFF
 * exactly when tray_cuda_trace finds a hit for the same ray.                                              */
int tray_cuda_trace_any(tray_scene* scene, const tray_ray* rays, uint64_t n, tray_hit* hits,
                        float* ms_kernel, float* ms_total);
int tray_cuda_trace_any_device(tray_scene* scene, const tray_ray* d_rays, uint64_t n, tray_hit* d_hits,
                               void* stream, float* ms_kernel);

/* ---- frame operator: the render loop body (src/rt_cpu/rt_cpu.rs:35-91, rt_gpu_software.hlsl:47-144) */

/* Render the pixels of one frame that belong to shard `shard_index` of `shard_count`
 * (interleaved 32x8-pixel tiles: tile k belongs to shard k % shard_count; 0/1 = whole frame).
 * Rays are generated on the device from `view` (rt_cpu.rs:38-55); bounce rays per rt_cpu.rs:61-80.
 * Results stay on the device in compact per-shard buffers (tile order; every shard's buffers have the size of
 * shard 0's, so they can be gathered) — fetch them with tray_cuda_frame_download; returns after the
 * kernels have been enqueued on the scene stream unless a timing pointer is non-NULL.
 *   ms_primary / ms_bounce   CUDA-event time of the primary / bounce traversal kernel (NULL ok)   */
int tray_cuda_render(tray_scene* scene, const tray_view* view, uint32_t width, uint32_t height,
                     uint32_t frame_count, uint32_t flags, uint32_t shard_index, uint32_t shard_count,
                     float* ms_primary, float* ms_bounce);

/* Same frame, timed as a whole: *ms_frame is the CUDA-event time from the first ray-generation launch to the
 * end of the last traversal kernel — what the reference's timestamp queries bracket
 * (rt_gpu_software.rs:296-301,337-344).  Synchronises.                                                  */
int tray_cuda_render_timed(tray_scene* scene, const tray_view* view, uint32_t width, uint32_t height,
                           uint32_t frame_count, uint32_t flags, uint32_t shard_index, uint32_t shard_count,
                           float* ms_frame);

/* Number of pixels (= primary rays) shard `shard_index` owns for a width x height frame. */
uint64_t tray_cuda_shard_pixels(uint32_t width, uint32_t height, uint32_t shard_index, uint32_t shard_count);
/* Entries of that shard's compact buffers: its tiles x 256 (pixels outside the frame included as padding). */
uint64_t tray_cuda_shard_items(uint32_t width, uint32_t height, uint32_t shard_index, uint32_t shard_count);

/* Copy the last rendered frame to HOST buffers, each width*height entries in row-major pixel order
 * (pixels that belong to other shards are written as zero bytes).  Any pointer may be NULL.  `bounce_rays` receives the
 * generated bounce rays (tmax = 0 where the primary ray missed) so a checker can trace the very
 * same rays.                                                                                      */
int tray_cuda_frame_download(tray_scene* scene, tray_hit* primary, tray_hit* bounce,
                             tray_ray* bounce_rays, uint8_t* rgba);

/* Asynchronous readback of the last frame's RGBA8 (row-major, width*height*4 bytes) into HOST memory — pinned memory
 * if the copy is to overlap anything.  `begin` enqueues the untile on the frame's stream and the copy on the scene's own
 * copy stream and returns; the next tray_cuda_render overlaps the copy.  TRAY_READBACK_SLOTS staging buffers (slot 0 .. 3): cycle
 * through two or three of them, and `wait` for a slot before reading its host frame (begin on a slot still in flight waits for
 * it first).
 * After a frame rendered into a frame target (tray_cuda_scene_set_frame_target) the WHOLE target is read back — every
 * shard's pixels: call it on the device that owns the frame, stream-ordered after the barrier that completes the frame.
 * The error status travels with the frame: every frame slot has its own device error word, `begin` takes the word of the
 * frame it reads (on that frame's stream, so a later frame on the slot is not affected) and `wait` reports it — a stack
 * overflow as TRAY_ERR_OVERFLOW, once, for that frame alone, also with two frames in flight (tests/test_deep_stack.py). */
#define TRAY_READBACK_SLOTS 4
int tray_cuda_frame_readback_begin(tray_scene* scene, uint8_t* rgba_host, uint32_t slot);
int tray_cuda_frame_readback_wait(tray_scene* scene, uint32_t slot);

/* Device pointers of the last frame's buffers, for a caller that gathers them itself (NCCL / peer copy).
 * Layout: the COMPACT per-shard arrays in tile order — tray_cuda_shard_items(w, h, 0, shards) entries each (every shard's
 * buffers have shard 0's size), work item j = pixel (tile k = shard + (j / 256) * shards in row-major 32x8 tiles; inside a
 * tile 8 sub-tiles of 8x4 pixels) — NOT row-major frames: assemble a frame with tray_cuda_untile_rgba (or render into a
 * frame target).  The pointers are invalidated by a later tray_cuda_render that grows the buffers (a larger frame, fewer
 * shards, or the first TRAY_RENDER_KEEP_RAYS).                                                                         */
int tray_cuda_frame_device_ptrs(tray_scene* scene, void** d_primary, void** d_bounce, void** d_rgba);

/* Assemble a row-major width x height RGBA8 frame on the device from the compact buffer of ONE shard
 * (`d_compact` = that shard's rgba in local order, e.g. as received from another GPU by an NCCL gather).
 * Enqueued on the stream of the last rendered frame (the scene stream unless two frames are in flight); pixels of other
 * shards in `d_frame` are left untouched.                                                                            */
int tray_cuda_untile_rgba(tray_scene* scene, const void* d_compact, uint32_t width, uint32_t height,
                          uint32_t shard_index, uint32_t shard_count, void* d_frame);

/* ---- fused framebuffer exchange over peer memory (multi-GPU, SURVEY.md §8e option 1) ---------------------------
 * The reference has one GPU and one framebuffer (rt_gpu_software.rs:177-180).  With rays sharded over N GPUs the only
 * exchange is "every shard's pixels reach ONE frame".  Instead of gathering compact shards with a collective and
 * untiling them, a scene can be given a FRAME TARGET: a row-major width x height RGBA8 frame that may live on
 * another GPU of the box (a peer mapping opened from a CUDA IPC handle).  The traversal kernels then store each
 * finished pixel straight into that frame over NVLink while they are still tracing, so the transfer overlaps the
 * traversal pixel by pixel and no collective or untile launch remains (only a completion barrier).
 *
 *   rank 0:  tray_cuda_frame_alloc -> tray_cuda_ipc_export -> (send the 64-byte handle to the other ranks)
 *   rank k:  tray_cuda_ipc_open -> tray_cuda_scene_set_frame_target(scene, mapped_ptr)
 *   all:     tray_cuda_render(.. TRAY_RENDER_RGBA ..) per frame; synchronise streams + barrier = frame complete   */
int tray_cuda_frame_alloc(int device, uint64_t bytes, void** d_ptr);          /* plain cudaMalloc: IPC-exportable   */
int tray_cuda_frame_free(int device, void* d_ptr);
int tray_cuda_ipc_export(int device, void* d_ptr, uint8_t handle[64]);        /* cudaIpcGetMemHandle                */
int tray_cuda_ipc_open(int device, const uint8_t handle[64], void** d_ptr);   /* cudaIpcOpenMemHandle + peer access */
int tray_cuda_ipc_close(int device, void* d_ptr);
/* Completion flags for that exchange, WITHOUT a kernel: a 32-bit word in device memory (tray_cuda_frame_alloc; it may be a peer
 * mapping) written / awaited by the stream front-end (cuStreamWriteValue32 / cuStreamWaitValue32), on the stream of the last
 * rendered frame.  A collective kernel cannot do this job once two frames are in flight: it would wait for an SM slot that the
 * next frame's persistent grid only frees when it drains.
 *   rank k > 0, after tray_cuda_render:  tray_cuda_frame_signal(scene, &flags_on_rank0[k], seq)     — "my pixels of frame seq are there"
 *   rank 0, after tray_cuda_render:      tray_cuda_frame_wait_flag(scene, &flags[k], seq) for every k — whatever follows on that
 *                                        stream (a copy to the host) sees the complete frame
 * wait_flag passes once (int32)(*flag - value) >= 0, so sequence numbers may wrap.  Waits should be on LOCAL memory.
 * before_next_frame != 0 puts the wait on the stream the NEXT tray_cuda_render will use instead: that frame starts only once
 * the flag has been reached (e.g. "rank 0 has copied the previous frame out of the target this frame is about to overwrite"). */
int tray_cuda_frame_signal(tray_scene* scene, void* d_flag, uint32_t value);
int tray_cuda_frame_wait_flag(tray_scene* scene, const void* d_flag, uint32_t value, int before_next_frame);

/* The exchange as ONE DMA copy per shard instead of a store per pixel.  Pixels stored straight into a peer frame leave the SM as
 * scattered 4-byte NVLink writes (measured: +13 % frame time on a 1/8 shard of a 4K frame, 8 GPUs); the alternative keeps the
 * compact buffer local and moves it with the copy engine:
 *   every rank, after tray_cuda_render (no frame target):  tray_cuda_frame_push(scene, staging_on_rank0 + shard * items * 4)
 *                                                           (+ tray_cuda_frame_signal)      — no SM slot needed
 *   rank 0, once the flags of all shards are in:            tray_cuda_untile_shards(scene, staging, w, h, shards, frame)
 * `staging` holds the shards back to back, tray_cuda_shard_items(w, h, 0, shards) uchar4 entries each.  Both run on the stream of
 * the last rendered frame. */
int tray_cuda_frame_push(tray_scene* scene, void* d_dst);
int tray_cuda_untile_shards(tray_scene* scene, const void* d_staging, uint32_t width, uint32_t height, uint32_t shards, void* d_frame);

/* RGBA8 of every later tray_cuda_render goes to `d_frame` (row-major, width*height*4 bytes, on this or a peer
 * device) instead of the scene's compact buffer; NULL restores the compact buffer.  The pointer is borrowed.        */
int tray_cuda_scene_set_frame_target(tray_scene* scene, void* d_frame);

/* ---- frames in flight ---------------------------------------------------------------------------------------------------
 * A persistent-warp launch ends with a drain phase: the work cursor runs dry 0.2-0.4 ms before the last long rays finish and the
 * SMs empty out (DESIGN.md §5).  With n = 2 a scene keeps TWO frames in flight: it owns two sets of frame buffers and work
 * cursors, consecutive tray_cuda_render calls alternate between them, the first on the scene stream and the second on a
 * stream of its own, so the ray generation and primary pass of frame k+1 fill the SM slots frame k's drain phases leave empty
 * (the reference's wgpu loop also keeps frames in flight when it is not timing them: queue.submit + frame.present without a
 * wait, rt_gpu_software.rs:333-335; under --benchmark it waits for each frame's timestamps, :337-338 — which is what
 * tray_cuda_start does).  Per frame nothing changes — same launches, same results.  "The last frame" of the
 * download / readback / device_ptrs calls is the frame of the latest tray_cuda_render.  A caller that orders its own work
 * (a collective, a timing event) against the frames uses the calls below.  n = 1 (default) restores one frame at a time; n = 3
 * (TRAY_MAX_FRAMES_IN_FLIGHT) keeps one more frame queued, which pays on short frames (a 1/8 shard of a 4K frame). */
#define TRAY_MAX_FRAMES_IN_FLIGHT 3
int tray_cuda_scene_set_frames_in_flight(tray_scene* scene, uint32_t n);
/* `stream` (NULL = the scene stream) waits for every frame enqueued so far, whichever slot it runs in. */
int tray_cuda_scene_fence(tray_scene* scene, void* stream);
/* Frames enqueued from now on start after the work already enqueued on `stream`. */
int tray_cuda_scene_after(tray_scene* scene, void* stream);
/* The cudaStream_t (as void*) frames of slot `which` (0 .. 2) run on, or — which = -1 — the stream of the last rendered frame:
 * work enqueued on it right after tray_cuda_render (a collective that completes the frame, a copy) is ordered behind that
 * frame and ahead of the next frame of the same slot, without holding back the frame in the other slot. */
int tray_cuda_scene_frame_stream(tray_scene* scene, int which, void** stream);

/* Run all subsequent work of this scene on `stream` (a cudaStream_t as void*; NULL restores the scene's own
 * stream) — lets a host that already owns a stream (torch, NCCL) order its collectives after the kernels. */
int tray_cuda_scene_set_stream(tray_scene* scene, void* stream);

/* Wait for everything enqueued on the scene stream. */
int tray_cuda_sync(tray_scene* scene);

/* Counters of the last call that counted: a tray_cuda_render with TRAY_RENDER_COUNTERS, or — while tray_cuda_set_counting
 * is on — a tray_cuda_trace / tray_cuda_trace_any call or a timed (ms_kernel != NULL) tray_cuda_trace_device /
 * tray_cuda_trace_any_device call.  The flag counts the render that carries it and nothing else; tray_cuda_set_counting
 * governs batch traces alone.  Neither changes the other.                                                               */
int tray_cuda_counters(tray_scene* scene, tray_counters* primary, tray_counters* bounce);
int tray_cuda_set_counting(tray_scene* scene, int enabled);

/* ---- per-ray cost: which rays and pixels are expensive ------------------------------------------------------------------
 * The counting kernels also keep each ray's tray_ray_cost.  Hits, bounce rays and RGBA are bit-identical with ray costs on or
 * off; the kernels that do not count are not touched.  Under tray_cuda_scene_set_variant every call below that traces is
 * refused (TRAY_ERR_ARG) before it changes any state, as counting is.
 *
 * tray_cuda_trace / tray_cuda_trace_any (any_hit != 0), and their _device forms, with one more output: costs[i] is the cost
 * of rays[i].  They always run the counting kernels, and update tray_cuda_counters exactly when the plain calls would, that
 * is, while tray_cuda_set_counting is on.  HOST buffers for tray_cuda_trace_cost, DEVICE buffers (and `stream`, ms_kernel as
 * tray_cuda_trace_device) for tray_cuda_trace_cost_device, where d_costs must be 16-byte aligned.                          */
int tray_cuda_trace_cost(tray_scene* scene, const tray_ray* rays, uint64_t n, int any_hit, tray_hit* hits,
                         tray_ray_cost* costs, float* ms_kernel, float* ms_total);
int tray_cuda_trace_cost_device(tray_scene* scene, const tray_ray* d_rays, uint64_t n, int any_hit, tray_hit* d_hits,
                                tray_ray_cost* d_costs, void* stream, float* ms_kernel);
/* While enabled (default: off), every tray_cuda_render with TRAY_RENDER_COUNTERS also keeps the cost of each of its rays, in
 * buffers of the frame's slot that travel with the frame like its hits (frames in flight included).  A switch, not a render
 * flag: the set of TRAY_RENDER_* flags stays as it is.                                                                     */
int tray_cuda_scene_set_ray_cost(tray_scene* scene, int enabled);
/* The last frame's costs to HOST buffers, width*height records each in row-major pixel order: `primary` the primary ray of
 * each pixel, `bounce` its bounce ray.  Pixels of other shards, and bounce records of pixels that shot no bounce ray, are zero.
 * Either pointer may be NULL.  TRAY_ERR_ARG if the last frame kept no costs (rendered without TRAY_RENDER_COUNTERS or with ray
 * costs off), or bounce != NULL for a frame without TRAY_RENDER_BOUNCE.  Reports the frame's error status as
 * tray_cuda_frame_download does.  Per device of a tray_group: download each shard from tray_cuda_group_scene(i).           */
int tray_cuda_frame_download_cost(tray_scene* scene, tray_ray_cost* primary, tray_ray_cost* bounce);

/* ---- the slot itself ------------------------------------------------------------------------- */

/* Drop-in for rt_gpu_software::start (rt_gpu_software.rs:24-32): upload, then render frames for
 * `render_time_s` seconds with the reference's timing protocol (one untimed warm-up frame before
 * each timed frame when `benchmark` != 0, rt_gpu_software.rs:289-301), and return in *out_min_ms the
 * MIN frame time in ms (rt_gpu_software.rs:339,376) and in *out_mean_ms the mean (rt_cpu.rs:113).
 * `animate` advances frame_count per frame (rt_cpu.rs:95-97).  Before the timed loop a few untimed
 * frames of each of the two bit-identical frame paths (two launches / TRAY_RENDER_OVERLAP) pick the
 * faster one for this scene and frame size; the environment variable TRAY_CUDA_OVERLAP=0|1 forces it. */
int tray_cuda_start(const void* bvh_bytes, uint64_t bvh_len,
                    const void* instance_bytes, uint64_t instance_len,
                    const void* tri_bytes, uint64_t tri_len, uint32_t tri_stride,
                    uint32_t tlas_start, int use_tlas,
                    const tray_view* view, uint32_t width, uint32_t height,
                    float render_time_s, int benchmark, int animate, int device,
                    float* out_min_ms, float* out_mean_ms, uint32_t* out_frames);

/* ---- CPU-style hit records -----------------------------------------------------------------------------------------------
 * `Traversable::traverse` returns RayHit {primitive_id, geometry_id, ..} (traversable/src/lib.rs:13-28): on the CPU `--tlas`
 * path geometry_id is the BLAS (= object) index and primitive_id indexes that BLAS's own BVH-ordered triangle array
 * (src/cwbvh.rs:144-166), where the GPU path — and tray_hit — carry ONE global triangle index
 * (`primitive_base_idx += tri_offset`, src/rt_gpu/mod.rs:45-47).  Give the scene the runner's running `tri_offset` per object
 * (n_geometries + 1 entries, tri_offsets[0] = 0, tri_offsets[n] = n_tris) and convert:
 *   geometry_id[i]  = g with tri_offsets[g] <= hits[i].prim < tri_offsets[g + 1]     (0xFFFFFFFF for a miss, as RayHit::none())
 *   primitive_id[i] = hits[i].prim - tri_offsets[g]                                   (0xFFFFFFFF for a miss)
 * Without a table (n_geometries = 0: a flat scene, `CwBvhScene`) geometry_id is 0xFFFFFFFF and primitive_id = prim.
 * HOST buffers; the lookup runs on the scene's device. */
int tray_cuda_scene_set_geometry_offsets(tray_scene* scene, const uint32_t* tri_offsets, uint32_t n_geometries);
int tray_cuda_hits_to_geometry(tray_scene* scene, const tray_hit* hits, uint64_t n, uint32_t* geometry_id, uint32_t* primitive_id);

/* ---- one process, several GPUs --------------------------------------------------------------------------------------------
 * The slot `start(..) -> f32` is one call from one host thread (rt_gpu_software.rs:24-32).  A tray_group keeps that shape on
 * a box with several GPUs: the BVH is replicated on `devices[0..n)` (NULL = devices 0..n-1), the frame's 32x8 tiles are dealt
 * round-robin to the devices, and every device's pixels reach ONE row-major RGBA8 frame on devices[0] through peer access
 * (cudaDeviceEnablePeerAccess — no IPC handles, no NCCL, no second process): by one DMA copy of the device's compact shard plus
 * one untile launch on devices[0], or stored pixel by pixel from the traversal kernels (tray_cuda_group_set_exchange).
 * Frame completion is a set of events: devices[0]'s stream waits for the event each other device records behind its last
 * launch / copy.  Results are bit-identical to the single-GPU frame (tests/test_gpu_group.py).
 *   tray_cuda_group_render          enqueue one frame on every device (shard i of n on devices[i]); asynchronous
 *   tray_cuda_group_render_timed    same, synchronous: *ms_frame = CUDA-event time on devices[0] from before the first launch
 *                                   (no device starts earlier) to the frame being complete
 *   tray_cuda_group_readback_begin / _wait   the complete frame -> HOST memory (pinned for overlap), double-buffered like
 *                                   tray_cuda_frame_readback_begin; with two frames in flight the group alternates two targets
 *   tray_cuda_group_scene           borrow the scene of devices[i] (counters, hit downloads of its shard, set_variant ..)
 * Moving geometry: refit every replica, tray_cuda_scene_refit on tray_cuda_group_scene(i) for each i; the group has no refit
 * call of its own, as its caller would still loop over the devices.  The same for tray_cuda_scene_refit_rebuild_tlas: call it
 * on tray_cuda_group_scene(i) for each i; the replicas stay byte-identical.                                                   */
typedef struct tray_group tray_group;
int  tray_cuda_group_create(const void* nodes, uint64_t n_nodes, const void* tris, uint64_t n_tris, uint32_t tri_stride,
                            const uint32_t* blas_offsets, uint32_t n_instances, uint32_t tlas_start,
                            const int* devices, int n_devices, tray_group** out_group);
void tray_cuda_group_destroy(tray_group* group);
int  tray_cuda_group_size(const tray_group* group);
int  tray_cuda_group_scene(tray_group* group, int i, tray_scene** out_scene);
int  tray_cuda_group_set_frames_in_flight(tray_group* group, uint32_t n);
/* How the shards reach devices[0]'s frame: push != 0 (default) — every device keeps its compact shard and moves it with ONE peer DMA
 * copy (cudaMemcpyPeerAsync) into a staging array on devices[0], which untiles all shards in one launch; push == 0 — the traversal
 * kernels store finished pixels straight into the frame over peer access (scattered 4-byte NVLink writes: cheaper on sparse
 * frames, 13 % dearer on a fully covered 4K frame over 8 GPUs).  Same bytes either way. */
int  tray_cuda_group_set_exchange(tray_group* group, int push);
int  tray_cuda_group_render(tray_group* group, const tray_view* view, uint32_t width, uint32_t height,
                            uint32_t frame_count, uint32_t flags);
int  tray_cuda_group_render_timed(tray_group* group, const tray_view* view, uint32_t width, uint32_t height,
                                  uint32_t frame_count, uint32_t flags, float* ms_frame);
int  tray_cuda_group_readback_begin(tray_group* group, uint8_t* rgba_host, uint32_t slot);
int  tray_cuda_group_readback_wait(tray_group* group, uint32_t slot);
int  tray_cuda_group_frame_ptr(tray_group* group, void** d_frame);      /* devices[0] pointer of the last frame (row-major RGBA8) */
int  tray_cuda_group_sync(tray_group* group);

/* tray_cuda_start on several GPUs of the box: same arguments (the device list replaces `device`), same timing protocol, the
 * frame time being tray_cuda_group_render_timed's. */
int tray_cuda_start_multi(const int* devices, int n_devices,
                          const void* bvh_bytes, uint64_t bvh_len,
                          const void* instance_bytes, uint64_t instance_len,
                          const void* tri_bytes, uint64_t tri_len, uint32_t tri_stride,
                          uint32_t tlas_start, int use_tlas,
                          const tray_view* view, uint32_t width, uint32_t height,
                          float render_time_s, int benchmark, int animate,
                          float* out_min_ms, float* out_mean_ms, uint32_t* out_frames);

/* Roofline denominators measured on this device: streaming 16-byte read bandwidth (GB/s) over a buffer of `bytes`
 * swept `iters` times by a chip-filling grid.  A buffer well under the L2 size measures L2 bandwidth (the roof the
 * node array lives under, SURVEY.md §8d), one much larger than L2 measures HBM read bandwidth.                   */
int tray_cuda_bandwidth_probe(int device, uint64_t bytes, int iters, float* out_gbs);

/* The third denominator: what the L1 delivers to a GATHER — every lane of a warp reading its own 16-byte record from a
 * different 128-byte line of an L1-resident table of `bytes` (<= 64 KiB), which is how a traversal warp reads nodes and
 * triangles.  Grid and block shape of the traversal kernels; `iters` rounds of 8 independent loads per lane.  Reported as
 * GB/s over the whole chip (divide by SMs x clock for bytes per clock per SM).                                          */
int tray_cuda_l1_gather_probe(int device, uint32_t bytes, int iters, float* out_gbs);

const char* tray_cuda_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* TRAY_CUDA_H */
