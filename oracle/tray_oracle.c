/*
 * tray_oracle.c — CPU oracle for the 8-wide CWBVH closest-hit path.  TEST INFRASTRUCTURE ONLY.
 *
 * PARITY UNPINNED (see tray_oracle.h).  The reference's CPU arithmetic is in the un-vendored crate
 * `obvhs` (Cargo.toml:26-29, floating HEAD); its published algorithm is restated here from the
 * reference's own in-tree twin of it — the HLSL the author keeps in step with the Rust — and from the
 * reference's call sites.  Build with -ffp-contract=off: Rust/glam never contract a*b+c into an FMA.
 *
 * What follows what (all paths into /root/reference):
 *   node decode + 8 slab tests   src/rt_gpu/rt_gpu_software_query.hlsl:213-303
 *   octant word                  src/rt_gpu/rt_gpu_software_query.hlsl:314-326
 *   traversal loop               src/rt_gpu/rt_gpu_software_query.hlsl:328-438
 *   two-level traversal          src/rt_gpu/rt_gpu_software_query_tlas.hlsl:333-500
 *   ray/triangle test            src/rt_gpu/rt_gpu_software_query.hlsl:89-129 (f32 records as on the
 *                                CPU path, src/rt_cpu/mod.rs:42, traversable/src/lib.rs:47-51)
 *   pixel -> ray, bounce ray     src/rt_cpu/rt_cpu.rs:38-55, 61-80
 *   hash / sampling              src/rt_gpu/sampling.hlsl:5-51
 *   shading                      src/rt_cpu/rt_cpu.rs:59,82-88,102-107
 *
 * Where the CPU path and its HLSL twin are known to differ (SURVEY.md §8c) this file resolves TOWARD
 * THE CPU PATH and says so at the site; orc_set_variant() flips the two that touch the traversal.
 */
#include "tray_oracle.h"

#include <immintrin.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define F32_MAX 3.402823466e+38f
#define F32_EPSILON 1.1920929e-7f      /* sampling.hlsl:3 */
#define BOX_EPSILON 0.0001f            /* query.hlsl:274 */
#define ORC_STACK 32                   /* obvhs traversal stack depth, src/cwbvh.rs:87-89 */

static uint32_t g_variant = ORC_VARIANT_DEFAULT;
void orc_set_variant(uint32_t flags) { g_variant = flags; }
static uint32_t g_stack_limit = ORC_STACK;
int orc_set_stack_limit(uint32_t entries) {
    if (entries < 1 || entries > ORC_STACK_MAX) return -1;
    g_stack_limit = entries;
    return 0;
}
uint32_t orc_stack_limit(void) { return g_stack_limit; }
unsigned orc_abi_version(void) { return 3u; }
int orc_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

static inline float as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline uint32_t load_u32(const uint8_t* p) { uint32_t u; memcpy(&u, p, 4); return u; }
static inline float load_f32(const uint8_t* p) { float f; memcpy(&f, p, 4); return f; }
static inline uint32_t firstbithigh(uint32_t x) { return 31u - (uint32_t)__builtin_clz(x); }

/* glam Vec3A (SSE2) dot: (x*x' + y*y') + z*z', every op rounded (SURVEY.md §7 "bit-level float parity") */
static inline float dot3(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
/* glam cross: component = a.y*b.z - a.z*b.y etc., mul, mul, sub */
static inline void cross3(const float a[3], const float b[3], float o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}
/* glam Vec3A::normalize (SSE2): v / sqrt(dot(v,v)) per component */
static inline void normalize3(float v[3]) {
    float len = sqrtf(dot3(v, v));
    v[0] = v[0] / len; v[1] = v[1] / len; v[2] = v[2] / len;
}

/* ---- prepared ray: the state `Ray::new` + traverse_bvh set up once per ray ------------------- */
typedef struct prep_ray {
    float o[3], d[3], inv[3];
    float dt[3];        /* the direction the TRIANGLE test sees: d, or the unpatched one (ORC_VARIANT_ZERODIR_BOX_ONLY) */
    float tmin;
    float box_tmin;     /* lower clamp of the slab test: EPSILON (query.hlsl:274) or ray.tmin (ORC_VARIANT_BOX_TMIN_RAY) */
    uint32_t oct_inv4;
} prep_ray;

/* query.hlsl:334 zero-direction fix-up, then the cached reciprocal of obvhs `Ray` (CPU path,
 * SURVEY.md §8c vi: multiply by inv_direction), then query.hlsl:314-326. */
static inline void prepare_ray(const orc_ray* r, prep_ray* p) {
    for (int a = 0; a < 3; a++) {
        p->o[a] = r->o[a];
        p->d[a] = (r->d[a] == 0.0f) ? F32_EPSILON : r->d[a];
        p->inv[a] = 1.0f / p->d[a];
        p->dt[a] = (g_variant & ORC_VARIANT_ZERODIR_BOX_ONLY) ? r->d[a] : p->d[a];
    }
    p->tmin = r->tmin;
    p->box_tmin = (g_variant & ORC_VARIANT_BOX_TMIN_RAY) ? r->tmin : BOX_EPSILON;
    p->oct_inv4 = (p->d[0] < 0.0f ? 0u : 0x04040404u) | (p->d[1] < 0.0f ? 0u : 0x02020202u) |
                  (p->d[2] < 0.0f ? 0u : 0x01010101u);
}

/* ---- CwBvhNode::intersect_ray, twin cwbvh_node_intersect (query.hlsl:213-303) ---------------- */
static inline uint32_t node_intersect_scalar(const uint8_t* n, const prep_ray* r, float max_distance) {
    float p[3] = { load_f32(n + 0), load_f32(n + 4), load_f32(n + 8) };
    float adj_inv[3], adj_org[3];
    for (int a = 0; a < 3; a++) {
        float scale = as_float((uint32_t)n[12 + a] << 23);            /* query.hlsl:237-240 */
        if (g_variant & ORC_VARIANT_BOX_DIVIDE) {
            adj_inv[a] = scale / r->d[a];                              /* query.hlsl:241 */
            adj_org[a] = (p[a] - r->o[a]) / r->d[a];                   /* query.hlsl:242 */
        } else {
            adj_inv[a] = scale * r->inv[a];                            /* CPU path: * ray.inv_direction */
            adj_org[a] = (p[a] - r->o[a]) * r->inv[a];
        }
    }
    const uint8_t* meta = n + 24;
    const uint8_t* lo[3] = { n + 32, n + 48, n + 64 };
    const uint8_t* hi[3] = { n + 40, n + 56, n + 72 };
    uint32_t hit_mask = 0;
    for (int i = 0; i < 2; i++) {
        uint32_t meta4 = load_u32(meta + 4 * i);
        uint32_t is_inner4 = (meta4 & (meta4 << 1)) & 0x10101010u;     /* query.hlsl:251 */
        uint32_t inner_mask4 = (is_inner4 >> 4) * 0xffu;
        uint32_t bit_index4 = (meta4 ^ (r->oct_inv4 & inner_mask4)) & 0x1f1f1f1fu;
        uint32_t child_bits4 = (meta4 >> 5) & 0x07070707u;
        for (int j = 0; j < 4; j++) {
            int c = 4 * i + j;
            float tmin3[3], tmax3[3];
            for (int a = 0; a < 3; a++) {
                /* near/far plane by ray sign, query.hlsl:266-273 */
                uint8_t qn = r->d[a] < 0.0f ? hi[a][c] : lo[a][c];
                uint8_t qf = r->d[a] < 0.0f ? lo[a][c] : hi[a][c];
                tmin3[a] = (float)qn * adj_inv[a] + adj_org[a];        /* query.hlsl:285 (mul, add) */
                tmax3[a] = (float)qf * adj_inv[a] + adj_org[a];        /* query.hlsl:286 */
            }
            float tmin = fmaxf(fmaxf(fmaxf(tmin3[0], tmin3[1]), tmin3[2]), r->box_tmin);   /* :288 */
            float tmax = fminf(fminf(fminf(tmax3[0], tmax3[1]), tmax3[2]), max_distance);  /* :289 */
            if (tmin <= tmax) {                                                            /* :291 */
                uint32_t child_bits = (child_bits4 >> (8 * j)) & 0xffu;
                uint32_t bit_index = (bit_index4 >> (8 * j)) & 0xffu;
                hit_mask |= child_bits << bit_index;                                       /* :297 */
            }
        }
    }
    return hit_mask;
}

/* The same test with the 8 children in one AVX2 vector — what a CPU implementation worth timing does (obvhs runs it on
 * glam's SSE2 vectors).  Same operations in the same order per child (u8 -> f32 exact, mul, add, max, min, compare), so
 * the mask is bit-identical to node_intersect_scalar; it falls back to the scalar code when a per-node constant is not
 * finite (denormal direction components), where vector max/min and fmaxf/fminf treat NaN differently. */
__attribute__((target("avx2")))
static uint32_t node_intersect_avx2(const uint8_t* n, const prep_ray* r, float max_distance) {
    float adj_inv[3], adj_org[3];
    for (int a = 0; a < 3; a++) {
        float scale = as_float((uint32_t)n[12 + a] << 23);
        adj_inv[a] = scale * r->inv[a];
        adj_org[a] = (load_f32(n + 4 * a) - r->o[a]) * r->inv[a];
        if (!isfinite(adj_inv[a]) || !isfinite(adj_org[a])) return node_intersect_scalar(n, r, max_distance);
    }
    __m256 tn[3], tf[3];
    for (int a = 0; a < 3; a++) {
        const __m256 qlo = _mm256_cvtepi32_ps(_mm256_cvtepu8_epi32(_mm_loadl_epi64((const __m128i*)(n + 32 + 16 * a))));
        const __m256 qhi = _mm256_cvtepi32_ps(_mm256_cvtepu8_epi32(_mm_loadl_epi64((const __m128i*)(n + 40 + 16 * a))));
        const int neg = r->d[a] < 0.0f;
        const __m256 ai = _mm256_set1_ps(adj_inv[a]), ao = _mm256_set1_ps(adj_org[a]);
        tn[a] = _mm256_add_ps(_mm256_mul_ps(neg ? qhi : qlo, ai), ao);
        tf[a] = _mm256_add_ps(_mm256_mul_ps(neg ? qlo : qhi, ai), ao);
    }
    const __m256 tmin = _mm256_max_ps(_mm256_max_ps(_mm256_max_ps(tn[0], tn[1]), tn[2]), _mm256_set1_ps(r->box_tmin));
    const __m256 tmax = _mm256_min_ps(_mm256_min_ps(_mm256_min_ps(tf[0], tf[1]), tf[2]), _mm256_set1_ps(max_distance));
    unsigned hits = (unsigned)_mm256_movemask_ps(_mm256_cmp_ps(tmin, tmax, _CMP_LE_OQ));
    const uint32_t oct = r->oct_inv4 & 0xffu;
    uint32_t hit_mask = 0;
    while (hits) {
        const unsigned c = (unsigned)__builtin_ctz(hits);
        hits &= hits - 1;
        const uint32_t m = n[24 + c];
        const uint32_t inner = (m & (m << 1)) & 0x10u;
        const uint32_t bit_index = (m ^ (inner ? oct : 0u)) & 0x1fu;
        hit_mask |= ((m >> 5) & 7u) << bit_index;
    }
    return hit_mask;
}

static int g_use_avx2 = -1;
static inline uint32_t node_intersect(const uint8_t* n, const prep_ray* r, float max_distance) {
    if (g_use_avx2 < 0) g_use_avx2 = __builtin_cpu_supports("avx2") && !getenv("TRAY_ORACLE_SCALAR");
    if (g_use_avx2 && !(g_variant & ORC_VARIANT_BOX_DIVIDE)) return node_intersect_avx2(n, r, max_distance);
    return node_intersect_scalar(n, r, max_distance);
}
void orc_set_simd(int on) { g_use_avx2 = on && __builtin_cpu_supports("avx2"); }
int orc_simd(void) { if (g_use_avx2 < 0) g_use_avx2 = __builtin_cpu_supports("avx2") && !getenv("TRAY_ORACLE_SCALAR"); return g_use_avx2; }

uint32_t orc_node_intersect(const uint8_t* node80, const orc_ray* ray, float tmax) {
    prep_ray p; prepare_ray(ray, &p);
    return node_intersect(node80, &p, tmax);
}

/* ---- RtTriangle::intersect, twin intersect_ray_tri (query.hlsl:89-129) -----------------------
 * Record = {v0, e1 = v0 - v1, e2 = v2 - v0 [, ng = cross(e1,e2)]}, 16-byte padded vectors.
 * Returns t, or +inf for a miss, with the range test `t >= tmin && t <= tmax` of query.hlsl:120. */
/* IEEE binary16 -> binary32, exact (f16tof32 of unpack_2x16f_uint, query.hlsl:75-85) */
static inline float half_to_float(uint32_t h) {
    uint32_t sign = (h & 0x8000u) << 16, e = (h >> 10) & 0x1fu, m = h & 0x3ffu;
    if (e == 0) {
        if (m == 0) return as_float(sign);
        float f = (float)m * 5.9604644775390625e-8f;                   /* subnormal: m * 2^-24, exact */
        return (sign ? -f : f);
    }
    if (e == 31) return as_float(sign | 0x7f800000u | (m << 13));
    return as_float(sign | ((e + 112u) << 23) | (m << 13));
}

float orc_half_to_float(uint16_t h) { return half_to_float(h); }

/* v0, e1 = v0 - v1, e2 = v2 - v0 of one record.  Stride 48/64: the CPU path's f32 RtTriangle.  Stride 24: the wgpu
 * path's RtCompressedTriangle {v0: [f32;3], e: [u32;3]}, e[k] = half(e2[k]) | half((v1 - v0)[k]) << 16
 * (src/rt_gpu/mod.rs:39-43, unpack query.hlsl:75-85, e1 negated at query.hlsl:91) — NOT the parity path. */
static inline void tri_load(const uint8_t* rec, uint32_t stride, float v0[3], float e1[3], float e2[3]) {
    v0[0] = load_f32(rec + 0); v0[1] = load_f32(rec + 4); v0[2] = load_f32(rec + 8);
    if (stride == 24) {
        for (int k = 0; k < 3; k++) {
            uint32_t e = load_u32(rec + 12 + 4 * k);
            e2[k] = half_to_float(e & 0xffffu);
            e1[k] = -half_to_float(e >> 16);
        }
    } else {
        e1[0] = load_f32(rec + 16); e1[1] = load_f32(rec + 20); e1[2] = load_f32(rec + 24);
        e2[0] = load_f32(rec + 32); e2[1] = load_f32(rec + 36); e2[2] = load_f32(rec + 40);
    }
}

static inline float tri_intersect(const uint8_t* rec, uint32_t stride, const prep_ray* r, float tmax) {
    float v0[3], e1[3], e2[3];
    tri_load(rec, stride, v0, e1, e2);
    float ng[3];
    if (stride == 64) { ng[0] = load_f32(rec + 48); ng[1] = load_f32(rec + 52); ng[2] = load_f32(rec + 56); }
    else cross3(e1, e2, ng);                                           /* query.hlsl:93 */
    float c[3] = { v0[0] - r->o[0], v0[1] - r->o[1], v0[2] - r->o[2] };  /* :96 */
    float rr[3]; cross3(r->dt, c, rr);                                 /* :97 */
    float inv_det = 1.0f / dot3(ng, r->dt);                            /* :98 */
    float u = dot3(rr, e2) * inv_det;                                  /* :100 */
    float v = dot3(rr, e1) * inv_det;                                  /* :101 */
    float w = 1.0f - u - v;                                            /* :102 */
    uint32_t hit = as_uint(u) | as_uint(v) | as_uint(w);               /* :112 (-0.0 rejects) */
    /* :116 tests the sign bit.  On x86 an invalid operation (inf - inf, 0 * inf: dot(r, e2) or dot(r, e1) overflowing with
     * opposite signs) gives the default NaN 0xFFC00000, whose sign bit is set, so the CPU path rejects a NaN u, v or w.  Other
     * hosts' default NaN has the sign clear (aarch64: 0x7FC00000), so the rejection is written out: same answer everywhere.
     * (A NaN already in a record or ray is not a case the reference defines; it is rejected here as well.) */
    if (isnan(u) || isnan(v) || isnan(w)) return INFINITY;
    if (inv_det != 0.0f && (hit & 0x80000000u) == 0) {                 /* :116 */
        float t = dot3(ng, c) * inv_det;                               /* :118 */
        if (t >= r->tmin && t <= tmax) return t;                       /* :119 (tmin = ray.tmin on the CPU path) */
    }
    return INFINITY;
}

float orc_intersect_tri(const orc_scene* s, uint32_t prim, const orc_ray* ray) {
    prep_ray p; prepare_ray(ray, &p);
    return tri_intersect(s->tris + (uint64_t)prim * s->tri_stride, s->tri_stride, &p, ray->tmax);
}

/* closest-hit update.  CPU path (obvhs ray_traverse): `if t < ray.tmax` — the FIRST of equal-t
 * triangles wins; the HLSL twin's `tt <= t` (query.hlsl:120) lets the LAST win (SURVEY.md §8a a11). */
static inline int closer(float t, float tmax) {
    return (g_variant & ORC_VARIANT_TIE_LAST) ? (t <= tmax) : (t < tmax);
}

/* ---- CwBvh::ray_traverse / ray_traverse_tlas_blas; twins query.hlsl:328-438, query_tlas.hlsl:333-500 */
/* `any_hit`: stop at the first accepted triangle (the "faster anyhit query" rt_cpu.rs:78-79 asks for; the reference's
 * own intersects_bl_bvh, query.hlsl:440-445, runs the full closest-hit loop).  Same order of tests up to that point. */
static int g_oplog_detail = 0;   /* step log flavour (orc_trace_oplog_detail): 'T'/'U' first / later triangle of a group, lower case = the test moved tmax */
/* `cap`: stack entries the traversal may hold; `peak` (optional): the most it held at once */
static int trace_one_ex(const orc_scene* s, const orc_ray* ray, orc_hit* out, orc_count* cnt, uint8_t* oplog, int any_hit,
                        uint32_t cap, uint32_t* peak) {
    uint32_t n_ops = 0;   /* optional step log: 'N' node fetch+test, 'T' triangle test, 'I' instance entry */
    prep_ray r; prepare_ray(ray, &r);
    uint32_t stack[ORC_STACK_MAX][2];
    uint32_t size = 0, max_size = 0;
    const int tlas = s->use_tlas;
    uint32_t tlas_stack_size = 0xFFFFFFFFu;                /* query_tlas.hlsl:343 INVALID = in the TLAS */
    uint32_t bvh_offset = tlas ? s->tlas_start : 0u;       /* query_tlas.hlsl:344 */
    uint32_t cur_x = 0, cur_y = 0x80000000u;               /* root group, query.hlsl:343 */
    float best_t = ray->tmax;                              /* ray.tmax shrinks as hits are found */
    uint32_t best_prim = ORC_INVALID_PRIM;
    uint32_t n_nodes = 0, n_tris = 0, n_insts = 0;
    int overflow = 0;
    if (s->n_nodes == 0) { cur_y = 0; }

    for (;;) {
        uint32_t tri_x, tri_y;
        if (cur_y & 0xff000000u) {                                         /* query.hlsl:354 */
            uint32_t hits_imask = cur_y;
            uint32_t child_index_offset = firstbithigh(hits_imask);        /* :358 */
            uint32_t child_index_base = cur_x;
            cur_y &= ~(1u << child_index_offset);                          /* :362 */
            if (cur_y & 0xff000000u) {                                     /* :365-368 */
                if (size >= cap) { overflow = 1; break; }
                stack[size][0] = cur_x; stack[size][1] = cur_y; size++;
                if (size > max_size) max_size = size;
            }
            uint32_t slot_index = (child_index_offset - 24u) ^ (r.oct_inv4 & 0xffu);      /* :370 */
            uint32_t relative_index = (uint32_t)__builtin_popcount(hits_imask & ~(0xffffffffu << slot_index)); /* :371 */
            uint32_t child_node_index = child_index_base + relative_index;                /* :373 */
            const uint8_t* node = s->nodes + (uint64_t)(bvh_offset + child_node_index) * 80u;  /* tlas:383 */
            n_nodes++;                                                     /* PROFILE_RT aabb_hit_count/8, :377-379 */
            if (oplog) oplog[n_ops++] = 'N';
            uint32_t hitmask = node_intersect(node, &r, best_t);           /* :380 */
            uint32_t imask = node[15];                                     /* :381 */
            cur_x = load_u32(node + 16);                                   /* :383 */
            tri_x = load_u32(node + 20);                                   /* :384 */
            cur_y = (hitmask & 0xff000000u) | imask;                       /* :386 */
            tri_y = hitmask & 0x00ffffffu;                                 /* :387 */
        } else {
            tri_x = cur_x; tri_y = cur_y;                                  /* :391 */
            cur_x = 0; cur_y = 0;
        }

        int first_of_group = 1;
        while (tri_y != 0) {                                               /* :396 */
            uint32_t local = firstbithigh(tri_y);                          /* :398 */
            tri_y &= ~(1u << local);                                       /* :401 */
            uint32_t global = tri_x + local;                               /* :403 */
            if (tlas && tlas_stack_size == 0xFFFFFFFFu) {
                /* TLAS leaf: `global` is an instance slot (query_tlas.hlsl:410-446) */
                if (tri_y != 0) {
                    if (size >= cap) { overflow = 1; break; }
                    stack[size][0] = tri_x; stack[size][1] = tri_y; size++;       /* tlas:420-423 */
                    if (size > max_size) max_size = size;
                }
                if (cur_y & 0xff000000u) {
                    if (size >= cap) { overflow = 1; break; }
                    stack[size][0] = cur_x; stack[size][1] = cur_y; size++;       /* tlas:425-428 */
                    if (size > max_size) max_size = size;
                }
                tlas_stack_size = size;                                           /* tlas:431 */
                bvh_offset = s->blas_offsets[global];                             /* tlas:439 */
                n_insts++;
                if (oplog) oplog[n_ops++] = 'I';
                cur_x = 0; cur_y = 0x80000000u;                                   /* tlas:443 */
                break;
            }
            n_tris++;                                                      /* PROFILE_RT tri_hit_count, :407-409 */
            float t = tri_intersect(s->tris + (uint64_t)global * s->tri_stride, s->tri_stride, &r, best_t);
            if (oplog) {
                uint8_t c = 'T';
                if (g_oplog_detail) { c = first_of_group ? 'T' : 'U'; if (closer(t, best_t)) c |= 0x20; }
                oplog[n_ops++] = c; first_of_group = 0;
            }
            if (closer(t, best_t)) { best_t = t; best_prim = global; }     /* :410-413 with the CPU tie rule */
            if (any_hit && best_prim != ORC_INVALID_PRIM) break;
        }
        if (overflow) break;
        if (any_hit && best_prim != ORC_INVALID_PRIM) break;

        if ((cur_y & 0xff000000u) == 0) {                                  /* :417 */
            if (size == 0) break;                                          /* :420-424 */
            if (tlas && size == tlas_stack_size) {                         /* tlas:480-486 */
                tlas_stack_size = 0xFFFFFFFFu;
                bvh_offset = s->tlas_start;
            }
            size--;
            cur_x = stack[size][0]; cur_y = stack[size][1];                /* :426 */
        }
    }
    if (best_prim != ORC_INVALID_PRIM) { out->t = best_t; out->prim = best_prim; }
    else { out->t = INFINITY; out->prim = ORC_INVALID_PRIM; }              /* RayHit::none() */
    if (cnt) { cnt->nodes = n_nodes; cnt->tris = n_tris; cnt->insts = n_insts; }
    if (peak) *peak = max_size;
    return overflow ? -4 : 0;
}

static int trace_one(const orc_scene* s, const orc_ray* ray, orc_hit* out, orc_count* cnt, uint8_t* oplog) {
    return trace_one_ex(s, ray, out, cnt, oplog, 0, g_stack_limit, NULL);
}

int orc_trace_any(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits, orc_count* counts,
                  orc_totals* totals, int nthreads) {
    int rc = 0;
    uint64_t tn = 0, tt = 0, ti = 0, th = 0;
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(dynamic, 2048) num_threads(nthreads) reduction(+:tn,tt,ti,th) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        orc_count c;
        int e = trace_one_ex(s, &rays[i], &hits[i], &c, NULL, 1, g_stack_limit, NULL);
        if (e < rc) rc = e;
        if (counts) counts[i] = c;
        tn += c.nodes; tt += c.tris; ti += c.insts; th += hits[i].prim != ORC_INVALID_PRIM;
    }
    if (totals) { totals->rays = n; totals->nodes = tn; totals->tris = tt; totals->insts = ti; totals->hits = th; }
    return rc;
}

int orc_trace(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits, orc_count* counts,
              orc_totals* totals, int nthreads) {
    int rc = 0;
    uint64_t tn = 0, tt = 0, ti = 0, th = 0;
    if (nthreads <= 0) nthreads = orc_max_threads();
    /* rayon into_par_iter over rays, src/rt_cpu/rt_cpu.rs:35-37 */
#pragma omp parallel for schedule(dynamic, 2048) num_threads(nthreads) reduction(+:tn,tt,ti,th) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        orc_count c;
        int e = trace_one(s, &rays[i], &hits[i], &c, NULL);
        if (e < rc) rc = e;
        if (counts) counts[i] = c;
        tn += c.nodes; tt += c.tris; ti += c.insts; th += hits[i].prim != ORC_INVALID_PRIM;
    }
    if (totals) { totals->rays = n; totals->nodes = tn; totals->tris = tt; totals->insts = ti; totals->hits = th; }
    return rc;
}

int orc_stack_need(const orc_scene* s, const orc_ray* rays, uint64_t n, uint32_t* need, int any_hit, int nthreads) {
    int rc = 0;
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(dynamic, 2048) num_threads(nthreads) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        orc_hit h;
        int e = trace_one_ex(s, &rays[i], &h, NULL, NULL, any_hit, ORC_STACK_MAX, &need[i]);
        if (e < rc) rc = e;
    }
    return rc;
}

/* Per-ray step log for scheduling studies (tests/tools): offsets[i]..offsets[i+1] index `ops`, one byte per step in
 * the ray's own order.  `counts` must come from a previous orc_trace over the same rays. */
int orc_trace_oplog(const orc_scene* s, const orc_ray* rays, uint64_t n, const orc_count* counts,
                    uint8_t* ops, const uint64_t* offsets, int nthreads) {
    int rc = 0;
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(dynamic, 2048) num_threads(nthreads) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        orc_hit h; orc_count c;
        int e = trace_one(s, &rays[i], &h, &c, ops + offsets[i]);
        if (e < rc) rc = e;
        if (c.nodes + c.tris + c.insts != counts[i].nodes + counts[i].tris + counts[i].insts) rc = -5;
    }
    return rc;
}

/* The same log with triangle groups and tmax updates marked: 'T' / 'U' = first / later triangle of a group, lower case =
 * the test moved the ray's tmax (tests/tools/sched_sim.c, policy 4). */
int orc_trace_oplog_detail(const orc_scene* s, const orc_ray* rays, uint64_t n, const orc_count* counts,
                           uint8_t* ops, const uint64_t* offsets, int nthreads) {
    g_oplog_detail = 1;
    const int rc = orc_trace_oplog(s, rays, n, counts, ops, offsets, nthreads);
    g_oplog_detail = 0;
    return rc;
}

int orc_brute_force(const orc_scene* s, const orc_ray* rays, uint64_t n, orc_hit* hits,
                    uint32_t* n_ties, int nthreads) {
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        prep_ray r; prepare_ray(&rays[i], &r);
        float best = rays[i].tmax; uint32_t prim = ORC_INVALID_PRIM; uint32_t ties = 0;
        for (uint64_t k = 0; k < s->n_tris; k++) {
            /* full-range test (tmax = ray.tmax) so that ties with the winner can be counted */
            float t = tri_intersect(s->tris + k * s->tri_stride, s->tri_stride, &r, rays[i].tmax);
            if (t < best) { best = t; prim = (uint32_t)k; ties = 1; }
            else if (t == best && prim != ORC_INVALID_PRIM) ties++;
        }
        if (prim != ORC_INVALID_PRIM) { hits[i].t = best; hits[i].prim = prim; }
        else { hits[i].t = INFINITY; hits[i].prim = ORC_INVALID_PRIM; }
        if (n_ties) n_ties[i] = ties;
    }
    return 0;
}

/* ---- camera -> primary ray (src/rt_cpu/rt_cpu.rs:38-55) -------------------------------------- */
/* glam Mat4 * Vec4 (column-major): ((c0*x + c1*y) + c2*z) + c3*w, mul and add rounded separately */
static inline void mat4_mul_vec4(const float m[16], const float v[4], float o[4]) {
    for (int k = 0; k < 4; k++)
        o[k] = ((m[0 + k] * v[0] + m[4 + k] * v[1]) + m[8 + k] * v[2]) + m[12 + k] * v[3];
}

void orc_primary_ray(const orc_view* vw, uint32_t w, uint32_t h, uint32_t px, uint32_t py, orc_ray* out) {
    float uvx = (float)px / (float)w;                    /* frag_coord.as_vec2() / target_size */
    float uvy = (float)py / (float)h;
    uvy = 1.0f - uvy;
    float ndcx = uvx * 2.0f - 1.0f, ndcy = uvy * 2.0f - 1.0f;
    float clip[4] = { ndcx, ndcy, 1.0f, 1.0f };
    float vs[4]; mat4_mul_vec4(vw->proj_inv, clip, vs);
    float ww = vs[3];
    vs[0] = vs[0] / ww; vs[1] = vs[1] / ww; vs[2] = vs[2] / ww; vs[3] = vs[3] / ww;   /* vs /= vs.w */
    float wp[4]; mat4_mul_vec4(vw->view_inv, vs, wp);
    float d[3] = { wp[0] - vw->eye[0], wp[1] - vw->eye[1], wp[2] - vw->eye[2] };
    normalize3(d);
    out->o[0] = vw->eye[0]; out->o[1] = vw->eye[1]; out->o[2] = vw->eye[2];
    out->tmin = 0.0f;
    out->d[0] = d[0]; out->d[1] = d[1]; out->d[2] = d[2];
    out->tmax = F32_MAX;                                  /* Ray::new(eye, dir, 0.0, f32::MAX) */
}

void orc_primary_rays(const orc_view* v, uint32_t w, uint32_t h, orc_ray* out, int nthreads) {
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(static) num_threads(nthreads)
    for (int64_t i = 0; i < (int64_t)w * h; i++)
        orc_primary_ray(v, w, h, (uint32_t)(i % w), (uint32_t)(i / w), &out[i]);   /* rt_cpu.rs:38-41 */
}

/* ---- sampling.hlsl:5-51 ---------------------------------------------------------------------- */
uint32_t orc_uhash(uint32_t a, uint32_t b) {
    uint32_t x = (a * 1597334673u) ^ (b * 3812015801u);
    x = x ^ (x >> 16); x *= 0x7feb352du;
    x = x ^ (x >> 15); x *= 0x846ca68bu;
    x = x ^ (x >> 16);
    return x;
}
float orc_hash_noise(uint32_t x, uint32_t y, uint32_t frame) {
    uint32_t urnd = orc_uhash(x, (y << 11) + frame);
    return (float)urnd * (1.0f / (float)0xffffffffu);      /* unormf, sampling.hlsl:17-20 */
}

/* sin(2*pi*u), cos(2*pi*u) for u in [0,1].  The reference calls the platform's sin/cos on u*TAU
 * (sampling.hlsl:30-36), which is not bit-portable between any two machines; the bounce-ray
 * DIRECTION is an input distribution, not a parity item, so the oracle and the CUDA kernel both use
 * this fixed quadrant reduction + fmaf Horner polynomial, which IS bit-reproducible everywhere. */
void orc_sincos_tau(float u, float* s, float* c) {
    float q4 = u * 4.0f;
    float qf = rintf(q4);
    float r = q4 - qf;                                      /* exact, |r| <= 0.5 */
    float x = r * 1.57079632679489661923f;
    float x2 = x * x;
    float sp = fmaf(x2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(sp, x2, -1.6666654611e-1f);
    float sn = fmaf(x * x2, sp, x);
    float cp = fmaf(x2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(cp, x2, 4.166664568298827e-2f);
    float cs = fmaf(x2 * x2, cp, fmaf(x2, -0.5f, 1.0f));
    int q = (int)qf & 3;
    if (q == 0) { *s = sn; *c = cs; }
    else if (q == 1) { *s = cs; *c = -sn; }
    else if (q == 2) { *s = -sn; *c = -cs; }
    else { *s = -cs; *c = sn; }
}

/* ---- bounce ray (src/rt_cpu/rt_cpu.rs:61-76; basis sampling.hlsl:39-51) ---------------------- */
void orc_bounce_ray(const orc_scene* s, const orc_view* vw, const orc_ray* pr, const orc_hit* hit,
                    uint32_t px, uint32_t py, uint32_t frame_count, orc_ray* out) {
    memset(out, 0, sizeof(*out));
    if (!(hit->t < F32_MAX)) return;                                    /* rt_cpu.rs:61 */
    const uint8_t* rec = s->tris + (uint64_t)hit->prim * s->tri_stride;
    float v0[3], e1[3], e2[3];
    tri_load(rec, s->tri_stride, v0, e1, e2);
    float n[3];
    if (s->tri_stride == 64) { n[0] = load_f32(rec + 48); n[1] = load_f32(rec + 52); n[2] = load_f32(rec + 56); }
    else cross3(e1, e2, n);
    normalize3(n);                                                      /* RtTriangle::compute_normal */
    float nd[3] = { -pr->d[0], -pr->d[1], -pr->d[2] };
    float sgn = copysignf(1.0f, dot3(n, nd));                           /* f32::signum: +-1, signum(0)=+1 (rt_cpu.rs:65) */
    n[0] *= sgn; n[1] *= sgn; n[2] *= sgn;
    float org[3];
    for (int a = 0; a < 3; a++)                                         /* eye + d*t - d*0.01 (rt_cpu.rs:67) */
        org[a] = (vw->eye[a] + pr->d[a] * hit->t) - pr->d[a] * 0.01f;
    float u0 = orc_hash_noise(px, py, frame_count);                     /* rt_cpu.rs:70-73 */
    float u1 = orc_hash_noise(px, py, frame_count + 1024u);
    float rr = sqrtf(u0);                                               /* sampling.hlsl:30-36 */
    float sn, cs; orc_sincos_tau(u1, &sn, &cs);
    float l[3] = { rr * cs, rr * sn, sqrtf(fmaxf(0.0f, 1.0f - u0)) };
    float sign = n[2] >= 0.0f ? 1.0f : -1.0f;                           /* sampling.hlsl:40-50 */
    float a = -1.0f / (sign + n[2]);
    float b = n[0] * n[1] * a;
    float b1[3] = { 1.0f + sign * n[0] * n[0] * a, sign * b, -sign * n[0] };
    float b2[3] = { b, sign + n[1] * n[1] * a, -n[1] };
    float d[3];
    for (int k = 0; k < 3; k++)                                         /* Mat3::from_cols(b1,b2,n) * l */
        d[k] = (b1[k] * l[0] + b2[k] * l[1]) + n[k] * l[2];
    normalize3(d);
    out->o[0] = org[0]; out->o[1] = org[1]; out->o[2] = org[2]; out->tmin = 0.0f;
    out->d[0] = d[0]; out->d[1] = d[1]; out->d[2] = d[2]; out->tmax = F32_MAX;
}

/* the grey level of a result of kind `mode` (ORC_SHADE_*), gamma-encoded and truncated as rt_cpu.rs:104-106 */
uint8_t orc_shade(uint32_t mode, float t) {
    float col;
    if (mode == ORC_SHADE_PRIMARY) col = 1.0f / t;                      /* rt_cpu.rs:59 (1/inf = 0) */
    else if (mode == ORC_SHADE_OCCLUSION) col = t < F32_MAX ? 0.0f : 1.0f;   /* any-hit AO: visibility only */
    else col = t < F32_MAX ? t / (1.0f + t) : 1.0f;                      /* rt_cpu.rs:82-87 */
    float g = powf(col, 2.2f) * 255.0f;
    return (uint8_t)(g < 0.0f ? 0.0f : (g > 255.0f ? 255.0f : g));
}

/* ---- one frame of rt_cpu::start (src/rt_cpu/rt_cpu.rs:35-91, 102-107) ------------------------ */
int orc_render(const orc_scene* s, const orc_view* vw, uint32_t w, uint32_t h, uint32_t frame_count,
               uint32_t flags, orc_hit* primary, orc_hit* bounce, orc_ray* bounce_rays, uint8_t* rgba,
               orc_totals* ptot, orc_totals* btot, int nthreads) {
    int rc = 0;
    uint64_t pn = 0, pt = 0, pi = 0, ph = 0, bn = 0, bt = 0, bi = 0, bh = 0, br = 0;
    if (nthreads <= 0) nthreads = orc_max_threads();
#pragma omp parallel for schedule(dynamic, 1024) num_threads(nthreads) \
    reduction(+:pn,pt,pi,ph,bn,bt,bi,bh,br) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)w * h; i++) {
        uint32_t px = (uint32_t)(i % w), py = (uint32_t)(i / w);
        orc_ray ray; orc_primary_ray(vw, w, h, px, py, &ray);
        orc_hit hit; orc_count c;
        int e = trace_one(s, &ray, &hit, &c, NULL);
        if (e < rc) rc = e;
        pn += c.nodes; pt += c.tris; pi += c.insts; ph += hit.prim != ORC_INVALID_PRIM;
        if (primary) primary[i] = hit;
        uint32_t shade_mode = ORC_SHADE_PRIMARY; float shade_t = hit.t;  /* rt_cpu.rs:59 */
        orc_hit ao; ao.t = INFINITY; ao.prim = ORC_INVALID_PRIM;
        orc_ray aoray; memset(&aoray, 0, sizeof(aoray));
        if ((flags & ORC_RENDER_BOUNCE) && hit.t < F32_MAX) {
            orc_bounce_ray(s, vw, &ray, &hit, px, py, frame_count, &aoray);
            e = trace_one(s, &aoray, &ao, &c, NULL);
            if (e < rc) rc = e;
            br++; bn += c.nodes; bt += c.tris; bi += c.insts; bh += ao.prim != ORC_INVALID_PRIM;
            shade_mode = ORC_SHADE_BOUNCE; shade_t = ao.t;              /* rt_cpu.rs:82-87 */
        }
        if (bounce) bounce[i] = ao;
        if (bounce_rays) bounce_rays[i] = aoray;
        if (rgba && (flags & ORC_RENDER_RGBA)) {
            const uint8_t v8 = orc_shade(shade_mode, shade_t);
            rgba[4 * i + 0] = v8; rgba[4 * i + 1] = v8; rgba[4 * i + 2] = v8; rgba[4 * i + 3] = 255;
        }
    }
    if (ptot) { ptot->rays = (uint64_t)w * h; ptot->nodes = pn; ptot->tris = pt; ptot->insts = pi; ptot->hits = ph; }
    if (btot) { btot->rays = br; btot->nodes = bn; btot->tris = bt; btot->insts = bi; btot->hits = bh; }
    return rc;
}
