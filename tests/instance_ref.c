/*
 * instance_ref.c — serial reference of the traversal of instanced scenes (tray_cuda_scene_set_instances).  TEST INFRASTRUCTURE ONLY.
 *
 * The oracle's two-level loop (oracle/tray_oracle.c trace_one_ex: the same node order, triangle order, stack and tie rule) with
 * the one thing the oracle does not have: a transform per TLAS leaf.  Entering leaf j, the ray becomes
 *     o'_i = ((W_i0 o_x + W_i1 o_y) + W_i2 o_z) + W_i3,   d'_i = (W_i0 d_x + W_i1 d_y) + W_i2 d_z
 * (W = world_to_object of the leaf's instance, d the caller's direction, tmin and the running tmax unchanged; zero components of d'
 * patched at the instance's scale, object_zero_patch), and back at the
 * TLAS it is the world ray again.  Node and triangle tests are the oracle's own exported ones (orc_node_intersect,
 * orc_intersect_tri), so everything the oracle decides about one ray against one node or triangle is decided here the same way.
 * The bounce ray of a frame takes the object-space normal to world space through the transpose of W before it is normalised.
 * tests/test_instances.py compiles it with oracle/Makefile's flags and links the oracle library.
 */
#include <math.h>
#include <string.h>

#include "../oracle/tray_oracle.h"

#define INVALID 0xFFFFFFFFu

static uint32_t firstbithigh(uint32_t x) { return 31u - (uint32_t)__builtin_clz(x); }

/* d' = W d with its zero components patched at the instance's scale (traverse.cuh object_zero_patch): component i becomes 2^-23
 * times 2^r, r = floor(log2 max_j |W_ij|), where |r| > 3, and 2^-23 itself where |r| <= 3 */
static void object_zero_patch(float d[3], const float* W) {
    for (int i = 0; i < 3; i++) {
        int e;
        frexpf(fmaxf(fmaxf(fabsf(W[4 * i]), fabsf(W[4 * i + 1])), fabsf(W[4 * i + 2])), &e);
        if (d[i] == 0.0f) d[i] = (e - 1 > 3 || e - 1 < -3) ? ldexpf(1.1920929e-7f, e - 1) : 1.1920929e-7f;
    }
}

static void xform_ray(const float* W, const orc_ray* in, orc_ray* out) {
    for (int i = 0; i < 3; i++) {
        const float* m = W + 4 * i;
        out->o[i] = ((m[0] * in->o[0] + m[1] * in->o[1]) + m[2] * in->o[2]) + m[3];
        out->d[i] = (m[0] * in->d[0] + m[1] * in->d[1]) + m[2] * in->d[2];
    }
    out->tmin = in->tmin; out->tmax = in->tmax;
    object_zero_patch(out->d, W);
}

/* One ray of scene `s` (two-level: blas_offsets[j] = the BLAS root of TLAS leaf j) with world_to_object w2o[12 j ..] and instance
 * leaf_inst[j] at leaf j; W == NULL: no transforms (the oracle's own traversal).  Returns 0, or -4 on a stack overflow at `cap`. */
static int trace_one(const orc_scene* s, const float* w2o, const uint32_t* leaf_inst, const orc_ray* ray, int any_hit, uint32_t cap,
                     orc_hit* out, uint32_t* inst_out, orc_count* cnt, uint32_t* peak) {
    uint32_t stack[ORC_STACK_MAX][2];
    uint32_t size = 0, max_size = 0;
    const int tlas = s->use_tlas;
    uint32_t tlas_stack_size = INVALID, bvh_offset = tlas ? s->tlas_start : 0u;
    uint32_t cur_x = 0, cur_y = 0x80000000u;
    float best_t = ray->tmax;
    uint32_t best_prim = INVALID, best_inst = INVALID, cur_inst = INVALID;
    uint32_t n_nodes = 0, n_tris = 0, n_insts = 0;
    int overflow = 0;
    orc_ray r = *ray;                                    /* the ray of the current tree: world, or the instance's object space */
    if (s->n_nodes == 0) cur_y = 0;
    for (;;) {
        uint32_t tri_x, tri_y;
        if (cur_y & 0xff000000u) {
            const uint32_t hits_imask = cur_y, off = firstbithigh(hits_imask), base = cur_x;
            cur_y &= ~(1u << off);
            if (cur_y & 0xff000000u) {
                if (size >= cap) { overflow = 1; break; }
                stack[size][0] = cur_x; stack[size][1] = cur_y; size++;
                if (size > max_size) max_size = size;
            }
            /* the octant row of the (zero-patched) direction: a zero component counts as positive */
            const uint32_t oct_inv = (r.d[0] < 0.0f ? 0u : 4u) | (r.d[1] < 0.0f ? 0u : 2u) | (r.d[2] < 0.0f ? 0u : 1u);
            const uint32_t slot = (off - 24u) ^ oct_inv;
            const uint32_t rel = (uint32_t)__builtin_popcount(hits_imask & ~(0xffffffffu << slot));
            const uint8_t* node = s->nodes + (uint64_t)(bvh_offset + base + rel) * 80u;
            n_nodes++;
            const uint32_t hitmask = orc_node_intersect(node, &r, best_t);
            uint32_t nx, ny;
            memcpy(&nx, node + 16, 4); memcpy(&ny, node + 20, 4);
            cur_x = nx; tri_x = ny;
            cur_y = (hitmask & 0xff000000u) | node[15];
            tri_y = hitmask & 0x00ffffffu;
        } else {
            tri_x = cur_x; tri_y = cur_y;
            cur_x = 0; cur_y = 0;
        }
        while (tri_y != 0) {
            const uint32_t local = firstbithigh(tri_y);
            tri_y &= ~(1u << local);
            const uint32_t global = tri_x + local;
            if (tlas && tlas_stack_size == INVALID) {
                if (tri_y != 0) {
                    if (size >= cap) { overflow = 1; break; }
                    stack[size][0] = tri_x; stack[size][1] = tri_y; size++;
                    if (size > max_size) max_size = size;
                }
                if (cur_y & 0xff000000u) {
                    if (size >= cap) { overflow = 1; break; }
                    stack[size][0] = cur_x; stack[size][1] = cur_y; size++;
                    if (size > max_size) max_size = size;
                }
                tlas_stack_size = size;
                bvh_offset = s->blas_offsets[global];
                if (w2o) { xform_ray(w2o + 12ull * global, ray, &r); cur_inst = leaf_inst[global]; }
                else cur_inst = global;
                n_insts++;
                cur_x = 0; cur_y = 0x80000000u;
                break;
            }
            n_tris++;
            orc_ray q = r; q.tmax = best_t;
            const float t = orc_intersect_tri(s, global, &q);
            if (t < best_t) { best_t = t; best_prim = global; best_inst = cur_inst; }
            if (any_hit && best_prim != INVALID) break;
        }
        if (overflow) break;
        if (any_hit && best_prim != INVALID) break;
        if ((cur_y & 0xff000000u) == 0) {
            if (size == 0) break;
            if (tlas && size == tlas_stack_size) {
                tlas_stack_size = INVALID;
                bvh_offset = s->tlas_start;
                r = *ray;
            }
            size--;
            cur_x = stack[size][0]; cur_y = stack[size][1];
        }
    }
    if (best_prim != INVALID) { out->t = best_t; out->prim = best_prim; }
    else { out->t = INFINITY; out->prim = INVALID; best_inst = INVALID; }
    if (inst_out) *inst_out = best_inst;
    if (cnt) { cnt->nodes = n_nodes; cnt->tris = n_tris; cnt->insts = n_insts; }
    if (peak) *peak = max_size;
    return overflow ? -4 : 0;
}

/* n rays; w2o / leaf_inst NULL: the untransformed two-level traversal.  `peak` (optional): stack entries each ray held at most. */
int inst_trace(const orc_scene* s, const float* w2o, const uint32_t* leaf_inst, const orc_ray* rays, uint64_t n, int any_hit, uint32_t cap,
               orc_hit* hits, uint32_t* inst, orc_count* counts, uint32_t* peak) {
    int rc = 0;
    if (cap == 0 || cap > ORC_STACK_MAX) return -1;
#pragma omp parallel for schedule(dynamic, 1024) reduction(min:rc)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        const int e = trace_one(s, w2o, leaf_inst, &rays[i], any_hit, cap, &hits[i], inst ? &inst[i] : NULL, counts ? &counts[i] : NULL,
                                peak ? &peak[i] : NULL);
        if (e < rc) rc = e;
    }
    return rc;
}

/* v times the power of two that puts its largest |component| in [1, 2); a zero vector stays zero (traverse.cuh scale_pow2) */
static void scale_pow2(float v[3]) {
    int e;
    frexpf(fmaxf(fmaxf(fabsf(v[0]), fabsf(v[1])), fabsf(v[2])), &e);
    for (int k = 0; k < 3; k++) v[k] = ldexpf(v[k], 1 - e);
}

/* The bounce ray of pixel (px, py) after primary ray `pr` hit `hit` in instance `k` (world_to_object w2o[12 k ..]; NULL: no
 * transform): oracle/tray_oracle.c orc_bounce_ray with the normal taken to world space, n'_i = (W_0i n_0 + W_1i n_1) + W_2i n_2,
 * brought to [1, 2) by a power of two before and after that product. */
static void bounce_one(const orc_scene* s, const orc_view* vw, const orc_ray* pr, const orc_hit* hit, const float* W, uint32_t px, uint32_t py,
                       uint32_t frame_count, orc_ray* out) {
    memset(out, 0, sizeof *out);
    if (!(hit->t < 3.402823466e+38f)) return;
    const uint8_t* rec = s->tris + (uint64_t)hit->prim * s->tri_stride;
    float v[12];
    memcpy(v, rec, s->tri_stride == 24 ? 24 : 48);
    float e1[3], e2[3], n[3];
    if (s->tri_stride == 24) {
        for (int k = 0; k < 3; k++) {
            uint32_t e; memcpy(&e, rec + 12 + 4 * k, 4);
            e2[k] = orc_half_to_float((uint16_t)(e & 0xffffu));
            e1[k] = -orc_half_to_float((uint16_t)(e >> 16));
        }
    } else {
        for (int k = 0; k < 3; k++) { e1[k] = v[4 + k]; e2[k] = v[8 + k]; }
    }
    if (s->tri_stride == 64) memcpy(n, rec + 48, 12);
    else { n[0] = e1[1] * e2[2] - e1[2] * e2[1]; n[1] = e1[2] * e2[0] - e1[0] * e2[2]; n[2] = e1[0] * e2[1] - e1[1] * e2[0]; }
    if (W) {
        float w[3];
        scale_pow2(n);
        for (int i = 0; i < 3; i++) w[i] = (W[i] * n[0] + W[4 + i] * n[1]) + W[8 + i] * n[2];
        n[0] = w[0]; n[1] = w[1]; n[2] = w[2];
        scale_pow2(n);
    }
    float len = sqrtf((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]);
    n[0] = n[0] / len; n[1] = n[1] / len; n[2] = n[2] / len;
    const float sgn = copysignf(1.0f, (n[0] * -pr->d[0] + n[1] * -pr->d[1]) + n[2] * -pr->d[2]);
    n[0] *= sgn; n[1] *= sgn; n[2] *= sgn;
    float org[3];
    for (int a = 0; a < 3; a++) org[a] = (vw->eye[a] + pr->d[a] * hit->t) - pr->d[a] * 0.01f;
    const float u0 = orc_hash_noise(px, py, frame_count), u1 = orc_hash_noise(px, py, frame_count + 1024u);
    const float rr = sqrtf(u0);
    float sn, cs; orc_sincos_tau(u1, &sn, &cs);
    const float l[3] = { rr * cs, rr * sn, sqrtf(fmaxf(0.0f, 1.0f - u0)) };
    const float sign = n[2] >= 0.0f ? 1.0f : -1.0f;
    const float a = -1.0f / (sign + n[2]);
    const float b = n[0] * n[1] * a;
    const float b1[3] = { 1.0f + sign * n[0] * n[0] * a, sign * b, -sign * n[0] };
    const float b2[3] = { b, sign + n[1] * n[1] * a, -n[1] };
    float d[3];
    for (int k = 0; k < 3; k++) d[k] = (b1[k] * l[0] + b2[k] * l[1]) + n[k] * l[2];
    len = sqrtf((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]);
    out->o[0] = org[0]; out->o[1] = org[1]; out->o[2] = org[2]; out->tmin = 0.0f;
    out->d[0] = d[0] / len; out->d[1] = d[1] / len; out->d[2] = d[2] / len; out->tmax = 3.402823466e+38f;
}

/* the bounce rays of a w x h frame (row-major) from its primary rays, hits and hit instances; w2o_by_inst NULL: no transforms */
void inst_bounce_rays(const orc_scene* s, const orc_view* vw, uint32_t w, uint32_t h, uint32_t frame_count, const orc_ray* primary,
                      const orc_hit* hits, const uint32_t* inst, const float* w2o_by_inst, orc_ray* out) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < (int64_t)w * h; i++) {
        const float* W = (w2o_by_inst && hits[i].prim != INVALID) ? w2o_by_inst + 12ull * inst[i] : NULL;
        bounce_one(s, vw, &primary[i], &hits[i], W, (uint32_t)(i % w), (uint32_t)(i / w), frame_count, &out[i]);
    }
}
