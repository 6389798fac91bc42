/*
 * hit_attr_ref.c — serial reference of the hit attributes (tray_cuda_hit_attributes).  TEST INFRASTRUCTURE ONLY.
 *
 * For one (ray, prim[, W]) it restates what the triangle test of oracle/tray_oracle.c computes: the record's v0, e1, e2 (tri_load,
 * stride 24 through orc_half_to_float), the zero-direction patch of prepare_ray (or the caller's direction under
 * ORC_VARIANT_ZERODIR_BOX_ONLY), Ng (the record's for stride 64, cross(e1, e2) otherwise), u and v.  On an instanced scene the
 * ray is first taken to object space as tests/instance_ref.c takes it, and Ng goes to world space through the transpose of W.
 * It also returns its own t = dot(Ng, v0 - o) / det, unrestricted by tmin / tmax, so that tests/test_hit_attributes.py can hold
 * it to the oracle's t bit for bit.
 * Compiled with oracle/Makefile's flags (-O3 -ffp-contract=off) and linked against the oracle library.
 */
#include <math.h>
#include <string.h>

#include "../oracle/tray_oracle.h"

#define INVALID 0xFFFFFFFFu
#define F32_EPSILON 1.1920929e-7f

static float dot3(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
static void cross3(const float a[3], const float b[3], float o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

/* out = {u, v, ng[3]}, *t_out = the test's t.  W: world_to_object (12 floats, row-major 3x4) or NULL. */
static void attr_one(const uint8_t* rec, uint32_t stride, const float* W, const orc_ray* ray, int zerodir_box_only, float out[5], float* t_out) {
    float o[3], d[3];
    for (int i = 0; i < 3; i++) {
        if (W) {
            const float* m = W + 4 * i;
            o[i] = ((m[0] * ray->o[0] + m[1] * ray->o[1]) + m[2] * ray->o[2]) + m[3];
            d[i] = (m[0] * ray->d[0] + m[1] * ray->d[1]) + m[2] * ray->d[2];
        } else {
            o[i] = ray->o[i]; d[i] = ray->d[i];
        }
        if (!zerodir_box_only && d[i] == 0.0f) d[i] = F32_EPSILON;
    }
    float v0[3], e1[3], e2[3], ng[3];
    memcpy(v0, rec, 12);
    if (stride == 24) {
        for (int k = 0; k < 3; k++) {
            uint32_t e; memcpy(&e, rec + 12 + 4 * k, 4);
            e2[k] = orc_half_to_float((uint16_t)(e & 0xffffu));
            e1[k] = -orc_half_to_float((uint16_t)(e >> 16));
        }
    } else {
        memcpy(e1, rec + 16, 12); memcpy(e2, rec + 32, 12);
    }
    if (stride == 64) memcpy(ng, rec + 48, 12);
    else cross3(e1, e2, ng);
    const float c[3] = { v0[0] - o[0], v0[1] - o[1], v0[2] - o[2] };
    float r[3]; cross3(d, c, r);
    const float inv_det = 1.0f / dot3(ng, d);
    out[0] = dot3(r, e2) * inv_det;
    out[1] = dot3(r, e1) * inv_det;
    *t_out = dot3(ng, c) * inv_det;
    if (W) {
        for (int i = 0; i < 3; i++) out[2 + i] = (W[i] * ng[0] + W[4 + i] * ng[1]) + W[8 + i] * ng[2];
    } else {
        out[2] = ng[0]; out[3] = ng[1]; out[4] = ng[2];
    }
}

/* n hits: attrs (5 floats each) and t; the miss record (all bytes 0xFF, t too) for prim == INVALID, prim >= n_tris and, with
 * w2o (world_to_object by instance, 12 floats each), inst[i] >= n_inst. */
void attr_ref(const uint8_t* tris, uint64_t n_tris, uint32_t stride, const float* w2o, uint32_t n_inst, const orc_ray* rays,
              const orc_hit* hits, const uint32_t* inst, uint64_t n, int zerodir_box_only, float* attrs, float* t) {
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t prim = hits[i].prim;
        if (prim == INVALID || prim >= n_tris || (w2o && inst[i] >= n_inst)) {
            memset(attrs + 5 * i, 0xff, 20);
            memset(t + i, 0xff, 4);
            continue;
        }
        attr_one(tris + (uint64_t)prim * stride, stride, w2o ? w2o + 12ull * inst[i] : NULL, &rays[i], zerodir_box_only, attrs + 5 * i, t + i);
    }
}
