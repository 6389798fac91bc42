/*
 * tlas_ref.c — the TLAS leg of the serial build reference over boxes the caller gives.  TEST INFRASTRUCTURE ONLY.
 *
 * tray_cuda_scene_refit_rebuild_tlas builds a TLAS over the exact boxes of the BLAS roots, in canonical instance order, with
 * the TLAS leg of the device builder.  This is the serial statement of that leg: oracle/build_ref.c's own PLOC, reinsertion and
 * collapse, compiled here from that file unchanged and run in the order orc_build_ref runs them for its TLAS.
 * tests/test_refit_tlas.py compiles it (with oracle/Makefile's flags) and checks it against orc_build_ref's TLAS first.
 */
#include "../oracle/build_ref.c"

typedef struct orc_tlas_result {
    uint8_t* nodes; uint32_t n_nodes;         /* 80-byte TLAS nodes, child indices relative to the TLAS root */
    uint32_t* perm;                           /* perm[j] = the box (instance) behind TLAS leaf entry j */
    int force_exact;                          /* some node exponent byte >= 167 */
} orc_tlas_result;

/* n boxes (box_lo / box_hi: n x 3 floats); params as orc_build_ref's.  Returns 0, -1 on bad arguments, -2 out of memory. */
int orc_build_ref_tlas(const float* box_lo, const float* box_hi, uint32_t n, const orc_build_params* prm, orc_tlas_result* out) {
    memset(out, 0, sizeof *out);
    if (!prm || !box_lo || !box_hi || n == 0 || n >= 0x7fffffffu || prm->max_leaf < 1 || prm->max_leaf > 3 || prm->radius > 64) return -1;
    const int r = prm->radius == 0 ? 14 : (int)prm->radius;
    Ploc tp;
    int rc = ploc_run(box_lo, box_hi, n, NULL, r, &tp);
    if (rc) return rc;
    uint8_t* nodes = (uint8_t*)calloc((size_t)n + 1, 80);
    uint32_t* perm = (uint32_t*)malloc((size_t)n * 4);
    uint32_t tn = 0, tl = 0;
    int force_exact = 0;
    if (!nodes || !perm) { rc = -2; goto done; }
    rc = optimize_run(tp.nd, n, tp.n_nodes, prm->passes, prm->visits, prm->rounds, NULL);
    if (rc) goto done;
    rc = collapse_run(&tp, n, 0, prm->max_leaf, nodes, (uint64_t)n + 1, perm, &tn, &tl, &force_exact);
    if (rc) goto done;
    out->nodes = nodes; out->n_nodes = tn; out->perm = perm; out->force_exact = force_exact;
    nodes = NULL; perm = NULL;
done:
    free(nodes); free(perm); free(tp.nd); free(tp.roots);
    return rc;
}

void orc_tlas_free(orc_tlas_result* r) {
    if (!r) return;
    free(r->nodes); free(r->perm);
    memset(r, 0, sizeof *r);
}
