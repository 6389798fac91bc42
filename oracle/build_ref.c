/*
 * build_ref.c — serial reference of the device CWBVH builder (tray_racing_b200/csrc/build_gpu.cu).  TEST INFRASTRUCTURE ONLY.
 *
 * A second statement of tray_build::build_tlas from the rules written down in build_gpu.cu and DESIGN.md §4, as a plain
 * single-threaded program: no prefix sums, no shared-memory halo, no single-block PLOC tail, no atomics.  Those are the parts
 * of the device code it checks.  Every float operation is IEEE and separately rounded on both sides (-ffp-contract=off here,
 * -fmad=false there), and every step of the device build is deterministic by design, so the output bytes must be equal.  The
 * one exception is the SAH statistics: the device adds float warp sums with a double atomicAdd in no fixed order.
 */
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "tray_oracle.h"

/* ---- min / max -----------------------------------------------------------------------------------------------------------
 * The device's fminf / fmaxf order -0.0 below +0.0: fminf(+0, -0) = -0 and fmaxf(+0, -0) = +0 whichever argument comes first.
 * The scene bounds (ordered-int atomics) use the same total order.  So a box corner at zero is -0.0 when any primitive below
 * it has -0.0 there (min) and +0.0 when any has +0.0 (max).  A NaN argument loses to the other one. */
static inline float rmin(float a, float b) {
    if (isnan(b)) return a;
    if (isnan(a)) return b;
    return (a < b || (a == b && signbit(a))) ? a : b;
}
static inline float rmax(float a, float b) {
    if (isnan(b)) return a;
    if (isnan(a)) return b;
    return (a > b || (a == b && !signbit(a))) ? a : b;
}

typedef orc_bvh2_node Node;      /* leaf: left = -1, right = primitive; inner: left / right child node */

static inline float half_area3(const float lo[3], const float hi[3]) {
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
}
static inline float union_half_area(const float alo[3], const float ahi[3], const float blo[3], const float bhi[3]) {
    const float dx = rmax(ahi[0], bhi[0]) - rmin(alo[0], blo[0]);
    const float dy = rmax(ahi[1], bhi[1]) - rmin(alo[1], blo[1]);
    const float dz = rmax(ahi[2], bhi[2]) - rmin(alo[2], blo[2]);
    return dx * dy + dy * dz + dz * dx;
}

/* ---- Morton keys ---------------------------------------------------------------------------------------------------------- */
static uint64_t spread21(uint64_t v) {      /* bit k of v goes to bit 3k */
    uint64_t r = 0;
    for (int k = 0; k < 21; k++) r |= ((v >> k) & 1u) << (3 * k);
    return r;
}

typedef struct { uint64_t key; uint32_t idx; } KeyIdx;
static int cmp_key(const void* a, const void* b) {
    const KeyIdx* x = (const KeyIdx*)a; const KeyIdx* y = (const KeyIdx*)b;
    if (x->key != y->key) return x->key < y->key ? -1 : 1;
    return x->idx < y->idx ? -1 : (x->idx > y->idx);     /* equal keys keep input order: a stable sort */
}

/* ---- PLOC ------------------------------------------------------------------------------------------------------------------
 * One run over n boxes: leaves are nodes [0, n) in Morton order, inner nodes follow in creation order.  With `seg`, clusters
 * merge only inside their segment and the run ends with one root per segment, in segment order. */
typedef struct { Node* nd; uint32_t n_nodes; int* roots; uint32_t n_roots; uint32_t iters; } Ploc;

static int ploc_run(const float* blo, const float* bhi, uint32_t n, const uint32_t* seg, int r, Ploc* out) {
    memset(out, 0, sizeof *out);
    Node* nd = (Node*)calloc((size_t)2 * n, sizeof(Node));
    uint32_t* nseg = (uint32_t*)calloc((size_t)2 * n, sizeof(uint32_t));
    KeyIdx* ki = (KeyIdx*)malloc((size_t)n * sizeof(KeyIdx));
    int *cl = (int*)malloc((size_t)n * sizeof(int)), *cl2 = (int*)malloc((size_t)n * sizeof(int)), *nn = (int*)malloc((size_t)n * sizeof(int));
    if (!nd || !nseg || !ki || !cl || !cl2 || !nn) { free(nd); free(nseg); free(ki); free(cl); free(cl2); free(nn); return -2; }
    float s0[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, s1[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    for (uint32_t i = 0; i < n; i++)
        for (int a = 0; a < 3; a++) { s0[a] = rmin(s0[a], blo[3 * (size_t)i + a]); s1[a] = rmax(s1[a], bhi[3 * (size_t)i + a]); }
    for (uint32_t i = 0; i < n; i++) {
        uint64_t q[3];
        for (int a = 0; a < 3; a++) {
            const float c = 0.5f * (blo[3 * (size_t)i + a] + bhi[3 * (size_t)i + a]);
            const float ext = s1[a] - s0[a];
            float u = ext > 0.f ? (c - s0[a]) / ext : 0.f;
            u = rmin(rmax(u, 0.f), 1.f);
            q[a] = (uint64_t)rmin(u * 2097152.f, 2097151.f);
        }
        uint64_t key = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
        if (seg) key = ((uint64_t)seg[i] << 42) | (key >> 21);     /* the segment above a 42-bit Morton code */
        ki[i].key = key; ki[i].idx = i;
    }
    qsort(ki, n, sizeof(KeyIdx), cmp_key);
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t p = ki[i].idx;
        for (int a = 0; a < 3; a++) { nd[i].lo[a] = blo[3 * (size_t)p + a]; nd[i].hi[a] = bhi[3 * (size_t)p + a]; }
        nd[i].left = -1; nd[i].right = (int32_t)p; nd[i].count = 1; nd[i].parent = -1;
        nseg[i] = seg ? seg[p] : 0u;
        cl[i] = (int)i;
    }
    free(ki);
    uint32_t m = n, next = n, iters = 0;
    int rc = 0;
    while (m > 1) {
        /* nearest neighbour of every position among [i - r, i + r] of its segment: the smallest merged half-area, ties to
         * the lower position (strict <) */
        for (uint32_t i = 0; i < m; i++) {
            const Node* ci = &nd[cl[i]];
            float best = 3.4e38f; int best_j = -1;
            const int j0 = (int)i - r < 0 ? 0 : (int)i - r, j1 = (int)i + r > (int)m - 1 ? (int)m - 1 : (int)i + r;
            for (int j = j0; j <= j1; j++) {
                if (j == (int)i || nseg[cl[j]] != nseg[cl[i]]) continue;
                const Node* cj = &nd[cl[j]];
                const float a = union_half_area(ci->lo, ci->hi, cj->lo, cj->hi);
                if (a < best) { best = a; best_j = j; }
            }
            nn[i] = best_j;
        }
        /* mutual pairs merge; the lower position leads and creates the parent; new nodes are numbered in lead order and the
         * surviving clusters keep their order */
        uint32_t leads = 0, keeps = 0;
        for (uint32_t i = 0; i < m; i++) {
            const int j = nn[i];
            const int mutual = j >= 0 && nn[j] == (int)i;
            if (mutual && (int)i > j) continue;
            int c = cl[i];
            if (mutual) {
                const int l = cl[i], rg = cl[j];
                Node* d = &nd[next + leads++];
                for (int a = 0; a < 3; a++) { d->lo[a] = rmin(nd[l].lo[a], nd[rg].lo[a]); d->hi[a] = rmax(nd[l].hi[a], nd[rg].hi[a]); }
                d->left = l; d->right = rg; d->count = nd[l].count + nd[rg].count; d->parent = -1;
                nseg[d - nd] = nseg[l];
                c = (int)(d - nd);
            }
            cl2[keeps++] = c;
        }
        if (leads == 0) {
            if (!seg) rc = -3;                 /* a flat run that stalls is an error; a forest is done */
            break;
        }
        next += leads; m = keeps; iters++;
        int* t = cl; cl = cl2; cl2 = t;
    }
    free(cl2); free(nn); free(nseg);
    if (rc) { free(nd); free(cl); return rc; }
    out->nd = nd; out->n_nodes = next; out->roots = cl; out->n_roots = m; out->iters = iters;
    return 0;
}

/* ---- reinsertion ---------------------------------------------------------------------------------------------------------
 * Passes of (find, then `rounds` rounds of lock / check / cycle filter / apply, then one refit).  Between the rounds of a pass
 * the boxes are stale, exactly as on the device: the find of the next pass is the first to see the refit boxes. */
typedef struct { int* parent; float* gain; int* target; uint64_t* lock; uint8_t *win, *drop, *dirty; } Opt;

static inline int sibling_of(const Node* nd, const int* parent, int x) {
    const int p = parent[x];
    return nd[p].left == x ? nd[p].right : nd[p].left;
}

static void opt_find(const Node* nd, Opt* o, uint32_t v, uint32_t max_visits) {
    o->gain[v] = 0.f; o->target[v] = -1;
    const int p = o->parent[v];
    if (p < 0 || o->parent[p] < 0) return;                      /* the root and its children stay where they are */
    const float* Llo = nd[v].lo; const float* Lhi = nd[v].hi;
    const float aL = half_area3(Llo, Lhi);
    float best = 0.f; int best_x = -1;
    float d = half_area3(nd[p].lo, nd[p].hi);                   /* removing v deletes its parent */
    const int s = sibling_of(nd, o->parent, (int)v);
    float pblo[3], pbhi[3];                                     /* box of the path node once v is gone */
    memcpy(pblo, nd[s].lo, sizeof pblo); memcpy(pbhi, nd[s].hi, sizeof pbhi);
    int pivot = p, region = s, skip_root = 1;                   /* re-inserting next to the own sibling is the identity */
    uint32_t visits = 0;
    int stack_n[48]; float stack_c[48];
    for (;;) {
        /* branch and bound over `region`: cost of inserting at x = area(x U v) + the growth it induces on the way down */
        int sp = 0; stack_n[sp] = region; stack_c[sp] = 0.f; sp++;
        while (sp && visits < max_visits) {
            sp--; const int x = stack_n[sp]; const float cind = stack_c[sp];
            visits++;
            const float m = union_half_area(nd[x].lo, nd[x].hi, Llo, Lhi);
            if (!(skip_root && x == region)) {
                const float g = d - (cind + m);
                if (g > best) { best = g; best_x = x; }
            }
            if (nd[x].left >= 0) {
                const float cchild = cind + m - half_area3(nd[x].lo, nd[x].hi);
                if (d - (cchild + aL) > best && sp + 2 <= 48) {  /* a full stack drops the push */
                    stack_n[sp] = nd[x].right; stack_c[sp] = cchild; sp++;
                    stack_n[sp] = nd[x].left; stack_c[sp] = cchild; sp++;
                }
            }
        }
        skip_root = 0;
        /* climb one level: the new pivot's other child is the next region, and the pivot itself is a candidate */
        const int up = o->parent[pivot];
        if (up < 0 || visits >= max_visits) break;
        if (pivot != p) d += half_area3(nd[pivot].lo, nd[pivot].hi) - half_area3(pblo, pbhi);
        region = sibling_of(nd, o->parent, pivot);
        pivot = up;
        float nlo[3], nhi[3];
        for (int a = 0; a < 3; a++) { nlo[a] = rmin(pblo[a], nd[region].lo[a]); nhi[a] = rmax(pbhi[a], nd[region].hi[a]); }
        if (o->parent[pivot] >= 0) {                            /* insertion above a path node, never above the root */
            const float g = d - half_area3(nlo, nhi);
            if (g > best) { best = g; best_x = pivot; }
        }
        memcpy(pblo, nlo, sizeof pblo); memcpy(pbhi, nhi, sizeof pbhi);
    }
    if (best_x >= 0 && best > aL * 1e-6f) { o->gain[v] = best; o->target[v] = best_x; }
}

/* the six nodes a move rewires: v, its parent p, its sibling, its grandparent, the target x and x's parent (when it has one) */
static int opt_six(const Node* nd, const int* parent, int v, int x, int out[6]) {
    const int p = parent[v];
    int k = 0;
    out[k++] = v; out[k++] = p; out[k++] = sibling_of(nd, parent, v); out[k++] = parent[p]; out[k++] = x;
    if (parent[x] >= 0) out[k++] = parent[x];
    return k;
}
static inline uint64_t opt_key(const Opt* o, uint32_t v) {
    uint32_t g; memcpy(&g, &o->gain[v], 4);
    return ((uint64_t)g << 32) | v;                             /* a total order over the moves */
}

static void refit(Node* nd, uint32_t nn, const int* parent) {
    /* every inner node becomes the union of its children; reverse pre-order visits children before their parent */
    int* order = (int*)malloc((size_t)nn * sizeof(int));
    int* stack = (int*)malloc((size_t)nn * sizeof(int));
    uint32_t k = 0;
    for (uint32_t r = 0; r < nn; r++) {
        if (parent[r] >= 0) continue;
        int sp = 0; stack[sp++] = (int)r;
        while (sp) {
            const int x = stack[--sp];
            order[k++] = x;
            if (nd[x].left >= 0) { stack[sp++] = nd[x].left; stack[sp++] = nd[x].right; }
        }
    }
    while (k--) {
        Node* x = &nd[order[k]];
        if (x->left < 0) continue;
        const Node *l = &nd[x->left], *r = &nd[x->right];
        for (int a = 0; a < 3; a++) { x->lo[a] = rmin(l->lo[a], r->lo[a]); x->hi[a] = rmax(l->hi[a], r->hi[a]); }
        x->count = l->count + r->count;
    }
    free(order); free(stack);
}

static double inner_cost(const Node* nd, uint32_t first_inner, uint32_t nn) {
    double c = 0.0;
    for (uint32_t i = first_inner; i < nn; i++) c += (double)half_area3(nd[i].lo, nd[i].hi);
    return c;
}

static void set_parents(const Node* nd, uint32_t first_inner, uint32_t nn, int* parent) {
    for (uint32_t i = 0; i < nn; i++) parent[i] = -1;
    for (uint32_t i = first_inner; i < nn; i++) { parent[nd[i].left] = (int)i; parent[nd[i].right] = (int)i; }
}

static int optimize_run(Node* nd, uint32_t n_leaves, uint32_t nn, uint32_t passes, uint32_t max_visits, uint32_t rounds,
                        orc_build_stats* st) {
    if (passes == 0 || nn <= n_leaves + 2) return 0;           /* no statistics either, as on the device */
    Opt o;
    o.parent = (int*)malloc((size_t)nn * sizeof(int)); o.gain = (float*)malloc((size_t)nn * sizeof(float));
    o.target = (int*)malloc((size_t)nn * sizeof(int)); o.lock = (uint64_t*)malloc((size_t)nn * sizeof(uint64_t));
    o.win = (uint8_t*)malloc(nn); o.drop = (uint8_t*)malloc(nn); o.dirty = (uint8_t*)malloc(nn);
    if (!o.parent || !o.gain || !o.target || !o.lock || !o.win || !o.drop || !o.dirty) {
        free(o.parent); free(o.gain); free(o.target); free(o.lock); free(o.win); free(o.drop); free(o.dirty); return -2;
    }
    set_parents(nd, n_leaves, nn, o.parent);
    const double before = inner_cost(nd, n_leaves, nn);
    uint32_t moves = 0;
    int six[6];
    for (uint32_t pass = 0; pass < passes; pass++) {
        for (uint32_t v = 0; v < nn; v++) opt_find(nd, &o, v, max_visits);
        memset(o.dirty, 0, nn);
        for (uint32_t round = 0; round < rounds; round++) {
            memset(o.lock, 0, (size_t)nn * sizeof(uint64_t));
            /* lock: every move claims its six nodes; the largest key holds each.  From the second round on, a move found
             * before earlier rounds is dropped when one of its nodes was rewired, its target now lies in the subtree it
             * moves, or v has become a child of the root. */
            for (uint32_t v = 0; v < nn; v++) {
                if (o.target[v] < 0) continue;
                if (round > 0) {
                    int stale = 0;
                    const int k = opt_six(nd, o.parent, (int)v, o.target[v], six);
                    for (int q = 0; q < k; q++) if (o.dirty[six[q]]) stale = 1;
                    for (int a = o.target[v]; a >= 0 && !stale; a = o.parent[a]) if ((uint32_t)a == v) stale = 1;
                    if (stale || o.parent[o.parent[v]] < 0) { o.target[v] = -1; continue; }
                }
                const uint64_t key = opt_key(&o, v);
                const int k = opt_six(nd, o.parent, (int)v, o.target[v], six);
                for (int q = 0; q < k; q++) if (o.lock[six[q]] < key) o.lock[six[q]] = key;
            }
            /* a move that holds all six of its nodes wins */
            for (uint32_t v = 0; v < nn; v++) {
                o.win[v] = 0;
                if (o.target[v] < 0) continue;
                const uint64_t key = opt_key(&o, v);
                const int k = opt_six(nd, o.parent, (int)v, o.target[v], six);
                int mine = 1;
                for (int q = 0; q < k; q++) if (o.lock[six[q]] != key) mine = 0;
                o.win[v] = (uint8_t)mine;
            }
            /* cycle filter, computed for every winner on the tree before any move of the round is applied: a winner steps
             * back when the walk up from its target meets the moving node of a higher-keyed winner */
            for (uint32_t v = 0; v < nn; v++) {
                o.drop[v] = 0;
                if (o.target[v] < 0 || !o.win[v]) continue;
                const uint64_t key = opt_key(&o, v);
                for (int a = o.target[v]; a >= 0; a = o.parent[a])
                    if ((uint32_t)a != v && o.target[a] >= 0 && o.win[a] && opt_key(&o, (uint32_t)a) > key) { o.drop[v] = 1; break; }
            }
            /* apply.  The six-node sets of the winners are disjoint and a move reads and writes only its own six nodes, so
             * applying them one after another, in increasing v, gives what the device's concurrent rewiring gives. */
            for (uint32_t v = 0; v < nn; v++) {
                if (o.target[v] < 0 || !o.win[v] || o.drop[v]) continue;
                const int x = o.target[v];
                const int k = opt_six(nd, o.parent, (int)v, x, six);
                for (int q = 0; q < k; q++) o.dirty[six[q]] = 1;
                const int s = sibling_of(nd, o.parent, (int)v);
                const int p = o.parent[v], g = o.parent[p];
                if (nd[g].left == p) nd[g].left = s; else nd[g].right = s;     /* cut: s takes p's place under g */
                o.parent[s] = g;
                const int q = o.parent[x];                                      /* paste: p between x and its parent */
                if (nd[q].left == x) nd[q].left = p; else nd[q].right = p;
                o.parent[p] = q;
                nd[p].left = x; nd[p].right = (int)v;
                o.parent[x] = p;
                o.target[v] = -1;
                moves++;
            }
        }
        refit(nd, nn, o.parent);
    }
    if (st) {
        st->sah_before = before; st->sah_after = inner_cost(nd, n_leaves, nn);
        st->reinsert_moves = moves; st->reinsert_passes = passes;
    }
    free(o.parent); free(o.gain); free(o.target); free(o.lock); free(o.win); free(o.drop); free(o.dirty);
    return 0;
}

/* ---- collapse and encode ------------------------------------------------------------------------------------------------ */
typedef struct { int id[8]; int n; } Kids;

/* children of the wide node that replaces BVH2 subtree `root`: first open the largest-area subtree that has to stay inner
 * (more than max_leaf primitives), then spend free slots on the small subtree with the largest area x primitive count */
static void gather_kids(const Node* nd, int root, uint32_t max_leaf, Kids* k) {
    k->n = 0;
    if (nd[root].count <= max_leaf || nd[root].left < 0) k->id[k->n++] = root;
    else { k->id[k->n++] = nd[root].left; k->id[k->n++] = nd[root].right; }
    for (int phase = 0; phase < 2; phase++) {
        while (k->n < 8) {
            int best = -1; float best_a = -1.f;
            for (int i = 0; i < k->n; i++) {
                const Node* c = &nd[k->id[i]];
                if (c->left < 0) continue;
                const int big = c->count > max_leaf;
                if ((phase == 0) != big) continue;
                const float a = half_area3(c->lo, c->hi) * (phase == 0 ? 1.f : (float)c->count);
                if (a > best_a) { best_a = a; best = i; }
            }
            if (best < 0) break;
            const int c = k->id[best];
            k->id[best] = nd[c].left; k->id[k->n++] = nd[c].right;
        }
    }
}

/* smallest k with 255 * 2^k >= extent (extent at least 1e-20) */
static int quant_exponent(float extent) {
    extent = rmax(extent, 1e-20f);
    int k = (int)ceil(log2((double)extent / 255.0));
    while (ldexp(255.0, k) < (double)extent) k++;
    while (ldexp(255.0, k - 1) >= (double)extent) k--;
    return k;
}

static void encode_node(const Node* nd, int root, const Kids* k, uint32_t max_leaf, uint32_t child_base, uint32_t prim_base,
                        uint8_t* out80, uint32_t* prim_idx, int* inner_out, int* n_inner, int* force_exact) {
    const Node* n = &nd[root];
    /* slots by octant: greedy min-cost matching of (child centre - node centre) . (+-1, +-1, +-1), first strict minimum */
    float cost[8][8];
    for (int c = 0; c < k->n; c++) {
        const Node* ch = &nd[k->id[c]];
        float d[3];
        for (int a = 0; a < 3; a++) d[a] = 0.5f * (ch->lo[a] + ch->hi[a]) - 0.5f * (n->lo[a] + n->hi[a]);
        for (int s = 0; s < 8; s++)
            cost[c][s] = d[0] * ((s & 4) ? -1.f : 1.f) + d[1] * ((s & 2) ? -1.f : 1.f) + d[2] * ((s & 1) ? -1.f : 1.f);
    }
    int slot_child[8]; unsigned child_done = 0, slot_used = 0;
    for (int s = 0; s < 8; s++) slot_child[s] = -1;
    for (int r = 0; r < k->n; r++) {
        float bc = 3.4e38f; int bi = -1, bs = -1;
        for (int c = 0; c < k->n; c++) if (!((child_done >> c) & 1u))
            for (int s = 0; s < 8; s++) if (!((slot_used >> s) & 1u) && cost[c][s] < bc) { bc = cost[c][s]; bi = c; bs = s; }
        child_done |= 1u << bi; slot_used |= 1u << bs; slot_child[bs] = bi;
    }
    memset(out80, 0, 80);
    double scale[3];
    for (int a = 0; a < 3; a++) {
        memcpy(out80 + 4 * a, &n->lo[a], 4);
        const int e = quant_exponent(n->hi[a] - n->lo[a]);
        out80[12 + a] = (uint8_t)(e + 127);
        if (e + 127 >= 167) *force_exact = 1;
        scale[a] = ldexp(1.0, e);
    }
    memcpy(out80 + 16, &child_base, 4);
    memcpy(out80 + 20, &prim_base, 4);
    uint32_t tri_local = 0, imask = 0;
    *n_inner = 0;
    for (int s = 0; s < 8; s++) {
        if (slot_child[s] < 0) continue;
        const int c = k->id[slot_child[s]];
        for (int a = 0; a < 3; a++) {
            double ql = floor(((double)nd[c].lo[a] - (double)n->lo[a]) / scale[a]);
            double qh = ceil(((double)nd[c].hi[a] - (double)n->lo[a]) / scale[a]);
            ql = fmin(255.0, fmax(0.0, ql)); qh = fmin(255.0, fmax(0.0, qh));
            out80[32 + 16 * a + s] = (uint8_t)ql; out80[40 + 16 * a + s] = (uint8_t)qh;
        }
        const uint32_t cnt = nd[c].count;
        if (cnt > max_leaf) {
            imask |= 1u << s;
            out80[24 + s] = (uint8_t)((24 + s) | 0x20);
            inner_out[(*n_inner)++] = c;
        } else {
            out80[24 + s] = (uint8_t)((cnt == 1 ? 0x20 : cnt == 2 ? 0x60 : 0xE0) | tri_local);
            int stack[4]; int sp = 0; stack[sp++] = c;            /* the small subtree's primitives, left to right */
            while (sp) {
                const int x = stack[--sp];
                if (nd[x].left < 0) prim_idx[prim_base + tri_local++] = (uint32_t)nd[x].right;
                else { stack[sp++] = nd[x].right; stack[sp++] = nd[x].left; }
            }
        }
    }
    out80[15] = (uint8_t)imask;
}

/* Breadth-first, level by level: the wide nodes of a level are numbered in the order of their parents and, under one
 * parent, in slot order; primitives likewise.  forest: child_base_idx relative to the wide root of the node's tree. */
static int collapse_run(const Ploc* pl, uint32_t n_prims, int forest, uint32_t max_leaf, uint8_t* nodes, uint64_t node_cap,
                        uint32_t* prim_idx, uint32_t* n_nodes_out, uint32_t* levels_out, int* force_exact) {
    const uint32_t cap = n_prims + 1;
    int *items = (int*)malloc((size_t)cap * sizeof(int)), *items2 = (int*)malloc((size_t)cap * sizeof(int));
    uint32_t *root_of = (uint32_t*)malloc((size_t)cap * 4), *root_of2 = (uint32_t*)malloc((size_t)cap * 4);
    if (!items || !items2 || !root_of || !root_of2) { free(items); free(items2); free(root_of); free(root_of2); return -2; }
    for (uint32_t i = 0; i < pl->n_roots; i++) { items[i] = pl->roots[i]; root_of[i] = i; }
    uint32_t n_items = pl->n_roots, level_base = 0, prim_base = 0, levels = 0;
    int rc = 0;
    while (n_items) {
        if ((uint64_t)level_base + n_items > node_cap) { rc = -3; break; }
        const uint32_t next_base = level_base + n_items;
        uint32_t n_next = 0;
        for (uint32_t i = 0; i < n_items; i++) {
            Kids k; gather_kids(pl->nd, items[i], max_leaf, &k);
            const uint32_t my_root = forest ? root_of[i] : 0u;
            int inner[8], ni = 0;
            uint32_t nt = 0;
            for (int c = 0; c < k.n; c++) if (pl->nd[k.id[c]].count <= max_leaf) nt += pl->nd[k.id[c]].count;
            encode_node(pl->nd, items[i], &k, max_leaf, next_base + n_next - my_root, prim_base, nodes + (uint64_t)(level_base + i) * 80,
                        prim_idx, inner, &ni, force_exact);
            for (int c = 0; c < ni; c++) { items2[n_next] = inner[c]; root_of2[n_next] = my_root; n_next++; }
            prim_base += nt;
        }
        level_base = next_base; n_items = n_next; levels++;
        int* t = items; items = items2; items2 = t;
        uint32_t* u = root_of; root_of = root_of2; root_of2 = u;
    }
    free(items); free(items2); free(root_of); free(root_of2);
    if (rc) return rc;
    if (prim_base != n_prims) return -3;
    *n_nodes_out = level_base; *levels_out = levels;
    return 0;
}

/* ---- the whole build ---------------------------------------------------------------------------------------------------- */
int orc_build_ref(const float* tris9, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects,
                  const orc_build_params* prm, orc_build_result* out) {
    memset(out, 0, sizeof *out);
    if (!prm || (n_tris && !tris9)) return -1;
    if (n_tris == 0) return object_offsets ? -1 : 0;
    if (n_tris >= 0x7fffffffull || prm->max_leaf < 1 || prm->max_leaf > 3 || prm->radius > 64) return -1;
    const int tlas = object_offsets != NULL;
    if (tlas) {
        if (n_objects == 0 || n_objects >= (1u << 21) || object_offsets[0] != 0 || object_offsets[n_objects] != n_tris) return -1;
        for (uint32_t k = 0; k < n_objects; k++) if (object_offsets[k + 1] <= object_offsets[k]) return -1;
    }
    const uint32_t n = (uint32_t)n_tris;
    const int r = prm->radius == 0 ? 14 : (int)prm->radius;    /* 0 means obvhs' default search distance */
    float* blo = (float*)malloc((size_t)n * 12); float* bhi = (float*)malloc((size_t)n * 12);
    uint32_t* seg = tlas ? (uint32_t*)malloc((size_t)n * 4) : NULL;
    if (!blo || !bhi || (tlas && !seg)) { free(blo); free(bhi); free(seg); return -2; }
    for (uint32_t i = 0; i < n; i++) {
        const float* t = tris9 + 9 * (size_t)i;
        for (int a = 0; a < 3; a++) {
            blo[3 * (size_t)i + a] = rmin(t[a], rmin(t[3 + a], t[6 + a]));
            bhi[3 * (size_t)i + a] = rmax(t[a], rmax(t[3 + a], t[6 + a]));
        }
    }
    if (tlas) for (uint32_t k = 0; k < n_objects; k++) for (uint64_t i = object_offsets[k]; i < object_offsets[k + 1]; i++) seg[i] = k;
    Ploc pl, tp; memset(&tp, 0, sizeof tp);
    int rc = ploc_run(blo, bhi, n, seg, r, &pl);
    free(blo); free(bhi); free(seg);
    if (rc) return rc;
    uint8_t* nodes = NULL; uint32_t* pidx = NULL; uint32_t* blas = NULL; float *tlo = NULL, *thi = NULL;
    if (tlas && pl.n_roots != n_objects) { rc = -3; goto done; }
    rc = optimize_run(pl.nd, n, pl.n_nodes, prm->passes, prm->visits, prm->rounds, &out->stats);
    if (rc) goto done;
    const uint64_t blas_cap = (uint64_t)n + (tlas ? n_objects : 1), tlas_cap = tlas ? (uint64_t)n_objects + 1 : 0;
    nodes = (uint8_t*)calloc((size_t)(blas_cap + tlas_cap), 80);
    pidx = (uint32_t*)malloc((size_t)n * 4);
    if (!nodes || !pidx) { rc = -2; goto done; }
    uint32_t n_nodes = 0, levels = 0;
    int force_exact = 0;
    rc = collapse_run(&pl, n, tlas, prm->max_leaf, nodes, blas_cap, pidx, &n_nodes, &levels, &force_exact);
    if (rc) goto done;
    out->stats.ploc_iterations = pl.iters; out->stats.levels = levels;
    out->tlas_start = 0;
    if (tlas) {
        /* the TLAS: the same pipeline over the BLAS root boxes, flat; its primitives are object (= BLAS root node) numbers */
        tlo = (float*)malloc((size_t)n_objects * 12); thi = (float*)malloc((size_t)n_objects * 12);
        blas = (uint32_t*)malloc((size_t)n_objects * 4);
        if (!tlo || !thi || !blas) { rc = -2; goto done; }
        for (uint32_t k = 0; k < n_objects; k++) {
            memcpy(tlo + 3 * (size_t)k, pl.nd[pl.roots[k]].lo, 12); memcpy(thi + 3 * (size_t)k, pl.nd[pl.roots[k]].hi, 12);
        }
        rc = ploc_run(tlo, thi, n_objects, NULL, r, &tp);
        if (rc) goto done;
        rc = optimize_run(tp.nd, n_objects, tp.n_nodes, prm->passes, prm->visits, prm->rounds, NULL);
        if (rc) goto done;
        uint32_t tn = 0, tl = 0;
        rc = collapse_run(&tp, n_objects, 0, prm->max_leaf, nodes + (uint64_t)n_nodes * 80, tlas_cap, blas, &tn, &tl, &force_exact);
        if (rc) goto done;
        out->tlas_start = n_nodes;
        out->n_instances = n_objects;
        n_nodes += tn;
        out->stats.ploc_iterations += tp.iters; out->stats.levels += tl;
    }
    out->nodes = nodes; out->n_nodes = n_nodes; out->prim_indices = pidx; out->n_prims = n;
    out->blas_offsets = blas; out->force_exact = force_exact;
    out->stats.n_nodes = n_nodes;
    nodes = NULL; pidx = NULL; blas = NULL;
    /* the final BVH2 of the flat / forest run, with parents */
    out->bvh2 = pl.nd; out->n_bvh2 = pl.n_nodes; out->n_bvh2_leaves = n;
    {
        int* parent = (int*)malloc((size_t)pl.n_nodes * sizeof(int));
        if (parent) {
            set_parents(pl.nd, n, pl.n_nodes, parent);
            for (uint32_t i = 0; i < pl.n_nodes; i++) pl.nd[i].parent = parent[i];
            free(parent);
        }
    }
    pl.nd = NULL;
done:
    free(nodes); free(pidx); free(blas); free(tlo); free(thi);
    free(pl.nd); free(pl.roots); free(tp.nd); free(tp.roots);
    if (rc) orc_build_free(out);
    return rc;
}

void orc_build_free(orc_build_result* r) {
    if (!r) return;
    free(r->nodes); free(r->prim_indices); free(r->blas_offsets); free(r->bvh2);
    memset(r, 0, sizeof *r);
}
