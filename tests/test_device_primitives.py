"""The traversal's device primitives one by one, at their numeric edges.  tests/device_probe.cu puts batch entry points (one
thread per case) in front of the product's own tray:: functions in traverse.cuh — prepare_ray, node_test, node_test_fast,
tri_test, primary_dir, bounce_ray, uhash, hash_noise, sincos_tau, shade, child_order_fill — and these tests aim chosen inputs
at them: hand-encoded 80-byte nodes and triangle records, special float values, exact boundaries.  Each device result is held
to the oracle's function of the same name (bit for bit unless a test says otherwise), to a numpy restatement, or to a float64
evaluation of the same formula.

Set TRAY_PROBE_LIB to test another build of the probe (a patched traverse.cuh: `make -C tray_racing_b200/csrc probe
PROBE_INC=<dir> PROBE_LIB=<file>`); by default the module builds it with `make probe`."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import oracle_binding as ob
from tray_racing_b200 import host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tray_racing_b200", "csrc")
F32_MAX = np.float32(3.402823466e+38)
INF = np.float32(np.inf)
EPS = np.float32(1.1920929e-7)                  # the zero-direction patch (query.hlsl:334)
SHADE_PRIMARY, SHADE_BOUNCE, SHADE_OCCLUSION = 1, 2, 3
VARIANT_BOX_DIVIDE, VARIANT_ZERODIR_BOX_ONLY, VARIANT_BOX_TMIN_RAY = 1, 8, 4


def f32(x):
    return np.float32(x)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def from_bits(u):
    return np.asarray(u, dtype=np.uint32).view(np.float32)


def rays_of(o, d, tmin=0.0, tmax=F32_MAX):
    o, d = np.atleast_2d(np.asarray(o, np.float32)), np.atleast_2d(np.asarray(d, np.float32))
    n = max(len(o), len(d))
    r = np.zeros(n, ob.RAY_DTYPE)
    r["o"], r["d"], r["tmin"], r["tmax"] = o, d, tmin, tmax
    return r


# ---- the probe library ------------------------------------------------------------------------------------------------------
class Probe:
    def __init__(self, path):
        L = C.CDLL(path)
        vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int
        sig = {"probe_prepare_ray": [vp, u32, u32, vp], "probe_node_test": [vp, vp, u32, u32, u32, vp],
               "probe_tri_test": [vp, u32, vp, u32, u32, u32, vp], "probe_primary_dir": [vp, u32, u32, vp, vp, u32, vp],
               "probe_bounce_ray": [u32, vp, u32, vp, vp, vp, vp, vp, vp, vp, u32, vp],
               "probe_bounce_ray_inst": [u32, vp, u32, vp, vp, vp, vp, vp, vp, vp, vp, u32, vp], "probe_uhash": [vp, vp, u32, vp],
               "probe_hash_noise": [vp, vp, vp, u32, vp], "probe_sincos_tau": [vp, u32, vp, vp], "probe_shade": [u32, vp, u32, vp],
               "probe_child_order": [vp]}
        for name, args in sig.items():
            getattr(L, name).argtypes, getattr(L, name).restype = args, i32
        L.probe_lut_row.restype = u32
        self.L = L

    def _call(self, name, *args):
        rc = getattr(self.L, name)(*[a.ctypes.data if isinstance(a, np.ndarray) else a for a in args])
        assert rc == 0, f"{name}: CUDA error {rc}"

    def prepare_ray(self, rays, variant=0):
        rays = np.ascontiguousarray(rays, ob.RAY_DTYPE)
        out = np.zeros((len(rays), 12), np.uint32)
        self._call("probe_prepare_ray", rays, len(rays), variant, out)
        f = out[:, :10].copy().view(np.float32)
        return dict(d=f[:, 0:3], inv=f[:, 3:6], dt=f[:, 6:9], box_tmin=f[:, 9], oct_inv4=out[:, 10], wide=out[:, 11].astype(bool))

    def node_test(self, nodes, rays, which, variant=0):
        nodes = np.ascontiguousarray(nodes, np.uint8).reshape(-1, 80)
        rays = np.ascontiguousarray(rays, ob.RAY_DTYPE)
        out = np.zeros(len(rays), np.uint32)
        self._call("probe_node_test", nodes, rays, len(rays), which, variant, out)
        return out

    def tri_test(self, records, stride, rays, variant=0, variant_dir=False):
        rec = np.ascontiguousarray(records, np.uint8).reshape(-1)
        rays = np.ascontiguousarray(rays, ob.RAY_DTYPE)
        assert rec.size == stride * len(rays)
        out = np.zeros(len(rays), np.float32)
        self._call("probe_tri_test", rec, stride, rays, len(rays), variant, int(variant_dir), out)
        return out

    def primary_dir(self, view, w, h, px, py):
        px, py = np.ascontiguousarray(px, np.uint32), np.ascontiguousarray(py, np.uint32)
        out = np.zeros((len(px), 3), np.float32)
        self._call("probe_primary_dir", C.addressof(view), w, h, px, py, len(px), out)
        return out

    def bounce_ray(self, stride, records, view, px, py, pd, t, prim, frame_count, w2o=None):
        """w2o: None, or one world_to_object (3, 4) per case: the instanced form, with case i's InstanceRecord"""
        rec = np.ascontiguousarray(records, np.uint8).reshape(-1)
        a = [np.ascontiguousarray(x, dt) for x, dt in ((px, np.uint32), (py, np.uint32), (pd, np.float32), (t, np.float32),
                                                       (prim, np.uint32), (frame_count, np.uint32))]
        out = np.zeros((len(a[0]), 6), np.float32)
        if w2o is None:
            self._call("probe_bounce_ray", stride, rec, rec.size // stride, C.addressof(view), *a, len(a[0]), out)
        else:
            inst = np.zeros((len(a[0]), 16), np.float32)
            inst[:, :12] = np.asarray(w2o, np.float32).reshape(-1, 12)
            self._call("probe_bounce_ray_inst", stride, rec, rec.size // stride, C.addressof(view), *a, inst, len(a[0]), out)
        return out

    def uhash(self, a, b):
        a, b = np.ascontiguousarray(a, np.uint32), np.ascontiguousarray(b, np.uint32)
        out = np.zeros(len(a), np.uint32)
        self._call("probe_uhash", a, b, len(a), out)
        return out

    def hash_noise(self, x, y, f):
        x, y, f = (np.ascontiguousarray(v, np.uint32) for v in (x, y, f))
        out = np.zeros(len(x), np.float32)
        self._call("probe_hash_noise", x, y, f, len(x), out)
        return out

    def sincos_tau(self, u):
        u = np.ascontiguousarray(u, np.float32)
        s, c = np.zeros_like(u), np.zeros_like(u)
        self._call("probe_sincos_tau", u, len(u), s, c)
        return s, c

    def shade(self, mode, t):
        t = np.ascontiguousarray(t, np.float32)
        out = np.zeros(len(t), np.uint8)
        self._call("probe_shade", mode, t, len(t), out)
        return out

    def child_order(self):
        row = self.L.probe_lut_row()
        out = np.zeros(8 * row, np.uint8)
        self._call("probe_child_order", out)
        return out.reshape(8, row)[:, :256]


@pytest.fixture(scope="module")
def probe():
    path = os.environ.get("TRAY_PROBE_LIB")
    if not path:
        r = subprocess.run(["make", "-s", "-C", CSRC, "probe"], capture_output=True, text=True)
        assert r.returncode == 0, f"make probe failed:\n{r.stdout}\n{r.stderr}"
        path = os.path.join(ROOT, "tray_racing_b200", "libtray_probe.so")
    return Probe(path)


def _oracle_lib():
    L = ob.lib()
    L.orc_shade.restype, L.orc_shade.argtypes = C.c_uint8, [C.c_uint32, C.c_float]
    L.orc_bounce_ray.restype = None
    L.orc_bounce_ray.argtypes = [C.POINTER(ob.OrcScene), C.POINTER(ob.OrcView), C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                 C.c_uint32, C.c_void_p]
    L.orc_primary_ray.restype = None
    return L


# ---- node test --------------------------------------------------------------------------------------------------------------
EXP_BYTES = (0, 1, 100, 127, 166, 167, 200, 254, 255)
CHILD_BYTES = (0, 1, 127, 254, 255)
SUB = np.float32(1e-40)                                      # subnormal
D_SPECIAL = [1.0, -1.0, 0.5, -3.0, 0.0, -0.0, 1e-40, -1e-40, np.inf, -np.inf, np.nan,
             2.0 ** -64, -(2.0 ** -64), float(np.nextafter(f32(2.0 ** -64), f32(1))), float(np.nextafter(f32(2.0 ** -64), f32(0))),
             -float(np.nextafter(f32(2.0 ** -64), f32(1))), 2.0 ** -66, 2.0 ** -63, 1e-30]
P_SPECIAL = [0.0, -0.0, 1e-40, -1e-40, 1e30, -1e30, 1.0, -3.0, 100.0]
O_SPECIAL = [0.0, -0.0, 1e-40, 1.0, -1.0, 50.0, -1e30, 1e30, 3.0]
TMAX_SPECIAL = [0.0, 1e-4, float(F32_MAX), np.inf, 7.0]


def node_bytes(p, exps, metas, lo, hi):
    """one 80-byte node: p[3] f32, exponent bytes, meta[8], lo / hi [3][8] child bytes (imask and bases stay zero: the box test
    does not read them)"""
    n = np.zeros(80, np.uint8)
    n[0:12] = np.asarray(p, np.float32).view(np.uint8)
    n[12:15] = exps
    n[24:32] = metas
    for a in range(3):
        n[32 + 16 * a:40 + 16 * a] = lo[a]
        n[40 + 16 * a:48 + 16 * a] = hi[a]
    return n


def node_corpus():
    """(nodes[n, 80], rays[n]): special values on every axis, every meta byte, child bytes incl. lo > hi, exact boundaries and
    the cases on either side of the fused form's limit"""
    rng = np.random.default_rng(1234)
    nodes, rays = [], []
    metas_all = np.arange(256, dtype=np.uint8)

    def add(n, o, d, tmin=0.0, tmax=F32_MAX):
        nodes.append(n); rays.append(rays_of(o, d, tmin, tmax)[0])

    # 1. special values, combined: every exponent byte on every axis, every direction / origin / p / tmax kind
    k = 0
    for ax in range(3):
        for e in EXP_BYTES:
            for rep in range(60):
                exps = [127, 127, 127]
                exps[ax] = e
                if rep % 3 == 0:
                    exps[(ax + 1) % 3] = int(rng.choice(EXP_BYTES))
                metas = metas_all[(8 * k + np.arange(8)) % 256]
                k += 1
                lo = rng.choice(CHILD_BYTES, size=(3, 8)).astype(np.uint8)
                hi = rng.choice(CHILD_BYTES, size=(3, 8)).astype(np.uint8)
                p = rng.choice(P_SPECIAL, 3)
                o = rng.choice(O_SPECIAL, 3)
                d = rng.choice(D_SPECIAL, 3)
                tmax = rng.choice(TMAX_SPECIAL)
                add(node_bytes(p, exps, metas, lo, hi), o, d, 0.0, tmax)
    # 2. metas sweep on a plain hitting node: every byte 0..255 in every slot position, all children hit
    for k in range(32):
        metas = metas_all[(8 * k + np.arange(8)) % 256]
        add(node_bytes([0, 0, 0], [127] * 3, metas, np.zeros((3, 8), np.uint8), np.full((3, 8), 10, np.uint8)), [-1, -2, -3], [1, 1, 1])
        add(node_bytes([0, 0, 0], [127] * 3, metas, np.zeros((3, 8), np.uint8), np.full((3, 8), 10, np.uint8)), [20, 20, 20], [-1, -0.5, -2])
    # 3. exact boundaries, d = 1 (1/d = 1), scale 1, p = 0: t = q - o on each axis, exactly
    plain_meta = np.array([0x20 | s for s in range(8)], np.uint8)     # leaves, one triangle each at offset = slot
    for q in (0, 1, 5, 200, 255):
        for lo_b, hi_b in ((q, q), (q, min(q + 3, 255)), (min(q + 3, 255), q)):
            lo, hi = np.full((3, 8), lo_b, np.uint8), np.full((3, 8), hi_b, np.uint8)
            nd = node_bytes([0, 0, 0], [127] * 3, plain_meta, lo, hi)
            add(nd, [0, 0, 0], [1, 1, 1])                                       # tnear == tfar when lo == hi
            add(nd, [-1e-4, -1e-4, -1e-4], [1, 1, 1])                           # tnear == 1e-4 (q = 0)
            add(nd, [f32(q) - f32(1e-4)] * 3, [1, 1, 1])                        # tnear == 1e-4 exactly when representable
            tf = f32(hi_b) - f32(-1)
            for tm in (tf, np.nextafter(tf, f32(0)), np.nextafter(tf, INF)):     # tfar == tmax, one ulp either side
                add(nd, [-1, -1, -1], [1, 1, 1], 0.0, tm)
            for tm in (0.0, 1e-4, float(np.nextafter(f32(1e-4), f32(0)))):
                add(nd, [0, 0, 0], [1, 1, 1], 0.0, tm)
        # one axis only at the boundary, the others wide open
        lo, hi = np.zeros((3, 8), np.uint8), np.full((3, 8), 255, np.uint8)
        lo[1], hi[1] = q, q
        add(node_bytes([0, 0, 0], [127] * 3, plain_meta, lo, hi), [-1, 0, -1], [1, 1, 1])
    # 4. the fused form's limit: 2^23 * A overflows once A = scale * |1/d| reaches 2^105 (x axis: y and z convert with I2F).
    #    x: lo 0, hi 1, origin on p (b = 0) -> [0, A]; y, z: [1, 10].  The exact test hits every child; the fused form misses
    #    once A >= 2^105.  Exponent byte e, direction 2^-j: A = 2^(e - 127 + j).
    lo = np.array([[0] * 8, [1] * 8, [1] * 8], np.uint8)
    hi = np.array([[1] * 8, [10] * 8, [10] * 8], np.uint8)
    for e, j in ((166, 63), (166, 64), (166, 65), (166, 66), (166, 67), (169, 63), (169, 62), (170, 63), (167, 63), (160, 66),
                 (164, 66), (165, 66), (166, 66), (100, 66), (160, 64)):
        for sgn in (1, -1):
            nd = node_bytes([0, 0, 0], [e, 127, 127], plain_meta, lo, hi)
            dx = sgn * 2.0 ** -j
            for dxx in (dx, float(np.nextafter(f32(dx), f32(0))), float(np.nextafter(f32(dx), f32(sgn)))):
                # with a negative dx the near plane is hi: origin at p + scale so that [0, A] again
                o0 = 0.0 if sgn > 0 else float(f32(2.0 ** (e - 127)))
                add(nd, [o0, 0, 0], [dxx, 1, 1])
    return np.stack(nodes), np.array(rays, ob.RAY_DTYPE)


def decision_node(n):
    """the same boxes with child c a one-triangle leaf at offset c: the oracle's mask of it is the per-child hit decision"""
    m = n.copy()
    m[24:32] = [0x20 | c for c in range(8)]
    return m


def slot_space_mask(hit_byte, metas):
    """the device's slot-space mask (traverse.cuh node_test): child_bits << (meta & 31) for every hit child, no octant XOR"""
    out = 0
    for c in range(8):
        if (hit_byte >> c) & 1:
            m = int(metas[c])
            out |= (((m >> 5) & 7) << (m & 31)) & 0xFFFFFFFF
    return out


def oracle_mask_model(hit_byte, metas, oct_inv):
    """the oracle's mask (query.hlsl:251-297): inner children (meta bits 3 and 4) shift by (meta ^ oct_inv) & 31"""
    out = 0
    for c in range(8):
        if (hit_byte >> c) & 1:
            m = int(metas[c])
            inner = ((m & (m << 1)) & 0x10) != 0
            out |= (((m >> 5) & 7) << ((m ^ (oct_inv if inner else 0)) & 31)) & 0xFFFFFFFF
    return out


def oracle_decisions(nodes, rays, variant=0):
    ob.set_variant(variant)
    try:
        return np.array([ob.node_intersect(decision_node(n), r, r["tmax"]) for n, r in zip(nodes, rays)], np.uint32)
    finally:
        ob.set_variant(0)


@pytest.mark.gpu
def test_node_test_equals_oracle(probe):
    nodes, rays = node_corpus()
    dec = oracle_decisions(nodes, rays)
    assert (dec & ~np.uint32(0xFF)).max() == 0
    assert 0 < np.count_nonzero(dec) < len(dec)
    oct_inv = probe.prepare_ray(rays)["oct_inv4"] & 7
    # the oracle's own mask with the real metas is its per-child decisions under query.hlsl's bit rule
    for i in range(0, len(nodes), 7):
        assert ob.node_intersect(nodes[i], rays[i], rays[i]["tmax"]) == oracle_mask_model(dec[i], nodes[i][24:32], int(oct_inv[i]))
    want = np.array([slot_space_mask(h, n[24:32]) for h, n in zip(dec, nodes)], np.uint32)
    got_dec = probe.node_test(np.stack([decision_node(n) for n in nodes]), rays, 0)
    bad = np.nonzero(got_dec != dec)[0]
    assert bad.size == 0, f"{bad.size} of {len(dec)} per-child decisions differ, first {bad[:5]}"
    got = probe.node_test(nodes, rays, 0)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, f"{bad.size} of {len(want)} masks differ, first {bad[:5]}"


@pytest.mark.gpu
@pytest.mark.parametrize("variant", range(8))
def test_node_test_mode1_equals_oracle_under_variants(probe, variant):
    """node_test as MODE 1 calls it (box_tmin and the divide form per TRAY_VARIANT_*), against the oracle under the same
    switches; the tie rule does not reach the box test, so its bit is reused to switch the zero-direction reading"""
    nodes, rays = node_corpus()
    rng = np.random.default_rng(variant)
    rays = rays.copy()
    sel = rng.random(len(rays)) < 0.3
    rays["tmin"][sel] = rng.choice(np.float32([0.0, 1e-4, 0.5, 3.0, 1e-45, -1.0]), size=sel.sum())
    v = variant | (VARIANT_ZERODIR_BOX_ONLY if variant & 2 else 0)
    want = oracle_decisions(nodes, rays, v)
    got = probe.node_test(np.stack([decision_node(n) for n in nodes]), rays, 1, v)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, f"variant {v}: {bad.size} of {len(want)} decisions differ, first {bad[:5]}"


@pytest.mark.gpu
def test_node_test_fast_limit_and_guards(probe):
    """node_test_fast == node_test wherever 2^23 * A is finite (|A_x| < 2^105), it differs past that line, and every case the
    two guards (RayConst::wide, node_needs_exact) send to the fast form lies inside it — with cases two and three bits past
    each guard, so that moving either guard out by three bits shows up as a wrong mask.  The per-child decisions are compared
    on decision nodes; the fused form accumulates the hit children's contributions with an ADD (the predicated IMAD), which
    equals node_test's OR when they are disjoint, as every CWBVH encoding makes them — checked as a sum on the real metas."""
    nodes, rays = node_corpus()
    pr = probe.prepare_ray(rays)
    dnodes = np.stack([decision_node(n) for n in nodes])
    exact = probe.node_test(dnodes, rays, 0)
    fast = probe.node_test(dnodes, rays, 2)
    chosen = probe.node_test(dnodes, rays, 3)
    scale_x = from_bits(nodes[:, 12].astype(np.uint32) << 23)
    with np.errstate(all="ignore"):
        a_x = np.abs(scale_x * pr["inv"][:, 0])
    inside = (a_x < 2.0 ** 105) | np.isnan(a_x)
    bad = np.nonzero(inside & (fast != exact))[0]
    assert bad.size == 0, f"fused form differs inside its limit: {bad[:5]}"
    past = ~inside & (fast != exact)
    assert past.sum() >= 4, "the corpus must hold cases past 2^105 where the fused form goes wrong"
    assert np.isfinite(a_x[past]).any() and (a_x[past][np.isfinite(a_x[past])] < 2.0 ** 107).any()
    fast_path = ~pr["wide"] & (nodes[:, 12:15].max(axis=1) < 167)
    assert fast_path.sum() > 100
    assert inside[fast_path].all(), "a guard sends a case past the fused form's limit"
    assert a_x[fast_path & np.isfinite(a_x)].max() < 2.0 ** 103
    bad = np.nonzero(chosen != exact)[0]
    assert bad.size == 0, f"the kernel's choice of node test changes the mask: {bad[:5]}"
    # the accumulation on the real metas: a sum of the hit children's contributions (an OR where they are disjoint)
    fast_real, exact_real = probe.node_test(nodes, rays, 2), probe.node_test(nodes, rays, 0)
    total = np.array([sum((((int(m) >> 5) & 7) << (int(m) & 31)) & 0xFFFFFFFF for c, m in enumerate(n[24:32]) if (h >> c) & 1)
                      & 0xFFFFFFFF for h, n in zip(exact, nodes)], np.uint32)
    assert (fast_real[inside] == total[inside]).all()
    overlap = fast_real != exact_real
    assert (overlap[inside] == (total != exact_real)[inside]).all() and overlap[inside].any()
    # the cases that show a three-bit move of a guard: A = 2^105 with byte 166 and |1/d| = 2^66, and byte 169 with |1/d| = 2^63
    for e, inv in ((166, 2.0 ** 66), (169, 2.0 ** 63)):
        sel = (nodes[:, 12] == e) & (np.abs(pr["inv"][:, 0]) == inv) & (fast != exact)
        assert sel.any(), f"no wrong-mask case at byte {e}, |1/d| = 2^{int(math.log2(inv))}"


@pytest.mark.gpu
def test_prepare_ray(probe):
    vals = [1.0, -1.0, 0.0, -0.0, 1e-40, -1e-40, np.inf, -np.inf, np.nan, 2.0 ** -64, float(np.nextafter(f32(2.0 ** -64), f32(1))),
            float(np.nextafter(f32(2.0 ** -64), f32(0))), -(2.0 ** -64), 3.0, 1e30]
    d = np.array([(a, b, c) for a in vals for b in vals[:6] for c in vals[::3]], np.float32)
    rays = rays_of(np.zeros_like(d), d, tmin=0.25)
    for variant in (0, VARIANT_ZERODIR_BOX_ONLY | VARIANT_BOX_TMIN_RAY):
        g = probe.prepare_ray(rays, variant)
        patched = np.where(d == 0, EPS, d)
        assert (bits(g["d"]) == bits(patched)).all()
        assert (bits(g["dt"]) == bits(d if variant else patched)).all()
        with np.errstate(all="ignore"):
            inv = np.float32(1) / patched
        same = (bits(g["inv"]) == bits(inv)) | (np.isnan(g["inv"]) & np.isnan(inv))     # CUDA's NaN is canonical: no payload
        assert same.all(), f"1/d differs for d = {d[~same.all(axis=1)][:4]}"
        oct4 = np.where(patched[:, 0] < 0, 0, 0x04040404) | np.where(patched[:, 1] < 0, 0, 0x02020202) | np.where(patched[:, 2] < 0, 0, 0x01010101)
        assert (g["oct_inv4"] == oct4.astype(np.uint32)).all()
        m = np.fmax(np.fmax(np.abs(inv[:, 0]), np.abs(inv[:, 1])), np.abs(inv[:, 2]))      # fmaxf: a NaN loses to a number
        with np.errstate(invalid="ignore"):
            wide = ~(m < np.float32(2.0 ** 64))
        assert (g["wide"] == wide).all()
        assert (g["box_tmin"] == (np.float32(0.25) if variant else np.float32(1e-4))).all()


@pytest.mark.gpu
def test_child_order_table(probe):
    lut = probe.child_order()
    for oi in range(8):
        for t in range(1, 256):
            best = max((j for j in range(8) if (t >> j) & 1), key=lambda j: j ^ oi)
            assert lut[oi, t] == best, (oi, t)


# ---- triangle test ----------------------------------------------------------------------------------------------------------
def overflow_triangle(a=62, b=66):
    """a triangle in z = 0 with edges 2^a and an origin 2^b away in that plane, aimed along z: dot(r, e2) adds +2^(a+b) and
    -2^(a+b), which overflow with opposite signs when a + b >= 128, so u is inf - inf = NaN while ng and det stay finite and
    t = dot(ng, c) * inv_det = -0"""
    s, o = 2.0 ** a, 2.0 ** b
    tri = np.array([[0, 0, 0], [s, 0, 0], [s, s, 0]], np.float32)       # e1 = v0 - v1 = (-s, 0, 0), e2 = v2 - v0 = (s, s, 0)
    ray = rays_of([o, o, 0], [0, 0, 1], 0.0, F32_MAX)
    return tri, ray


def tri_numpy(rec48, rays):
    """u, v, w and t of the triangle test in numpy float32, every operation rounded as in the oracle and the kernel"""
    r = rec48.view(np.float32).reshape(-1, 12)
    v0, e1, e2 = r[:, 0:3], r[:, 4:7], r[:, 8:11]
    d = np.where(rays["d"] == 0, EPS, rays["d"]).astype(np.float32)
    o = rays["o"].astype(np.float32)

    def cross(a, b):
        return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                         a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)

    def dot(a, b):
        return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]

    with np.errstate(all="ignore"):
        ng = cross(e1, e2)
        c = v0 - o
        rr = cross(d, c)
        inv_det = np.float32(1) / dot(ng, d)
        u = dot(rr, e2) * inv_det
        v = dot(rr, e1) * inv_det
        w = (np.float32(1) - u) - v
        t = dot(ng, c) * inv_det
    return u, v, w, t, inv_det


def tri_corpus(rng_seed=7):
    """(tris[n, 3, 3], rays[n]) for strides 48 / 64: small-integer triangles with rays through vertices, along edges and through
    interior points (u, v or w exactly +-0), parallel rays (det = +-0), scaled by 2^k for k in -140 .. 70, and the overflow
    family of overflow_triangle"""
    rng = np.random.default_rng(rng_seed)
    tris, rays = [], []
    base = rng.integers(-3, 4, size=(64, 3, 3)).astype(np.float32)
    base[0] = [[0, 0, 0], [1, 0, 0], [0, 1, 0]]
    base[1] = [[0, 0, 0], [0, 1, 0], [1, 0, 0]]
    for k in list(range(-140, 71, 10)) + [-126, -149 + 24, 56, 58, 60, 62, 63, 64, 66, 68, 71]:
        s = np.float32(2.0 ** k) if k > -150 else np.float32(0)
        for t in base:
            bary = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (0.5, 0.5, 0), (0, 0.5, 0.5), (0.5, 0, 0.5), (0.25, 0.25, 0.5)]
            for wgt in bary:
                target = np.float32(wgt) @ t
                org = rng.integers(-4, 5, size=3).astype(np.float32) / 2
                d = target - org
                if not d.any():
                    continue
                for dd in (d, -d):
                    tris.append(t * s); rays.append(rays_of(org * s, dd)[0])
            # parallel to the plane: det = +-0
            n = np.cross(t[1] - t[0], t[2] - t[0])
            par = np.cross(n, [1, 0, 0]) if np.cross(n, [1, 0, 0]).any() else np.cross(n, [0, 1, 0])
            tris.append(t * s); rays.append(rays_of(t[0] * s - np.float32(par), par)[0])
    for a, b in ((60, 68), (61, 67), (62, 66), (62, 67), (63, 65), (63, 66), (61, 66), (62, 64), (60, 60)):
        tri, ray = overflow_triangle(a, b)
        tris.append(tri); rays.append(ray[0])
        tris.append(tri); rays.append(rays_of(ray["o"][0], [1e-3, 0, 1])[0])
    tris, rays = np.array(tris, np.float32), np.array(rays, ob.RAY_DTYPE)
    # tmax = +inf for a third, and bounded windows for some
    rays["tmax"][::3] = INF
    rays["tmin"][1::11] = np.float32(0.5)
    return tris, rays


def with_t_edges(tris, rays, t_ref):
    """each hit again with tmin == t and with tmax == t (accepted), and one ulp past each (rejected)"""
    hit = np.isfinite(t_ref)
    tt, tr, rr = t_ref[hit], tris[hit], rays[hit]
    out_t, out_r = [tris, tr, tr, tr, tr], [rays]
    for lo, hi in ((tt, None), (None, tt), (np.nextafter(tt, INF), None), (None, np.nextafter(tt, -INF))):
        r = rr.copy()
        if lo is not None:
            r["tmin"] = lo
        if hi is not None:
            r["tmax"] = hi
        out_r.append(r)
    return np.concatenate(out_t), np.concatenate(out_r)


def oracle_tri(tris, rays, stride, records=None, variant=0):
    rec = records if records is not None else np.ascontiguousarray(host.tri_records(tris, stride)).view(np.uint8).reshape(-1)
    orc = ob.Oracle(rec, rec, stride)
    ob.set_variant(variant)
    try:
        return np.array([orc.intersect_tri(i, rays[i]) for i in range(len(rays))], np.float32), rec
    finally:
        ob.set_variant(0)


def test_oracle_rejects_nan_barycentrics():
    """Known answer: the overflow triangle makes u = inf - inf = NaN with t = -0 in range.  The reference's x86 CPU path
    rejects it (the default NaN has its sign bit set); the oracle must say miss on every host, and so must any rule that
    replaces the sign test."""
    for a, b in ((62, 66), (63, 65), (60, 68)):
        tri, ray = overflow_triangle(a, b)
        rec = np.ascontiguousarray(host.tri_records(tri[None], 48)).view(np.uint8).reshape(-1)
        u, v, w, t, inv_det = tri_numpy(rec, ray)
        assert np.isnan(u[0]) and np.isnan(w[0]) and inv_det[0] != 0 and t[0] == 0, (a, b, u, v, w, t)
        for stride in (48, 64):
            r = np.ascontiguousarray(host.tri_records(tri[None], stride)).view(np.uint8).reshape(-1)
            assert math.isinf(ob.Oracle(r, r, stride).intersect_tri(0, ray)), f"oracle accepts a NaN barycentric ({a}, {b}, {stride})"
        # through the traversal as well: one leaf node over the triangle
        nodes, pidx, _ = host.build_cwbvh(tri[None])
        h = ob.Oracle(nodes, rec, 48).trace(ray)
        assert h["prim"][0] == ob.INVALID_PRIM and np.isinf(h["t"][0])


def test_nan_rule_equals_sign_rule_on_non_nan():
    """`hit < 0x40000000` (traverse.cuh tri_test) accepts exactly what the sign-bit test accepts whenever u, v, w are not NaN,
    and rejects every NaN — over the triangle corpus, u, v, w computed as the kernels compute them"""
    tris, rays = tri_corpus()
    rec = np.ascontiguousarray(host.tri_records(tris, 48)).view(np.uint8).reshape(-1)
    u, v, w, _, _ = tri_numpy(rec, rays)
    h = bits(u) | bits(v) | bits(w)
    nan = np.isnan(u) | np.isnan(v) | np.isnan(w)
    assert nan.sum() >= 9 and (~nan).sum() > 10000
    sign_rule, new_rule = (h & 0x80000000) == 0, h < 0x40000000
    assert (sign_rule[~nan] == new_rule[~nan]).all()
    assert not new_rule[nan].any()
    # with CUDA's canonical NaN (0x7FFFFFFF) the sign test would accept some of them
    hc = np.where(np.isnan(u), 0x7FFFFFFF, bits(u)) | np.where(np.isnan(v), 0x7FFFFFFF, bits(v)) | np.where(np.isnan(w), 0x7FFFFFFF, bits(w))
    assert ((hc & 0x80000000) == 0)[nan].any()


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [48, 64])
def test_tri_test_equals_oracle(probe, stride):
    tris, rays = tri_corpus()
    t0, _ = oracle_tri(tris, rays, stride)
    tris, rays = with_t_edges(tris, rays, t0)
    want, rec = oracle_tri(tris, rays, stride)
    assert np.isfinite(want).sum() > 2000
    for vd in (False, True):
        got = probe.tri_test(rec, stride, rays, variant_dir=vd)
        bad = np.nonzero(bits(got) != bits(want))[0]
        assert bad.size == 0, f"{bad.size} of {len(want)} differ (variant_dir={vd}), first {bad[:5]}: gpu {got[bad[:5]]} oracle {want[bad[:5]]}"
    # MODE 1's triangle direction: the caller's, zero components and all
    want_raw, _ = oracle_tri(tris, rays, stride, rec, VARIANT_ZERODIR_BOX_ONLY)
    got = probe.tri_test(rec, stride, rays, VARIANT_ZERODIR_BOX_ONLY, variant_dir=True)
    assert (bits(got) == bits(want_raw)).all()


HALF_SPECIAL = [0x0000, 0x8000, 0x0001, 0x8001, 0x03FF, 0x83FF, 0x0400, 0x7BFF, 0xFBFF, 0x7C00, 0xFC00, 0x7E00, 0xFE00,
                0x3C00, 0xBC00, 0x4000, 0xC000, 0x3800, 0x1000]


@pytest.mark.gpu
def test_tri_test_stride24_f16_edges(probe):
    """stride 24: f16 edges with subnormal halves, 65504, +-inf, NaN and -0, against small-integer v0 and aimed rays"""
    rng = np.random.default_rng(24)
    n = 20000
    rec = np.zeros((n, 6), np.uint32)
    rec[:, 0:3] = bits(rng.integers(-2, 3, size=(n, 3)).astype(np.float32))
    h = np.array(HALF_SPECIAL, np.uint32)
    lo = rng.choice(h, size=(n, 3))
    hi = rng.choice(h, size=(n, 3))
    plain = rng.random(n) < 0.5                                          # half the records: ordinary small edges
    lo[plain] = rng.choice(h[13:], size=(plain.sum(), 3))
    hi[plain] = rng.choice(h[13:], size=(plain.sum(), 3))
    rec[:, 3:6] = lo | (hi << 16)
    v0 = from_bits(rec[:, 0:3])
    with np.errstate(all="ignore"):
        e2 = lo.astype(np.uint16).view(np.float16).astype(np.float32)
        e1n = hi.astype(np.uint16).view(np.float16).astype(np.float32)   # v1 - v0
        bary = rng.choice([0.0, 0.25, 0.5, 1.0], size=(n, 2))
        target = v0 + np.float32(bary[:, :1]) * e1n + np.float32(bary[:, 1:]) * e2
    org = rng.integers(-4, 5, size=(n, 3)).astype(np.float32)
    d = np.nan_to_num(target - org, nan=1.0, posinf=1.0, neginf=-1.0).astype(np.float32)
    rays = rays_of(org, d, 0.0, F32_MAX)
    rays["tmax"][::4] = INF
    recb = rec.view(np.uint8).reshape(-1)
    want, _ = oracle_tri(None, rays, 24, recb)
    assert np.isfinite(want).sum() > 500
    for vd in (False, True):
        got = probe.tri_test(recb, 24, rays, variant_dir=vd)
        bad = np.nonzero(bits(got) != bits(want))[0]
        assert bad.size == 0, f"{bad.size} differ, first {bad[:5]}"


# ---- ray generation ---------------------------------------------------------------------------------------------------------
CAMERA = host.Camera((0.3, 1.1, 3.9), (0.0, 1.0, 0.0), 40.0)


def orc_view(view):
    v = ob.OrcView()
    C.memmove(C.byref(v), C.byref(view), C.sizeof(ob.OrcView))
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (2, 1), (1, 3), (7, 5), (33, 9), (101, 37), (640, 360), (16384, 8)])
def test_primary_dir_equals_oracle(probe, w, h):
    view = host.view_from_camera(CAMERA, w, h)
    ref = ob.primary_rays(view, w, h)
    i = np.arange(w * h)
    got = probe.primary_dir(view, w, h, i % w, i // w)
    assert (bits(got) == bits(ref["d"])).all(), f"{(bits(got) != bits(ref['d'])).any(axis=1).sum()} pixels differ"


def normal_records(stride):
    """triangles whose normal has nz = +-0, +-1, -1 + ulp, -1 + a few ulps, and generic ones; stride 64 stores ng as given"""
    ns = [(1, 0, 0), (0, 1, 0), (1, 1, 0), (0, 0, 1), (0, 0, -1), (0.3, -0.2, 0.9), (-0.5, 0.5, -0.7)]
    for z in (-1 + 2.0 ** -24, -1 + 2.0 ** -23, -1 + 2.0 ** -20, 1 - 2.0 ** -24):
        ns.append((math.sqrt(max(0.0, 1 - z * z)), 0.0, z))
    ns.append((0.0, -0.0, -1.0))
    tris = []
    for n in ns:
        n = np.asarray(n, np.float64)
        a = np.cross(n, [1, 0, 0]) if abs(n[0]) < 0.9 else np.cross(n, [0, 1, 0])
        a /= np.linalg.norm(a)
        b = np.cross(n, a)
        tris.append(np.array([[0, 0, 0], a, b], np.float32))              # cross(v0 - v1, v2 - v0) = cross(-a, b) ~ -n
    tris = np.array(tris, np.float32)
    rec = np.ascontiguousarray(host.tri_records(tris, stride)).view(np.uint8).reshape(-1)
    if stride == 64:
        r = rec.view(np.float32).reshape(-1, 16)
        r[:, 12:15] = np.array(ns, np.float32)
        rec = r.view(np.uint8).reshape(-1)
    return tris, rec, np.array(ns, np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_bounce_ray_equals_oracle(probe, stride):
    L = _oracle_lib()
    tris, rec, ns = normal_records(stride)
    view = host.view_from_camera(CAMERA, 64, 64)
    ov = orc_view(view)
    orc = ob.Oracle(rec, rec, stride)
    rng = np.random.default_rng(stride)
    cases = []
    fcs = [0, 1, 5, 1023, 1024, 2 ** 32 - 1, 2 ** 32 - 1024, 2 ** 32 - 1025, 2 ** 32 - 1023, 2 ** 31]
    for prim in range(len(ns)):
        n = ns[prim].astype(np.float64)
        pds = [-n, n, np.array([0.3, -0.4, 0.866])]
        perp = np.cross(n, [0, 0, 1]) if abs(n[2]) < 0.9 else np.cross(n, [1, 0, 0])
        pds += [perp, -perp]                                              # grazing: dot(n, -d) = +-0 in f32
        if ns[prim][2] == 0 and ns[prim][0] == 0:
            pds.append(np.array([1.0, 0.0, 0.0]))
        for pd in pds:
            pd = (pd / np.linalg.norm(pd)).astype(np.float32)
            for fc in fcs:
                cases.append((prim, pd, int(rng.integers(0, 2048)), int(rng.integers(0, 2048)), fc, float(rng.choice([0.5, 3.0, 1e-3]))))
    px = np.array([c[2] for c in cases]); py = np.array([c[3] for c in cases])
    got = probe.bounce_ray(stride, rec, view, px, py, np.array([c[1] for c in cases]), np.array([c[5] for c in cases]),
                           np.array([c[0] for c in cases]), np.array([c[4] for c in cases], np.uint32))
    want = np.zeros((len(cases), 6), np.float32)
    for i, (prim, pd, x, y, fc, t) in enumerate(cases):
        pr = rays_of(view.eye[:], pd)
        hit = np.array([(t, prim)], ob.HIT_DTYPE)
        out = np.zeros(1, ob.RAY_DTYPE)
        L.orc_bounce_ray(C.byref(orc.scene), C.byref(ov), pr.ctypes.data, hit.ctypes.data, x, y, fc, out.ctypes.data)
        want[i, 0:3], want[i, 3:6] = out["o"][0], out["d"][0]
    bad = np.nonzero((bits(got) != bits(want)).any(axis=1))[0]
    assert bad.size == 0, f"{bad.size} of {len(cases)} differ, first {[cases[b][0::4] for b in bad[:3]]}"


def uhash_np(a, b):
    a, b = np.asarray(a, np.uint32), np.asarray(b, np.uint32)
    with np.errstate(over="ignore"):
        x = (a * np.uint32(1597334673)) ^ (b * np.uint32(3812015801))
        x = x ^ (x >> np.uint32(16)); x = x * np.uint32(0x7FEB352D)
        x = x ^ (x >> np.uint32(15)); x = x * np.uint32(0x846CA68B)
        x = x ^ (x >> np.uint32(16))
    return x


def hash_noise_np(x, y, f):
    with np.errstate(over="ignore"):
        return uhash_np(x, (np.asarray(y, np.uint32) << np.uint32(11)) + np.asarray(f, np.uint32)).astype(np.float32) * np.float32(2.0 ** -32)


@pytest.mark.gpu
def test_uhash_and_hash_noise(probe):
    rng = np.random.default_rng(5)
    edge = np.array([0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF, 0xFFFFFBFF, 0xFFFFFC00, 2047, 2048], np.uint32)
    a = np.concatenate([np.repeat(edge, len(edge)), rng.integers(0, 2 ** 32, 200000, dtype=np.uint32)])
    b = np.concatenate([np.tile(edge, len(edge)), rng.integers(0, 2 ** 32, 200000, dtype=np.uint32)])
    c = np.concatenate([np.tile(edge[::-1], len(edge)), rng.integers(0, 2 ** 32, 200000, dtype=np.uint32)])
    assert (probe.uhash(a, b) == uhash_np(a, b)).all()
    assert (bits(probe.hash_noise(a, b, c)) == bits(hash_noise_np(a, b, c))).all()
    L = ob.lib()
    for i in range(0, len(a), 997):
        assert L.orc_uhash(int(a[i]), int(b[i])) == uhash_np(a[i], b[i])


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_instanced_bounce_normals_at_exponent_edges(probe, stride):
    """bounce_ray<S, true> on the records of normal_records scaled by 2^k (k = -32 .. 32; stride 24 keeps f16 edges, |k| <= 8)
    under W = 2^k P (P a signed axis permutation, optionally composed with a rotation): every direction finite and of unit
    length and in the hemisphere of the float64 world normal (instance_ref.c's bounce_one is held to the kernel's frames bit for
    bit in test_instance_kernels.py)"""
    tris, _, ns = normal_records(stride)
    keep = np.nonzero(np.abs(ns[:, 2] + 1) > 1e-3)[0]
    view = host.view_from_camera(CAMERA, 64, 64)
    rng = np.random.default_rng(stride)
    ks = (-8, 8) if stride == 24 else (-32, -24, -16, -8, 8, 16, 24, 32)
    for k in ks:
        for rotate in (False, True):
            P = np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]
            A = (np.linalg.qr(rng.normal(size=(3, 3)))[0] if rotate else np.eye(3)) @ P             # object_to_world = 2^-k A
            obj = (tris.astype(np.float64).reshape(-1, 3) @ np.linalg.inv(A).T * 2.0 ** k).astype(np.float32).reshape(tris.shape)
            rec = np.ascontiguousarray(host.tri_records(obj, stride)).view(np.uint8).reshape(-1)
            W = np.zeros((3, 4)); W[:, :3] = np.linalg.inv(A) * 2.0 ** k
            n = 4096
            prim = keep[np.arange(n) % len(keep)].astype(np.uint32)
            pd = rng.normal(size=(n, 3)); pd /= np.linalg.norm(pd, axis=1, keepdims=True)
            px, py = rng.integers(0, 2048, n), rng.integers(0, 2048, n)
            got = probe.bounce_ray(stride, rec, view, px, py, pd, np.full(n, 2.0), prim, np.zeros(n), np.tile(W, (n, 1, 1)))
            d = got[:, 3:6].astype(np.float64)
            assert np.isfinite(d).all(), (k, rotate)
            assert np.abs(np.linalg.norm(d, axis=1) - 1).max() <= 1e-6, (k, rotate)
            t3 = obj.astype(np.float64)[prim]
            nf = np.cross(t3[:, 0] - t3[:, 1], t3[:, 2] - t3[:, 0]) @ W[:, :3]                 # W^T n, by rows
            nf /= np.linalg.norm(nf, axis=1, keepdims=True)
            nf *= np.where((nf * -pd).sum(1) >= 0, 1.0, -1.0)[:, None]
            assert ((d * nf).sum(1) >= -1e-6).all(), (k, rotate)


# ---- float64 checks of the sampler ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bounce_directions_against_float64_and_distribution(probe):
    """Over 2^20 pixel x frame samples: the device's bounce direction within 2e-6 of a float64 evaluation of the same
    formula, in the hemisphere of the face normal turned toward the primary ray, with cos^2(theta) and the azimuth uniform
    (scipy KS, fixed seed, p > 1e-3)."""
    from scipy import stats
    stride = 48
    tris, rec, ns = normal_records(stride)
    keep = np.nonzero(np.abs(ns[:, 2] + 1) > 1e-3)[0]                  # away from the basis singularity nz = -1
    view = host.view_from_camera(CAMERA, 64, 64)
    n = 1 << 20
    i = np.arange(n)
    px, py, fc = (i % 1024).astype(np.uint32), ((i // 1024) % 256).astype(np.uint32), (i // (1024 * 256) * 7).astype(np.uint32)
    prim = keep[i % len(keep)].astype(np.uint32)
    pd = np.array([0.3, -0.4, -0.866], np.float32)
    pd = np.tile((pd / np.linalg.norm(pd)).astype(np.float32), (n, 1))
    got = probe.bounce_ray(stride, rec, view, px, py, pd, np.full(n, 2.0, np.float32), prim, fc)[:, 3:6].astype(np.float64)
    # float64: the face normal of the record, turned toward the primary ray, the same basis and the same (u0, u1)
    r = rec.view(np.float32).reshape(-1, 12).astype(np.float64)
    nf = np.cross(r[:, 4:7], r[:, 8:11])
    nf /= np.linalg.norm(nf, axis=1, keepdims=True)
    nf = nf[prim]
    nf *= np.where((nf * -pd.astype(np.float64)).sum(1) >= 0, 1.0, -1.0)[:, None]
    u0, u1 = hash_noise_np(px, py, fc).astype(np.float64), hash_noise_np(px, py, fc + np.uint32(1024)).astype(np.float64)
    l = np.stack([np.sqrt(u0) * np.cos(2 * np.pi * u1), np.sqrt(u0) * np.sin(2 * np.pi * u1), np.sqrt(np.maximum(0, 1 - u0))], 1)
    sign = np.where(nf[:, 2] >= 0, 1.0, -1.0)
    a = -1.0 / (sign + nf[:, 2])
    b = nf[:, 0] * nf[:, 1] * a
    b1 = np.stack([1 + sign * nf[:, 0] ** 2 * a, sign * b, -sign * nf[:, 0]], 1)
    b2 = np.stack([b, sign + nf[:, 1] ** 2 * a, -nf[:, 1]], 1)
    want = b1 * l[:, :1] + b2 * l[:, 1:2] + nf * l[:, 2:3]
    want /= np.linalg.norm(want, axis=1, keepdims=True)
    err = np.abs(got - want).max()
    assert err <= 2e-6, f"max |device - float64| = {err:.3g}"
    cos_t = (got * nf).sum(1)
    assert cos_t.min() >= -1e-6, "a bounce direction leaves the hemisphere"
    p1 = stats.kstest(np.clip(cos_t, 0, 1) ** 2, "uniform").pvalue
    phi = np.arctan2((got * b2).sum(1), (got * b1).sum(1)) % (2 * np.pi)
    p2 = stats.kstest(phi / (2 * np.pi), "uniform").pvalue
    print(f"bounce directions: max error vs float64 {err:.3g}, KS p(cos^2) = {p1:.3g}, p(azimuth) = {p2:.3g}")
    assert p1 > 1e-3 and p2 > 1e-3


@pytest.mark.gpu
def test_sincos_tau_error_bound(probe):
    """sin/cos(2 pi u) against float64 over 2^24 evenly spaced u and every float within 2^12 ulps of 0, 1/4, 1/2, 3/4, 1:
    <= 5e-7 absolute; bit for bit the oracle's on a sample"""
    u = [np.arange(1 << 24, dtype=np.float64) / (1 << 24)]
    for c in (0.0, 0.25, 0.5, 0.75, 1.0):
        cb = int(bits(np.float32(c)))
        k = np.arange(-4096, 4097)
        if c == 0.0:
            u.append(from_bits(np.arange(0, 4097, dtype=np.uint32)).astype(np.float64))
            u.append(-from_bits(np.arange(0, 4097, dtype=np.uint32)).astype(np.float64))
        else:
            u.append(from_bits((cb + k).astype(np.uint32)).astype(np.float64))
    u = np.concatenate(u).astype(np.float32)
    s, c = probe.sincos_tau(u)
    x = 2 * np.pi * u.astype(np.float64)
    err = max(np.abs(s - np.sin(x)).max(), np.abs(c - np.cos(x)).max())
    print(f"sincos_tau: max abs error {err:.3g} over {u.size} inputs")
    assert err <= 5e-7
    for i in range(0, u.size, 4099):
        assert tuple(np.float32(ob.sincos_tau(float(u[i])))) == (s[i], c[i])


# ---- shading ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, SHADE_PRIMARY, SHADE_BOUNCE, SHADE_OCCLUSION])
def test_shade_equals_oracle(probe, mode):
    """Every mode at t in {+-0, subnormal, 1, f32::MAX, +inf, NaN} and 2^20 log-spaced values: the byte equals orc_shade's,
    except where the float64 value of col^2.2 * 255 lies within 4 f32 ulps of an integer (powf is not bit-portable)."""
    L = _oracle_lib()
    special = np.array([0.0, -0.0, 1e-40, -1e-40, 1.0, F32_MAX, INF, -INF, np.nan, -1.0, 1e-4], np.float32)
    t = np.concatenate([special, np.logspace(-38, 38, 1 << 20, dtype=np.float64).astype(np.float32)])
    got = probe.shade(mode, t)
    want = np.array([L.orc_shade(mode, float(x)) for x in t], np.uint8)
    with np.errstate(all="ignore"):
        if mode == SHADE_PRIMARY:
            col = np.float32(1) / t
        elif mode == SHADE_OCCLUSION:
            col = np.where(t < F32_MAX, np.float32(0), np.float32(1))
        else:
            col = np.where(t < F32_MAX, t / (np.float32(1) + t), np.float32(1)).astype(np.float32)
        g = np.power(col.astype(np.float64), 2.2) * 255
    near = np.abs(g - np.round(g)) <= 4 * np.spacing(np.abs(g).astype(np.float32)).astype(np.float64)
    near &= np.isfinite(g) & (g != np.round(g))                         # exact integers (col 0 or 1) are exact in powf too
    diff = got != want
    print(f"shade mode {mode}: {near.sum()} of {t.size} cases within 4 ulps of an integer, {diff.sum()} differ")
    assert not (diff & ~near).any(), f"{(diff & ~near).sum()} bytes differ outside the rounding window: t = {t[diff & ~near][:5]}"
    assert (np.abs(got.astype(int) - want.astype(int)) <= 1).all()
