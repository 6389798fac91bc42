"""Instanced scenes (tray_cuda_scene_set_instances): BLAS placed by 3x4 transforms, only the TLAS rebuilt.

The TLAS must be what the device builder's TLAS leg builds (test_refit_tlas.tlas_reference) over the boxes of the rule stated in
include/tray_cuda.h, restated here in numpy (`instance_boxes`).  Traversal must be what tests/instance_ref.c traces: the oracle's
two-level loop, with the ray taken to object space at an instance and back at the TLAS.  The CPU tests hold that reference to
the oracle itself under identity transforms and the box rule to every transformed vertex; the `gpu` tests hold the device to
both, byte for byte and hit for hit, and to a double-precision brute force in world space."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_binding as ob
from conftest import ROOT, random_rays
from test_build_reference import many_small_objects, rays_at
from test_refit_tlas import tlas_reference
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu
KERNEL_STACK = 48
INVALID = 0xFFFFFFFF
F32_MAX = np.float32(3.402823466e+38)


# ---- the serial reference --------------------------------------------------------------------------------------------------


_ilib = None


def _inst_lib():
    """tests/instance_ref.c compiled with oracle/Makefile's flags, linked against the oracle library"""
    global _ilib
    if _ilib is None:
        ob.lib()
        d = tempfile.mkdtemp(prefix="tray_instance_ref_")
        try:
            so = os.path.join(d, "libinstance_ref.so")
            odir = os.path.join(ROOT, "oracle")
            subprocess.check_call(["/usr/bin/gcc", "-O3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared", "-o", so,
                                   os.path.join(ROOT, "tests", "instance_ref.c"), "-L" + odir, "-ltray_oracle", "-Wl,-rpath," + odir, "-lm"])
            L = C.CDLL(so)
        finally:
            shutil.rmtree(d, ignore_errors=True)
        vp = C.c_void_p
        L.inst_trace.restype = C.c_int
        L.inst_trace.argtypes = [vp, vp, vp, vp, C.c_uint64, C.c_int, C.c_uint32, vp, vp, vp, vp]
        L.inst_bounce_rays.restype = None
        L.inst_bounce_rays.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp, vp, vp]
        _ilib = L
    return _ilib


class Reference:
    """an instanced scene as instance_ref.c traces it: node bytes, records, blas_offsets (the root of every TLAS leaf),
    world_to_object by instance and the instance of every TLAS leaf (None: the plain two-level traversal)"""

    def __init__(self, nodes, rec, stride, blas, tlas_start, w2o=None, leaf_inst=None):
        self.orc = ob.Oracle(nodes, rec, stride, blas, tlas_start, True)
        self.w2o = None if w2o is None else np.ascontiguousarray(np.asarray(w2o, np.float32).reshape(-1, 12))
        self.leaf_inst = None if leaf_inst is None else np.ascontiguousarray(leaf_inst, np.uint32)
        self.w2o_leaf = None if w2o is None else np.ascontiguousarray(self.w2o[self.leaf_inst])

    @classmethod
    def of(cls, sc):
        """the reference of a device scene, from its downloaded bytes and transforms"""
        nodes, rec, _ = sc.download_bvh(prim_indices=False)
        i = sc.info()
        leaf, w2o = sc.download_instance_xforms()
        return cls(nodes, rec, i["tri_stride"], sc.download_instances(), i["tlas_start"], w2o, leaf)

    def trace(self, rays, any_hit=False, cap=KERNEL_STACK):
        """(hits, instance ids, counts (nodes, tris, insts), peak stack entries) per ray"""
        rays = np.ascontiguousarray(rays, dtype=ob.RAY_DTYPE)
        n = rays.shape[0]
        hits, inst = np.empty(n, ob.HIT_DTYPE), np.empty(n, np.uint32)
        cnt, peak = np.empty(n, ob.COUNT_DTYPE), np.empty(n, np.uint32)
        ptr = lambda a: None if a is None else a.ctypes.data
        rc = _inst_lib().inst_trace(C.byref(self.orc.scene), ptr(self.w2o_leaf), ptr(self.leaf_inst), rays.ctypes.data, n, int(any_hit), cap,
                                    hits.ctypes.data, inst.ctypes.data, cnt.ctypes.data, peak.ctypes.data)
        if rc != 0:
            raise RuntimeError(f"reference traversal failed ({rc})")
        return hits, inst, cnt, peak

    def bounce_rays(self, view, w, h, primary_rays, hits, inst, fc=0):
        out = np.empty(w * h, ob.RAY_DTYPE)
        v = ob._view(view)
        _inst_lib().inst_bounce_rays(C.byref(self.orc.scene), C.byref(v), w, h, fc, primary_rays.ctypes.data, hits.ctypes.data,
                                     inst.ctypes.data, None if self.w2o is None else self.w2o.ctypes.data, out.ctypes.data)
        return out


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same_hits(a, b):
    return np.array_equal(a["prim"], b["prim"]) and np.array_equal(bits(a["t"]), bits(b["t"]))


# ---- transforms, inverses and the box rule ---------------------------------------------------------------------------------


def rotation(rng):
    q = rng.normal(size=4)
    a, b, c, d = q / np.linalg.norm(q)
    return np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                     [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                     [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])


def xforms(kind, n, seed, spread=2.0):
    """n row-major 3x4 object_to_world float32 transforms of one kind"""
    rng = np.random.default_rng(seed)
    m = np.zeros((n, 3, 4))
    for k in range(n):
        R = np.eye(3)
        if kind in ("rotation", "mixed", "large"):
            R = rotation(rng)
        if kind == "uniform":
            R = np.eye(3) * rng.uniform(0.3, 3.0)
        if kind in ("nonuniform", "mixed"):
            R = R @ np.diag(rng.uniform(0.2, 3.0, 3))
        if kind == "mirror":
            R = rotation(rng) @ np.diag([-1.0, 1.0, 1.0])
        if kind == "shear":
            R = np.eye(3) + np.triu(rng.uniform(-0.8, 0.8, (3, 3)), 1)
        t = np.zeros(3)
        if kind != "identity":
            t = rng.uniform(-spread, spread, 3)
        if kind == "large":
            t = t + np.float64(1e6)
        m[k, :, :3], m[k, :, 3] = R, t
    return m.astype(np.float32)


def inverse(xf):
    """world_to_object in double: (n, 3, 4) float64"""
    m = np.asarray(xf, np.float64)
    W = np.linalg.inv(m[:, :, :3])
    return np.concatenate([W, -np.einsum("nij,nj->ni", W, m[:, :, 3])[:, :, None]], axis=2)


def root_box(node):
    """rule 1: the decoded box of a node, the union over its used slots of p + q 2^(e-127), in double"""
    node = np.asarray(node, np.uint8)
    p = node[0:12].view(np.float32).astype(np.float64)
    scale = np.ldexp(1.0, node[12:15].astype(np.int64) - 127)
    used = node[24:32] != 0
    q = node[32:80].reshape(3, 2, 8).astype(np.float64)       # axis, (lo, hi), slot
    lo = (p[:, None] + q[:, 0] * scale[:, None])[:, used].min(axis=1)
    hi = (p[:, None] + q[:, 1] * scale[:, None])[:, used].max(axis=1)
    return lo, hi


def f32_down(x):
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, np.float32(-np.inf)), f)


def f32_up(x):
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(np.inf)), f)


def instance_boxes(nodes, roots, xf):
    """rules 1-5 of tray_cuda_scene_set_instances: (lo, hi) float32 (n, 3) of every instance's TLAS primitive"""
    nodes = np.asarray(nodes, np.uint8).reshape(-1, 80)
    m = np.asarray(xf, np.float32).astype(np.float64)
    lo, hi = np.zeros((len(roots), 3), np.float32), np.zeros((len(roots), 3), np.float32)
    for k, r in enumerate(roots):
        bl, bh = root_box(nodes[r])
        c = np.array([[(bh if (i >> a) & 1 else bl)[a] for a in range(3)] for i in range(8)])
        M = m[k]
        v = np.stack([((M[i, 0] * c[:, 0] + M[i, 1] * c[:, 1]) + M[i, 2] * c[:, 2]) + M[i, 3] for i in range(3)], axis=1)
        mn, mx = v.min(axis=0), v.max(axis=0)
        pad = np.ldexp(max(np.abs(mn).max(), np.abs(mx).max()), -18)
        lo[k], hi[k] = f32_down(mn - pad), f32_up(mx + pad)
    return lo, hi


def identity(n):
    return np.tile(np.eye(3, 4, dtype=np.float32), (n, 1, 1))


# ---- CPU -------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("stride", [24, 48, 64])
def test_identity_reference_is_the_oracle(stride):
    """with W = I on the scene's own TLAS, instance_ref traces what orc_trace / orc_trace_any trace, bit for bit"""
    tris, offs = many_small_objects(300, seed=stride)
    r = ob.build_reference(tris, tri_stride=stride, object_offsets=offs)
    ts, blas = r["info"]["tlas_start"], r["blas_offsets"]
    ref = Reference(r["nodes"], r["tri_bytes"], stride, blas, ts, identity(blas.size), np.arange(blas.size))
    plain = Reference(r["nodes"], r["tri_bytes"], stride, blas, ts)
    rays = np.concatenate([random_rays(6000, seed=stride), rays_at(tris, 3000, seed=stride)])
    for any_hit in (False, True):
        want, cnt, _ = ref.orc.trace(rays, counts=True, any_hit=any_hit, stack_limit=KERNEL_STACK)
        for got, inst, gcnt, _ in (ref.trace(rays, any_hit), plain.trace(rays, any_hit)):
            assert same_hits(got, want), any_hit
            assert np.array_equal(gcnt, cnt), any_hit
            hit = want["prim"] != INVALID
            assert hit.sum() > 1000
            assert (inst[~hit] == INVALID).all()


@pytest.mark.parametrize("kind", ["rotation", "uniform", "nonuniform", "mirror", "shear", "large", "mixed"])
def test_box_rule_holds_every_transformed_vertex(kind):
    tris, offs = many_small_objects(60, seed=3)
    r = ob.build_reference(tris, object_offsets=offs)
    nodes, pi = r["nodes"].reshape(-1, 80), r["prim_indices"]
    rng = np.random.default_rng(4)
    roots = rng.integers(0, 60, size=200)                   # object k's BLAS root is node k
    xf = xforms(kind, roots.size, seed=5)
    lo, hi = instance_boxes(nodes, roots, xf)
    m = xf.astype(np.float64)
    for k, root in enumerate(roots):
        v = tris[offs[root]:offs[root + 1]].reshape(-1, 3).astype(np.float64)
        w = v @ m[k, :, :3].T + m[k, :, 3]
        assert (w >= lo[k]).all() and (w <= hi[k]).all(), (kind, k)
        assert np.isfinite(lo[k]).all() and np.isfinite(hi[k]).all()
    if kind == "large":
        assert (lo[:, 0] > 9e5).all()
    assert pi.size == tris.shape[0]


def test_wrappers_reject_bad_input_before_the_library():
    sc = cuda.TrayCudaScene.__new__(cuda.TrayCudaScene)
    sc._h = C.c_void_p()
    bad = [(np.zeros(0, np.uint32), np.zeros((0, 3, 4), np.float32)),            # no instances
           (np.zeros(2, np.uint32), np.zeros((2, 4, 4), np.float32)),            # 4x4, not 3x4
           (np.zeros(2, np.uint32), np.zeros((3, 3, 4), np.float32)),            # counts differ
           (np.zeros(2, np.float32), np.zeros((2, 3, 4), np.float32)),           # float roots
           (np.zeros((2, 1), np.uint32), np.zeros((2, 3, 4), np.float32)),       # 2-D roots
           (np.array([-1, 0]), np.zeros((2, 3, 4), np.float32)),                # negative root
           (np.zeros(2, np.uint32), np.zeros((2, 3, 4), np.int32))]             # integer transforms
    for roots, xf in bad:
        with pytest.raises(ValueError):
            sc.set_instances(roots, xf)


def test_instance_calls_without_a_scene():
    L = cuda.lib()
    roots, xf = np.zeros(1, np.uint32), identity(1)
    ms = C.c_float()
    assert L.tray_cuda_scene_set_instances(None, roots.ctypes.data, xf.ctypes.data, 1, 3, 0, C.byref(ms)) == -1
    assert L.tray_cuda_scene_download_instance_xforms(None, None, None) == -1
    assert L.tray_cuda_trace_instance(None, None, 0, 0, None, None, None, None) == -1
    assert L.tray_cuda_trace_instance_device(None, None, 0, 0, None, None, None, None) == -1
    assert L.tray_cuda_frame_download_instance(None, None, None) == -1


# ---- GPU -------------------------------------------------------------------------------------------------------------------


def placed(n_obj=64, n_inst=300, kind="mixed", seed=0, stride=48, **kw):
    """(scene, triangles, object offsets, roots, transforms): a built two-level scene with n_inst random instances of its objects"""
    tris, offs = many_small_objects(n_obj, seed=seed + 1)
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=offs)
    rng = np.random.default_rng(seed)
    roots = rng.integers(0, n_obj, size=n_inst).astype(np.uint32)
    xf = xforms(kind, n_inst, seed)
    sc.set_instances(roots, xf, **kw)
    return sc, tris, offs, roots, xf


def check_tlas(sc, roots, xf, max_leaf=3, radius=0, passes=4):
    """device TLAS bytes, blas_offsets and leaf_instance == tlas_reference over the numpy boxes; world_to_object within 1 ulp"""
    nodes, _, _ = sc.download_bvh(prim_indices=False)
    nodes = nodes.reshape(-1, 80)
    i = sc.info()
    ts = i["tlas_start"]
    lo, hi = instance_boxes(nodes, roots, xf)
    top, perm, exact = tlas_reference(lo, hi, max_leaf, radius, passes=passes)
    leaf, w2o = sc.download_instance_xforms()
    assert i["n_instances"] == len(roots) and i["n_nodes"] == ts + top.shape[0]
    assert np.array_equal(nodes[ts:], top), f"{int((nodes[ts:] != top).any(axis=1).sum())} TLAS nodes differ"
    assert np.array_equal(leaf, perm)
    assert np.array_equal(sc.download_instances(), np.asarray(roots, np.uint32)[perm])
    want = inverse(xf)
    err = np.abs(w2o.astype(np.float64) - want)
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    floor = 1e-12 * np.abs(want).max(axis=2, keepdims=True)           # numpy's own error where an entry is (nearly) zero
    assert ((err <= ulp) | (err <= floor)).all(), float((err / ulp).max())
    return exact


@gpu
@pytest.mark.parametrize("passes", [0, 4])
@pytest.mark.parametrize("radius", [1, 14, 64])
@pytest.mark.parametrize("max_leaf", [1, 2, 3])
@pytest.mark.parametrize("n_inst", [1, 2, 9, 1023, 1024, 1025, 5000])
def test_tlas_bytes(monkeypatch, n_inst, max_leaf, radius, passes):
    monkeypatch.setenv("TRAY_CUDA_BUILD_REINSERT", str(passes))
    sc, _, _, roots, xf = placed(n_obj=40, n_inst=n_inst, seed=n_inst + max_leaf, max_prims_per_leaf=max_leaf, search_radius=radius)
    try:
        assert np.unique(roots).size < n_inst or n_inst < 40          # instances share BLAS
        check_tlas(sc, roots, xf, max_leaf, radius, passes)
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
@pytest.mark.parametrize("kind", ["identity", "translation", "rotation", "uniform", "nonuniform", "mirror", "shear", "large", "mixed"])
def test_traversal_equals_the_reference(kind, stride):
    import torch
    n_inst = 500 if kind != "translation" else 2000
    sc, tris, offs, roots, xf = placed(n_obj=30 if kind != "translation" else 1, n_inst=n_inst, kind=kind, seed=7, stride=stride)
    try:
        ref = Reference.of(sc)
        # rays at instances (through their world-space triangles), random rays, rays from inside instances, zero components
        m = xf.astype(np.float64)
        rng = np.random.default_rng(1)
        k = rng.integers(0, n_inst, 4000)
        obj = tris.reshape(-1, 3, 3).astype(np.float64)
        tri = offs[roots[k]].astype(np.int64)
        c = np.einsum("nij,nj->ni", m[k, :, :3], obj[tri].mean(axis=1)) + m[k, :, 3]
        d = rng.normal(size=(4000, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
        at = np.zeros(4000, ob.RAY_DTYPE)
        at["o"] = (c - d * 3.0).astype(np.float32); at["d"] = d.astype(np.float32); at["tmax"] = F32_MAX
        at["d"][:200, 1:] = 0; at["d"][:200, 0] = 1                       # zero components
        inside = at.copy(); inside["o"] = c.astype(np.float32)
        rand = random_rays(6000, seed=3, lo=-2.5, hi=2.5)
        if kind == "large":
            rand["o"] += np.float32(1e6)
        rays = np.concatenate([at, inside, rand])
        for any_hit in (False, True):
            hits, ids = sc.traverse_instance(rays, any_hit=any_hit)
            want, wid, cnt, peak = ref.trace(rays, any_hit)
            assert same_hits(hits, want), any_hit
            assert np.array_equal(ids, wid), any_hit
            if kind != "large":                                # (at 1e6 an f32 origin is coarser than these objects)
                assert (want["prim"] != INVALID).sum() > 2000
            plain = sc.traverse(rays, any_hit=any_hit)
            assert same_hits(plain, want)
            h2, costs = sc.traverse_cost(rays, any_hit=any_hit)
            assert same_hits(h2, want)
            assert np.array_equal(costs["nodes"], cnt["nodes"]) and np.array_equal(costs["tris"], cnt["tris"])
            assert np.array_equal(costs["instances"], cnt["insts"]) and np.array_equal(costs["stack"], peak)
            sc.set_counting(True)
            sc.traverse(rays, any_hit=any_hit)
            tot = sc.counters()[0]
            sc.set_counting(False)
            assert tot["nodes"] == costs["nodes"].sum() and tot["tris"] == costs["tris"].sum() and tot["instances"] == costs["instances"].sum()
            # device form
            d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
            d_hits = torch.zeros(rays.size * 8, dtype=torch.uint8, device="cuda")
            d_ids = torch.zeros(rays.size, dtype=torch.int32, device="cuda")
            sc.traverse_instance_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr(), d_ids.data_ptr(), timed=True, any_hit=any_hit)
            assert same_hits(d_hits.cpu().numpy().view(ob.HIT_DTYPE), want)
            assert np.array_equal(d_ids.cpu().numpy().view(np.uint32), wid)
    finally:
        sc.close()


@gpu
def test_pipelined_host_path_and_one_blas_under_hundreds_of_instances():
    """>= 2^18 rays take the chunked host pipeline; one BLAS placed 800 times"""
    sc, tris, offs, roots, xf = placed(n_obj=1, n_inst=800, kind="mixed", seed=11, stride=48)
    try:
        ref = Reference.of(sc)
        rays = random_rays(1 << 19, seed=12, lo=-2.5, hi=2.5)
        hits, ids = sc.traverse_instance(rays)
        want, wid, _, _ = ref.trace(rays)
        assert same_hits(hits, want) and np.array_equal(ids, wid)
        assert np.unique(wid[wid != INVALID]).size > 100
    finally:
        sc.close()


def brute_force(tris, offs, roots, xf, rays):
    """(t, instance, object triangle, second-closest t, |cos| between ray and triangle) of the closest hit of every ray over every
    instance's world-space triangles, in double"""
    m = xf.astype(np.float64)
    obj = tris.reshape(-1, 3, 3).astype(np.float64)
    o, d = rays["o"].astype(np.float64), rays["d"].astype(np.float64)
    best = np.full(rays.size, np.inf); inst = np.full(rays.size, -1); tri = np.full(rays.size, -1)
    second = np.full(rays.size, np.inf); cos = np.zeros(rays.size)
    for k, r in enumerate(roots):
        t = obj[offs[r]:offs[r + 1]] @ m[k, :, :3].T + m[k, :, 3]        # (m, 3, 3) world vertices
        for j in range(t.shape[0]):
            v0, e1, e2 = t[j, 0], t[j, 1] - t[j, 0], t[j, 2] - t[j, 0]
            p = np.cross(d, e2); det = p @ e1
            with np.errstate(divide="ignore", invalid="ignore"):
                s = o - v0; u = (s * p).sum(1) / det
                q = np.cross(s, e1); v = (d * q).sum(1) / det; tt = (q @ e2) / det
            ok = (u >= 0) & (v >= 0) & (u + v <= 1) & (tt >= 0) & np.isfinite(tt)
            tt = np.where(ok, tt, np.inf)
            closer = tt < best
            n = np.cross(e1, e2)
            cos = np.where(closer, np.abs(d @ n) / np.linalg.norm(n), cos)
            second = np.where(closer, best, np.minimum(second, tt))
            best = np.where(closer, tt, best); inst = np.where(closer, k, inst); tri = np.where(closer, offs[r] + j, tri)
    return best, inst, tri, second, cos


@gpu
@pytest.mark.parametrize("kind", ["mixed", "mirror", "shear"])
def test_hits_agree_with_a_world_space_brute_force(kind):
    sc, tris, offs, roots, xf = placed(n_obj=20, n_inst=60, kind=kind, seed=21)
    try:
        pi = sc.download_bvh()[2]
        rng = np.random.default_rng(22)
        n = 3000
        k = rng.integers(0, roots.size, n)
        j = offs[roots[k]].astype(np.int64) + (rng.random(n) * (offs[roots[k] + 1] - offs[roots[k]]).astype(np.float64)).astype(np.int64)
        b = rng.uniform(0.1, 0.8, (n, 2)); b[b.sum(1) > 0.9] *= 0.45
        obj = tris.reshape(-1, 3, 3).astype(np.float64)[j]
        p = obj[:, 0] + b[:, :1] * (obj[:, 1] - obj[:, 0]) + b[:, 1:] * (obj[:, 2] - obj[:, 0])
        m = xf.astype(np.float64)
        target = np.einsum("nij,nj->ni", m[k, :, :3], p) + m[k, :, 3]
        d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
        rays = np.zeros(n, ob.RAY_DTYPE)
        rays["o"] = (target - 5 * d).astype(np.float32); rays["d"] = d.astype(np.float32); rays["tmax"] = F32_MAX
        hits, ids = sc.traverse_instance(rays)
        t, inst, tri, second, cos = brute_force(tris, offs, roots, xf, rays)
        unique = np.isfinite(t) & (second > t * (1 + 1e-5) + 1e-12)
        assert unique.sum() > n // 2
        assert np.array_equal(ids[unique], inst[unique])
        assert np.array_equal(pi[hits["prim"][unique]], tri[unique])
        # the f32 error of t grows as 1 / cos at grazing incidence: the 1e-5 bound holds away from it
        steep = unique & (cos > 0.1)
        assert steep.sum() > n // 3
        assert (np.abs(hits["t"][steep] - t[steep]) <= 1e-5 * t[steep]).all()
    finally:
        sc.close()


def reference_frame(ref, view, w, h, fc=0):
    """primary trace, transformed-normal bounce, bounce trace and shading, as the frame operator computes them"""
    prays = ob.primary_rays(view, w, h)
    ph, pid, pcnt, ppeak = ref.trace(prays)
    brays = ref.bounce_rays(view, w, h, prays, ph, pid, fc)
    bh, bid, bcnt, bpeak = ref.trace(brays)
    shoot = ph["t"] < F32_MAX
    bh["t"][~shoot] = np.inf; bh["prim"][~shoot] = INVALID; bid[~shoot] = INVALID
    shade = ob.lib().orc_shade
    shade.argtypes, shade.restype = [C.c_uint32, C.c_float], C.c_uint8
    g = np.array([shade(2, float(bh["t"][i])) if shoot[i] else shade(1, float(ph["t"][i])) for i in range(w * h)], np.uint8)
    rgba = np.stack([g, g, g, np.full_like(g, 255)], axis=1).reshape(h, w, 4)
    return dict(primary=ph, bounce=bh, bounce_rays=brays, rgba=rgba, pid=pid, bid=bid, pcost=(pcnt, ppeak), bcost=(bcnt, bpeak), shoot=shoot)


FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_COUNTERS | cuda.RENDER_KEEP_RAYS


def cornell_instances(cornell, stride=48):
    """the Cornell box built two-level, every object placed twice: where it is, and turned and shrunk beside itself"""
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets()
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=offs)
    n = offs.size - 1
    roots = np.concatenate([np.arange(n), np.arange(n)]).astype(np.uint32)
    ext = float(np.ptp(tris.reshape(-1, 3), axis=0).max())
    turn = xforms("mixed", n, seed=31, spread=0.05 * ext).astype(np.float64)
    moved = np.zeros((n, 3, 4))
    for k in range(n):                                         # turned and shrunk about the object's own centre, then shifted
        c = tris[offs[k]:offs[k + 1]].reshape(-1, 3).astype(np.float64).mean(axis=0)
        R = 0.7 * rotation(np.random.default_rng(k))
        moved[k, :, :3], moved[k, :, 3] = R, c - R @ c + turn[k, :, 3]
    xf = np.concatenate([identity(n), moved.astype(np.float32)])
    sc.set_instances(roots, xf)
    return sc, tris, offs, roots, xf


def check_frame(sc, want):
    """the last frame of `sc` (one shard) == the reference frame: hits, instances, bounce rays, RGBA, ray costs"""
    got = sc.download(primary=True, bounce=True, bounce_rays=True, rgba=True)
    ids = sc.download_instance(primary=True, bounce=True)
    cost = sc.download_cost(primary=True, bounce=True)
    sh = want["shoot"]
    assert same_hits(got["primary"], want["primary"]) and same_hits(got["bounce"], want["bounce"])
    assert np.array_equal(ids["primary"], want["pid"]) and np.array_equal(ids["bounce"], want["bid"])
    assert np.array_equal(got["bounce_rays"][sh].view(np.uint32), want["bounce_rays"][sh].view(np.uint32))
    assert np.array_equal(got["rgba"], want["rgba"])
    for name, (cnt, peak), mask in (("primary", want["pcost"], np.ones(sh.size, bool)), ("bounce", want["bcost"], sh)):
        c = cost[name]
        assert np.array_equal(c["nodes"][mask], cnt["nodes"][mask]) and np.array_equal(c["tris"][mask], cnt["tris"][mask]), name
        assert np.array_equal(c["instances"][mask], cnt["insts"][mask]) and np.array_equal(c["stack"][mask], peak[mask]), name


@gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
@pytest.mark.parametrize("in_flight", [1, 2, 3])
def test_frames_equal_the_reference_frame(cornell, in_flight, stride):
    sc, *_ = cornell_instances(cornell, stride)
    try:
        w, h = 200, 120
        view = host.view_from_camera(cornell.camera, w, h)
        ref = reference_frame(Reference.of(sc), view, w, h)
        assert ref["shoot"].sum() > 5000 and (ref["pid"] >= cornell.object_offsets().size - 1).any()
        sc.set_frames_in_flight(in_flight)
        sc.set_ray_cost(True)
        for overlap in (False, True, False):                 # OVERLAP is ignored on an instanced scene: the same frame
            sc.render(view, w, h, 0, FLAGS | (cuda.RENDER_OVERLAP if overlap else 0))
            sc.sync()
            check_frame(sc, ref)
        for shard in range(3):
            sc.render(view, w, h, 0, FLAGS, shard=shard, shards=3)
            sc.sync()
            got = sc.download(primary=True)
            ids = sc.download_instance(primary=True, bounce=True)
            own = cuda.shard_mask(w, h, shard, 3)
            assert same_hits(got["primary"][own], ref["primary"][own])
            assert np.array_equal(ids["primary"][own], ref["pid"][own]) and (ids["primary"][~own] == INVALID).all()
            assert np.array_equal(ids["bounce"][own], ref["bid"][own]) and (ids["bounce"][~own] == INVALID).all()
    finally:
        sc.close()


@gpu
def test_identity_instances_of_a_build_tlas_scene(cornell):
    """t is bit-identical to the plain scene on every ray and pixel; prim and instance differ only on equal-t ties"""
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets()
    plain = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        blas = plain.download_instances()
        sc.set_instances(blas, identity(blas.size))
        ref = Reference.of(sc)
        rays = rays_at(tris, 40000, seed=42)
        a, b = plain.traverse(rays), sc.traverse(rays)
        ids = sc.traverse_instance(rays)[1]
        assert np.array_equal(bits(a["t"]), bits(b["t"]))
        want, wid, _, _ = ref.trace(rays)
        assert same_hits(b, want) and np.array_equal(ids, wid)
        d = a["prim"] != b["prim"]
        orc = ob.Oracle(*plain.download_bvh(prim_indices=False)[:2], 48, blas, plain.info()["tlas_start"], True)
        for i in np.flatnonzero(d)[:200]:
            r = rays[i:i + 1].copy(); r["tmax"] = F32_MAX
            assert orc.intersect_tri(a["prim"][i], r) == orc.intersect_tri(b["prim"][i], r) == a["t"][i]
        assert (ids != INVALID).sum() > 20000
        w, h = 256, 144
        view = host.view_from_camera(cornell.camera, w, h)
        out = []
        for s in (plain, sc):
            s.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
            s.sync()
            out.append(s.download(primary=True, bounce=True, rgba=True))
        for k in ("primary", "bounce"):
            assert np.array_equal(bits(out[0][k]["t"]), bits(out[1][k]["t"])), k
        assert np.array_equal(out[0]["rgba"], out[1]["rgba"])
    finally:
        plain.close()
        sc.close()


def state(sc):
    nodes, rec, _ = sc.download_bvh(prim_indices=False)
    i = sc.info()
    return dict(nodes=nodes, rec=rec, blas=sc.download_instances(), xf=sc.download_instance_xforms(), exact=sc.exact_node_test(),
                info={k: v for k, v in i.items() if k not in ("device", "device_bytes", "l2_persist_bytes")})


def same_state(a, b):
    return (np.array_equal(a["nodes"], b["nodes"]) and np.array_equal(a["rec"], b["rec"]) and np.array_equal(a["blas"], b["blas"])
            and all(np.array_equal(x, y) for x, y in zip(a["xf"], b["xf"])) and a["exact"] == b["exact"] and a["info"] == b["info"])


@gpu
def test_sequences_equal_a_fresh_scene():
    tris, offs = many_small_objects(50, seed=51)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        rays = random_rays(8000, seed=52, lo=-2.5, hi=2.5)
        first = None
        for step, n in enumerate([300, 1200, 40, 1200, 700, 2]):
            rng = np.random.default_rng(step)
            roots = rng.integers(0, 50, n).astype(np.uint32)
            xf = xforms("mixed", n, seed=step + 60)
            t = {}
            sc.set_instances(roots, xf, timings=t)
            assert t["ms_set_instances"] > 0
            bytes_now = sc.info()["device_bytes"]
            if step == 1:
                first = bytes_now
            if step > 1:
                assert bytes_now == first, step               # no call after the largest one grows anything
            fresh = cuda.TrayCudaScene.build(tris, object_offsets=offs)
            try:
                fresh.set_instances(roots, xf)
                assert same_state(state(sc), state(fresh)), step
                a, b = sc.traverse_instance(rays), fresh.traverse_instance(rays)
                assert same_hits(a[0], b[0]) and np.array_equal(a[1], b[1]), step
            finally:
                fresh.close()
            check_tlas(sc, roots, xf)
    finally:
        sc.close()


@gpu
def test_refit_rebuild_tlas_on_an_instanced_scene():
    """refit every BLAS, then the TLAS of set_instances over the moved roots == a fresh scene refit and then instanced"""
    tris, offs = many_small_objects(40, seed=71)
    moved = host.jitter(tris, 72, frac=0.2)
    roots = np.random.default_rng(73).integers(0, 40, 500).astype(np.uint32)
    xf = xforms("mixed", 500, seed=74)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    fresh = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        sc.set_instances(roots, xf)
        t = {}
        sc.refit_rebuild_tlas(moved, timings=t)
        assert t["ms_refit_rebuild_tlas"] > 0
        fresh.refit(moved)
        fresh.set_instances(roots, xf)
        assert same_state(state(sc), state(fresh))
        rays = random_rays(8000, seed=75, lo=-2.5, hi=2.5)
        want, wid, _, _ = Reference.of(fresh).trace(rays)
        hits, ids = sc.traverse_instance(rays)
        assert same_hits(hits, want) and np.array_equal(ids, wid)
    finally:
        sc.close()
        fresh.close()


@gpu
def test_refusals_change_nothing():
    tris, offs = many_small_objects(20, seed=81)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    flat = cuda.TrayCudaScene.build(tris)
    L = cuda.lib()
    try:
        # a scene that is not instanced refuses the instance calls
        rays = random_rays(100, seed=1)
        with pytest.raises(cuda.TrayCudaError):
            sc.traverse_instance(rays)
        with pytest.raises(cuda.TrayCudaError):
            sc.download_instance_xforms()
        with pytest.raises(cuda.TrayCudaError):
            flat.set_instances(np.zeros(1, np.uint32), identity(1))             # no TLAS
        roots, xf = np.arange(20, dtype=np.uint32), xforms("mixed", 20, seed=82)
        sc.set_instances(roots, xf)
        before = state(sc)
        view = host.view_from_camera(host.Camera((0, 0, -4), (0, 0, 0), 60.0), 64, 32)
        sc.render(view, 64, 32, 0, cuda.RENDER_BOUNCE)
        sc.sync()
        frame_before = sc.download(primary=True, bounce=True)
        singular = xf.copy(); singular[3, :, :3] = 0
        nan = xf.copy(); nan[5, 1, 3] = np.nan
        huge = xf.copy(); huge[2] = np.eye(3, 4, dtype=np.float32); huge[2, :, 3] = np.finfo(np.float32).max   # box overflows f32
        tiny = xf.copy(); tiny[2, :, :3] = np.float32(1e-39) * np.eye(3, dtype=np.float32)     # inverse overflows f32
        bad_root = roots.copy(); bad_root[7] = 20 + 3                                              # a node that is no BLAS root
        ms = C.c_float()
        cases = [(bad_root, xf), (roots, singular), (roots, nan), (roots, huge), (roots, tiny)]
        for r, x in cases:
            with pytest.raises(cuda.TrayCudaError):
                sc.set_instances(r, x)
        assert L.tray_cuda_scene_set_instances(sc._h, roots.ctypes.data, xf.ctypes.data, 0, 3, 0, C.byref(ms)) == -1
        assert L.tray_cuda_scene_set_instances(sc._h, None, xf.ctypes.data, 20, 3, 0, C.byref(ms)) == -1
        assert L.tray_cuda_scene_set_instances(sc._h, roots.ctypes.data, xf.ctypes.data, 20, 4, 0, C.byref(ms)) == -1
        assert L.tray_cuda_scene_set_instances(sc._h, roots.ctypes.data, xf.ctypes.data, 20, 3, 65, C.byref(ms)) == -1
        with pytest.raises(cuda.TrayCudaError):
            sc.refit(tris)                                                     # its TLAS leaves are transformed boxes
        with pytest.raises(cuda.TrayCudaError):
            sc.set_variant(cuda.VARIANT_TIE_LAST)
        assert same_state(state(sc), before)
        after = sc.download(primary=True, bounce=True)
        assert same_hits(after["primary"], frame_before["primary"]) and same_hits(after["bounce"], frame_before["bounce"])
        # a scene with variants refuses set_instances
        other = cuda.TrayCudaScene.build(tris, object_offsets=offs)
        try:
            other.set_variant(cuda.VARIANT_TIE_LAST)
            with pytest.raises(cuda.TrayCudaError):
                other.set_instances(roots, xf)
            other.set_variant(0)
            other.set_instances(roots, xf)
        finally:
            other.close()
    finally:
        sc.close()
        flat.close()


@gpu
def test_group_replicas_are_one_device():
    if cuda.device_count() < 2:
        pytest.skip("one device")
    tris, offs = many_small_objects(30, seed=91)
    r = ob.build_reference(tris, object_offsets=offs)
    g = cuda.TrayCudaGroup(r["nodes"], r["tri_bytes"], 48, r["blas_offsets"], r["info"]["tlas_start"], devices=(0, 1))
    one = cuda.TrayCudaScene(r["nodes"], r["tri_bytes"], 48, r["blas_offsets"], r["info"]["tlas_start"])
    try:
        roots, xf = np.random.default_rng(92).integers(0, 30, 400).astype(np.uint32), xforms("mixed", 400, seed=93)
        for i in range(2):
            g.scene(i).set_instances(roots, xf)
        one.set_instances(roots, xf)
        rays = random_rays(5000, seed=94, lo=-2.5, hi=2.5)
        want = one.traverse_instance(rays)
        for i in range(2):
            s = g.scene(i)
            assert same_state(state(s), state(one))
            got = s.traverse_instance(rays)
            assert same_hits(got[0], want[0]) and np.array_equal(got[1], want[1])
    finally:
        g.close()
        one.close()
