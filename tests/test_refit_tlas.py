"""Refit every BLAS and rebuild the TLAS (tray_cuda_scene_refit_rebuild_tlas).

The BLAS part must be what a refit writes (test_refit.py's refit_reference); the TLAS what the device builder's TLAS leg builds
over the BLAS roots' exact boxes in canonical order (by blas_offsets value).  `tlas_reference` states that leg serially: it
runs oracle/build_ref.c's PLOC, reinsertion and collapse over given boxes (tests/tlas_ref.c).  The CPU tests hold it to
orc_build_ref's own TLAS; the `gpu` tests hold the device to it, to tray_cuda_scene_build_tlas on the moved triangles and to a
plain refit, byte for byte, and the rebuilt scene to a scene created fresh from its bytes and to the oracle, hit for hit."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import cwbvh_bytes as cb
import oracle_binding as ob
from conftest import ROOT, random_rays
from test_build_reference import from_ordered, many_small_objects, ordered, rays_at, soup, tri_boxes
from test_refit import (FLAGS, _moved_cases, fresh_like, frame, jitter, refit_reference, refit_two_level, rigid, same_frame,
                        same_hits)
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu
KERNEL_STACK = 48


# ---- the serial reference --------------------------------------------------------------------------------------------------


class _TlasResult(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("n_nodes", C.c_uint32), ("perm", C.c_void_p), ("force_exact", C.c_int)]


_tlib = None


def _tlas_lib():
    """tests/tlas_ref.c compiled with oracle/Makefile's flags into a temporary directory"""
    global _tlib
    if _tlib is None:
        d = tempfile.mkdtemp(prefix="tray_tlas_ref_")
        try:
            so = os.path.join(d, "libtlas_ref.so")
            subprocess.check_call(["/usr/bin/gcc", "-O3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                                   "-o", so, os.path.join(ROOT, "tests", "tlas_ref.c"), "-lm"])
            L = C.CDLL(so)
        finally:
            shutil.rmtree(d, ignore_errors=True)
        L.orc_build_ref_tlas.restype = C.c_int
        L.orc_build_ref_tlas.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(ob.OrcBuildParams), C.POINTER(_TlasResult)]
        L.orc_tlas_free.argtypes = [C.POINTER(_TlasResult)]
        _tlib = L
    return _tlib


def tlas_reference(lo, hi, max_leaf=3, radius=0, passes=4, visits=192, rounds=3):
    """(TLAS nodes (m, 80), perm, force_exact) of the TLAS leg over boxes [lo[i], hi[i]]: perm[j] = the box of TLAS leaf j"""
    lo = np.ascontiguousarray(lo, np.float32).reshape(-1, 3)
    hi = np.ascontiguousarray(hi, np.float32).reshape(-1, 3)
    prm = ob.OrcBuildParams(max_leaf, radius, passes, visits, rounds)
    res = _TlasResult()
    rc = _tlas_lib().orc_build_ref_tlas(lo.ctypes.data, hi.ctypes.data, lo.shape[0], C.byref(prm), C.byref(res))
    if rc != 0:
        raise RuntimeError(f"reference TLAS build failed ({rc})")
    try:
        nodes = np.frombuffer((C.c_uint8 * (res.n_nodes * 80)).from_address(res.nodes), np.uint8).reshape(-1, 80).copy()
        perm = np.frombuffer((C.c_uint32 * lo.shape[0]).from_address(res.perm), np.uint32).copy()
        return nodes, perm, bool(res.force_exact)
    finally:
        _tlas_lib().orc_tlas_free(C.byref(res))


def object_boxes(tris, offs):
    """exact box of every object (triangles offs[k] .. offs[k + 1]) under the device's min / max order"""
    o = ordered(np.asarray(tris, np.float32).reshape(-1, 3, 3))
    starts = np.asarray(offs, np.int64)[:-1]
    return from_ordered(np.minimum.reduceat(o.min(axis=1), starts, axis=0)), from_ordered(np.maximum.reduceat(o.max(axis=1), starts, axis=0))


def rebuild_reference(nodes, slot_tris, blas, tlas_start, max_leaf=3, radius=0):
    """(node array, blas_offsets) a rebuild must leave: every BLAS as refit_two_level refits it, then the TLAS of tlas_reference
    over the BLAS roots' boxes in canonical order (blas_offsets sorted)"""
    out, (nlo, nhi) = refit_reference(nodes, np.unique(blas), *tri_boxes(slot_tris))
    canon = np.sort(np.asarray(blas, np.uint32))
    top, perm, _ = tlas_reference(from_ordered(nlo[canon]), from_ordered(nhi[canon]), max_leaf, radius)
    return np.concatenate([out[:tlas_start], top]), canon[perm]


def tlas_at_the_tail(g):
    """a generated two-level tree with its TLAS region moved behind every BLAS: (nodes, blas, tlas_start).  BLAS child indices
    are relative to their root and TLAS ones to tlas_start, so only blas_offsets and tlas_start change."""
    ts, m = g.tlas_start, g.regions[-1][1]
    nodes = np.concatenate([g.nodes[:ts], g.nodes[ts + m:], g.nodes[ts:ts + m]])
    blas = np.where(g.blas >= ts + m, g.blas - m, g.blas).astype(np.uint32)
    return nodes, blas, len(g.nodes) - m


# ---- CPU -------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("passes", [0, 4])
@pytest.mark.parametrize("radius", [1, 14, 64])
@pytest.mark.parametrize("max_leaf", [1, 2, 3])
@pytest.mark.parametrize("n_obj", [1, 2, 9, 400, 1023, 1024, 1025, 3000])
def test_tlas_reference_is_the_tlas_of_the_build_reference(n_obj, max_leaf, radius, passes):
    """over the BLAS-root boxes of orc_build_ref's forest, the TLAS leg alone gives orc_build_ref's TLAS nodes and blas_offsets
    (object counts on both sides of the 1024 clusters where the device's PLOC tail takes over)"""
    tris, offs = many_small_objects(n_obj, seed=n_obj + max_leaf)
    r = ob.build_reference(tris, max_leaf=max_leaf, radius=radius, object_offsets=offs, passes=passes)
    ts = r["info"]["tlas_start"]
    top, perm, exact = tlas_reference(*object_boxes(tris, offs), max_leaf=max_leaf, radius=radius, passes=passes)
    assert np.array_equal(top, r["nodes"].reshape(-1, 80)[ts:])
    assert np.array_equal(perm, r["blas_offsets"])
    assert not exact


def test_rebuild_reference_on_a_reference_build():
    """rebuilding the TLAS of a reference build over moved triangles is the reference build of the moved triangles, TLAS for TLAS"""
    tris, offs = many_small_objects(300, seed=5)
    r = ob.build_reference(tris, object_offsets=offs)
    ts, pi = r["info"]["tlas_start"], r["prim_indices"]
    moved = rigid(tris, offs, 3)
    nodes, blas = rebuild_reference(r["nodes"], moved[pi], r["blas_offsets"], ts)
    want = ob.build_reference(moved, object_offsets=offs)
    assert np.array_equal(nodes[ts:], want["nodes"].reshape(-1, 80)[want["info"]["tlas_start"]:])
    assert np.array_equal(blas, want["blas_offsets"])
    assert np.array_equal(nodes[:ts], refit_two_level(r["nodes"], moved[pi], r["blas_offsets"], ts)[:ts])


def test_generated_trees_with_the_tlas_at_the_tail_stay_valid():
    """the tail layout of a generated tree traces like the tree it came from"""
    tris = cb.random_tris(500, 3)
    t, offs = cb.random_objects(tris, 6, 3)
    g = cb.random_tlas(t, offs, 3)
    s = g.scene(t, 48, 3)
    nodes, blas, ts = tlas_at_the_tail(g)
    rays = random_rays(2000, 3)
    a = s.oracle().trace(rays, stack_limit=KERNEL_STACK)
    b = ob.Oracle(nodes, s.rec, 48, blas, ts, True).trace(rays, stack_limit=KERNEL_STACK)
    assert same_hits(a, b)


def test_rebuild_arguments_without_a_device():
    """NULL scene or triangles are refused before any device is touched"""
    L = cuda.lib()
    t = np.zeros(9, np.float32)
    ms = C.c_float()
    assert L.tray_cuda_scene_refit_rebuild_tlas(None, t.ctypes.data, 1, 3, 0, C.byref(ms)) == -1
    assert L.tray_cuda_scene_refit_rebuild_tlas_device(None, t.ctypes.data, 1, 3, 0, None, None) == -1
    assert L.tray_cuda_scene_refit_rebuild_tlas(None, None, 0, 3, 0, None) == -1


# ---- GPU -------------------------------------------------------------------------------------------------------------------


def state(sc):
    """everything a rebuild may change: nodes, records, blas_offsets, info, exact node test"""
    nodes, rec, _ = sc.download_bvh(prim_indices=False)
    return dict(nodes=nodes.reshape(-1, 80), rec=rec, blas=sc.download_instances(), info=sc.info(), exact=sc.exact_node_test())


def same_state(a, b):
    """the same tree and scene info (on whichever device)"""
    info = lambda x: {k: v for k, v in x["info"].items() if k != "device"}
    return (np.array_equal(a["nodes"], b["nodes"]) and np.array_equal(a["rec"], b["rec"]) and np.array_equal(a["blas"], b["blas"])
            and info(a) == info(b) and a["exact"] == b["exact"])


def expected_exact(nodes):
    """the exact node test a scene created from these bytes takes"""
    return bool((np.asarray(nodes).reshape(-1, 80)[:, 12:15] >= 167).any())


@gpu
@pytest.mark.parametrize("max_leaf,radius", [(3, 0), (1, 5), (2, 64)])
def test_identity_on_builder_scenes(max_leaf, radius):
    tris, offs = many_small_objects(400, seed=8)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs, max_prims_per_leaf=max_leaf, search_radius=radius)
    try:
        before = state(sc)
        t = {}
        sc.refit_rebuild_tlas(tris, max_leaf, radius, timings=t)
        after = state(sc)
        assert np.array_equal(after["nodes"], before["nodes"]) and np.array_equal(after["rec"], before["rec"])
        assert np.array_equal(after["blas"], before["blas"])
        assert after["info"]["n_nodes"] == before["info"]["n_nodes"] and after["info"]["tlas_start"] == before["info"]["tlas_start"]
        assert t["ms_refit_rebuild_tlas"] > 0
    finally:
        sc.close()


def _builder_sequences():
    t, offs, cases = _moved_cases()
    four = [(name, cases[name]) for name in ["jitter", "rigid", "point", "planar", "signed_zero", "huge", "jitter"]]
    return {"four_objects": (t, offs, four)} | {
        f"{n}_objects": (lambda tr, of: (tr, of, [("rigid", rigid(tr, of, 4)), ("rigid2", rigid(tr, of, 5))]))(*many_small_objects(n, seed=n))
        for n in (400, 3000)}


@gpu
@pytest.mark.parametrize("name", ["four_objects", "400_objects", "3000_objects"])
def test_moved_builder_scenes(name):
    """the BLAS part is a plain refit's, the TLAS and blas_offsets are tray_cuda_scene_build_tlas's and orc_build_ref's on the
    moved triangles (huge and back: the exact node test turns on, then off)"""
    tris, offs, steps = _builder_sequences()[name]
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    twin = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        pi = sc.download_bvh()[2]
        ts = sc.info()["tlas_start"]
        for what, moved in steps:
            sc.refit_rebuild_tlas(moved)
            twin.refit(moved)
            got = state(sc)
            assert got["info"]["tlas_start"] == ts
            assert np.array_equal(got["nodes"][:ts], twin.download_bvh(prim_indices=False)[0].reshape(-1, 80)[:ts]), what
            built = cuda.TrayCudaScene.build(moved, object_offsets=offs)
            try:
                want = state(built)
            finally:
                built.close()
            bts = want["info"]["tlas_start"]
            assert np.array_equal(got["nodes"][ts:], want["nodes"][bts:]), what
            assert np.array_equal(got["blas"], want["blas"]), what
            assert got["info"]["n_nodes"] - ts == want["info"]["n_nodes"] - bts, what
            r = ob.build_reference(moved, object_offsets=offs)
            rts = r["info"]["tlas_start"]
            assert np.array_equal(got["nodes"][ts:], r["nodes"].reshape(-1, 80)[rts:]) and np.array_equal(got["blas"], r["blas_offsets"]), what
            assert got["exact"] == expected_exact(got["nodes"]) == (what == "huge"), what
            rays = rays_at(moved, 3000, seed=4) if what == "huge" else random_rays(3000, seed=3)
            orc = ob.Oracle(got["nodes"], got["rec"], 48, got["blas"], ts, True)
            assert same_hits(sc.traverse(rays), orc.trace(rays, stack_limit=KERNEL_STACK)), what
        assert np.array_equal(pi, sc.download_bvh()[2])
    finally:
        sc.close()
        twin.close()


def _other_producer(kind):
    """(scene, twin, slot triangles, moved slot triangles) of a two-level scene no builder made"""
    if kind == "host_tlas":
        from conftest import load_golden_mesh
        m = load_golden_mesh("cornell_box")
        p = host.PackedScene(m, use_tlas=True)
        mesh_tris = m.tris().reshape(-1, 3, 3)
        moved = rigid(mesh_tris, m.object_offsets(), 6)[p.prim_to_mesh_tri]
        return cuda.TrayCudaScene.from_packed(p), cuda.TrayCudaScene.from_packed(p), mesh_tris[p.prim_to_mesh_tri], moved
    (nodes, blas, ts), rec, slots, moved = _other_producer_bytes(kind)
    make = lambda: cuda.TrayCudaScene(nodes, rec, 48, blas, ts)
    return make(), make(), slots, moved


def _other_producer_bytes(kind):
    """((nodes, blas, tlas_start), records, slot triangles, moved slot triangles) of generated tree `kind` with its TLAS at the tail"""
    seed = int(kind[-1])
    tris = cb.random_tris(700, seed)
    t, offs = cb.random_objects(tris, 7, seed)
    g = cb.random_tlas(t, offs, seed, exact_node=seed == 1)
    s = g.scene(t, 48, seed)
    slots = s.tris.reshape(-1, 3, 3)
    return tlas_at_the_tail(g), s.rec, slots, jitter(slots, seed + 2)


@gpu
@pytest.mark.parametrize("max_leaf", [3, 1])
@pytest.mark.parametrize("kind", ["host_tlas", "generated0", "generated1", "generated3"])
def test_moved_other_producers(kind, max_leaf):
    """host-producer and generated two-level trees (permuted blas_offsets, a BLAS under two instances, loose exponents, gaps):
    the BLAS part is refit_two_level's, the TLAS the reference's over the numpy root boxes; the node array grows"""
    sc, twin, slots, moved = _other_producer(kind)
    try:
        old = state(sc)
        ts, n_inst = old["info"]["tlas_start"], old["info"]["n_instances"]
        twin.refit(moved)                                  # the same topology walk, no growth
        sc.refit_rebuild_tlas(moved, max_prims_per_leaf=max_leaf)
        got = state(sc)
        want_nodes, want_blas = rebuild_reference(old["nodes"], moved, old["blas"], ts, max_leaf)
        assert np.array_equal(got["nodes"][:ts], refit_two_level(old["nodes"], moved, old["blas"], ts)[:ts])
        assert np.array_equal(got["nodes"], want_nodes) and np.array_equal(got["blas"], want_blas)
        assert got["info"]["n_nodes"] == len(want_nodes) and got["info"]["tlas_start"] == ts
        assert got["exact"] == expected_exact(got["nodes"])
        # a created scene holds exactly n_nodes: the array grows to tlas_start + n_instances + 1 nodes (80 B each), the topology's
        # per-node arrays with it (40 B each), and the TLAS build's scratch is kept (n_instances x 384 B + 16 MiB)
        cap = ts + n_inst + 1
        assert cap > old["info"]["n_nodes"]
        assert got["info"]["device_bytes"] - twin.info()["device_bytes"] == (cap - old["info"]["n_nodes"]) * 120 + n_inst * 384 + (16 << 20)
        rays = random_rays(3000, seed=5)
        orc = ob.Oracle(got["nodes"], got["rec"], 48, got["blas"], ts, True)
        assert same_hits(sc.traverse(rays), orc.trace(rays, stack_limit=KERNEL_STACK))
        # a second call grows nothing
        sc.refit_rebuild_tlas(jitter(slots, 9), max_prims_per_leaf=max_leaf)
        assert sc.info()["device_bytes"] == got["info"]["device_bytes"]
    finally:
        sc.close()
        twin.close()


def test_growth_case_adds_tlas_nodes():
    """a rebuild with one instance per leaf gives generated tree 0 more TLAS nodes than it had: test_moved_other_producers
    writes past the old end of its node array"""
    sc_nodes, _, slots, _ = _other_producer_bytes("generated0")
    nodes, blas, ts = sc_nodes
    want, _ = rebuild_reference(nodes, slots, blas, ts, max_leaf=1)
    assert len(want) > len(nodes)


@gpu
def test_rebuilt_scene_traces_like_a_fresh_scene_and_the_oracle(cornell):
    import torch
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets()
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    fresh = None
    try:
        ts = sc.info()["tlas_start"]
        moved = rigid(tris, offs, 5)
        sc.refit_rebuild_tlas(moved)
        blas = sc.download_instances()
        fresh, nodes, rec = fresh_like(sc, 48, blas, ts)
        orc = ob.Oracle(nodes, rec, 48, blas, ts, True)
        rays = random_rays(20000, seed=9)
        for any_hit in (False, True):
            a, b = sc.traverse(rays, any_hit=any_hit), fresh.traverse(rays, any_hit=any_hit)
            want, cnt, _ = orc.trace(rays, counts=True, any_hit=any_hit, stack_limit=KERNEL_STACK)
            assert same_hits(a, b) and same_hits(a, want), any_hit
            ha, ca = sc.traverse_cost(rays, any_hit=any_hit)
            hb, cbb = fresh.traverse_cost(rays, any_hit=any_hit)
            assert same_hits(ha, hb) and np.array_equal(ca, cbb), any_hit
            for k, o in (("nodes", "nodes"), ("tris", "tris"), ("instances", "insts")):
                assert np.array_equal(ca[k], cnt[o]), (any_hit, k)
            d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
            d_hits = torch.zeros(rays.size * 8, dtype=torch.uint8, device="cuda")
            sc.traverse_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr(), timed=True, any_hit=any_hit)
            assert same_hits(d_hits.cpu().numpy().view(ob.HIT_DTYPE), want), any_hit
        w, h = 256, 144
        view = host.view_from_camera(cornell.camera, w, h, ts)
        for overlap in (False, True):
            assert same_frame(frame(sc, view, w, h, overlap), frame(fresh, view, w, h, overlap)), overlap
        ref = orc.render(view, w, h, 0)
        got = frame(sc, view, w, h)
        assert all(same_hits(got[k], ref[k]) for k in ("primary", "bounce"))
    finally:
        sc.close()
        if fresh is not None:
            fresh.close()


@gpu
@pytest.mark.parametrize("in_flight", [1, 2, 3])
def test_frames_before_a_rebuild_keep_their_results(cornell, in_flight):
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets()
    w, h = 320, 184
    never = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    view = host.view_from_camera(cornell.camera, w, h, never.info()["tlas_start"])
    fresh = None
    try:
        want_a = frame(never, view, w, h, fc=3)
        sc.set_frames_in_flight(in_flight)
        sc.set_ray_cost(True)
        for fc in range(in_flight):
            sc.render(view, w, h, fc + 3 - (in_flight - 1), FLAGS, timed=False)
        rgba = np.zeros((h, w, 4), np.uint8)
        sc.readback_begin(rgba, 0)
        sc.refit_rebuild_tlas(rigid(tris, offs, 11, frac=0.2))
        sc.readback_wait(0)
        assert np.array_equal(rgba, want_a["rgba"])
        a = sc.download(primary=True, bounce=True, rgba=True)
        a["cost"] = sc.download_cost(primary=True, bounce=True)
        a["counters"] = sc.counters()
        assert same_frame(a, want_a), "a frame rendered before the rebuild changed"
        b = frame(sc, view, w, h, fc=3)
        fresh, _, _ = fresh_like(sc, 48, sc.download_instances(), sc.info()["tlas_start"])
        assert same_frame(b, frame(fresh, view, w, h, fc=3))
        assert not same_hits(b["primary"], want_a["primary"])
    finally:
        for s in (never, sc, fresh):
            if s is not None:
                s.close()


@gpu
def test_rebuild_device_waits_for_the_callers_stream():
    import torch
    tris, offs = many_small_objects(3000, seed=71)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        moved = rigid(tris, offs, 3)
        base = torch.from_numpy(tris.reshape(-1)).cuda()
        delta = torch.from_numpy((moved - tris).reshape(-1)).cuda()
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            m = torch.rand(2048, 2048, device="cuda")
            for _ in range(20):                       # keeps the stream busy, so the vertices below are written late
                m = torch.tanh(m @ m)
            d = base + delta + m[0, 0] * 0
        ms = sc.refit_rebuild_tlas_device(d.data_ptr(), tris.shape[0], stream=s.cuda_stream, timed=True)
        assert ms > 0
        got = state(sc)
        r = ob.build_reference(d.cpu().numpy().reshape(-1, 3, 3), object_offsets=offs)
        ts, rts = got["info"]["tlas_start"], r["info"]["tlas_start"]
        assert np.array_equal(got["nodes"][ts:], r["nodes"].reshape(-1, 80)[rts:]) and np.array_equal(got["blas"], r["blas_offsets"])
    finally:
        sc.close()


def _refusal_scene(kind):
    """(scene, triangles) for a refusal"""
    if kind == "flat":
        return cuda.TrayCudaScene.build(soup(500, 1)), soup(500, 1)
    if kind in ("past_tlas", "blas_range"):
        if kind == "past_tlas":                        # generated trees keep BLAS regions behind the TLAS
            tris = cb.random_tris(300, 2)
            t, offs = cb.random_objects(tris, 4, 2)
            g = cb.random_tlas(t, offs, 2)
            s = g.scene(t, 48, 2)
            return s.cuda(), s.tris.reshape(-1, 3, 3)
        from test_refit import _broken
        sc, tris, _ = _broken("blas_range")
        return sc, tris
    if kind == "empty_blas":                           # BLAS 1 is a node with no children
        tris = soup(4, seed=81)
        lo, hi = tris.min(axis=(0, 1)), tris.max(axis=(0, 1))
        nodes = np.stack([cb.encode_node(lo, hi, [(0, lo, hi, 2), (1, lo, hi, 2)], leaf_offsets=[0, 2]), cb.encode_node(lo, hi, []),
                          cb.encode_node(lo, hi, [(0, lo, hi, 1), (1, lo, hi, 1)], leaf_offsets=[0, 1])])
        return cuda.TrayCudaScene(nodes, host.tri_records(tris), 48, np.array([0, 1], np.uint32), 2), tris
    tris, offs = many_small_objects(200, seed=82)
    return cuda.TrayCudaScene.build(tris, object_offsets=offs), tris


@gpu
@pytest.mark.parametrize("kind", ["flat", "null", "count", "nan", "inf", "overflow", "max_leaf", "radius", "past_tlas", "empty_blas",
                                  "blas_range"])
def test_refusals_change_nothing(kind):
    L = cuda.lib()
    sc, tris = _refusal_scene(kind)
    try:
        if kind in ("nan", "inf", "overflow"):
            sc.refit_rebuild_tlas(jitter(tris, 1))     # the walk has run and the array has its room: a refusal after both
        elif kind in ("past_tlas", "empty_blas"):
            sc.refit(jitter(tris, 1))                  # a refit takes these trees; its walk is the one the rebuild refuses
        before = state(sc)
        bad = jitter(tris, 2).copy()
        args = {}
        if kind == "nan":
            bad[5, 1, 2] = np.nan
        elif kind == "inf":
            bad[-1, 0, 0] = -np.inf
        elif kind == "overflow":
            bad[0, 2, 1] = np.float32(3e38)
            bad[7, 1, 1] = np.float32(-3e38)
        elif kind == "count":
            bad = bad[:-1]
        elif kind == "max_leaf":
            args = dict(max_prims_per_leaf=4)
        elif kind == "radius":
            args = dict(search_radius=65)
        if kind == "null":
            assert L.tray_cuda_scene_refit_rebuild_tlas(sc._h, None, bad.shape[0], 3, 0, None) == -1
        else:
            with pytest.raises(cuda.TrayCudaError, match="error -1"):
                sc.refit_rebuild_tlas(bad, **args)
        after = state(sc)
        assert same_state(before, after)                 # device_bytes (info) included: no growth either
        if kind == "max_leaf":
            with pytest.raises(cuda.TrayCudaError, match="error -1"):
                sc.refit_rebuild_tlas(bad, max_prims_per_leaf=0)
        if kind not in ("flat", "past_tlas", "empty_blas", "blas_range"):
            sc.refit_rebuild_tlas(jitter(tris, 3))     # a valid call afterwards
            assert not same_state(before, state(sc))
    finally:
        sc.close()


@gpu
def test_refused_rebuilds_release_their_device_memory():
    """ten refused calls (a BLAS behind the TLAS, found by the walk) take no more free device memory than the buffers of one walk"""
    import torch
    tris = cb.random_tris(3000, 4)
    t, offs = cb.random_objects(tris, 40, 4)
    g = cb.random_tlas(t, offs, 4)
    s = g.scene(t, 48, 4)
    sc = s.cuda()
    try:
        moved = s.tris.reshape(-1, 3, 3)
        with pytest.raises(cuda.TrayCudaError, match="error -1"):
            sc.refit_rebuild_tlas(moved)               # the walk, kept with the scene as a refit keeps it
        torch.cuda.synchronize()
        free = torch.cuda.mem_get_info()[0]
        for _ in range(10):
            with pytest.raises(cuda.TrayCudaError, match="error -1"):
                sc.refit_rebuild_tlas(moved)
        assert free - torch.cuda.mem_get_info()[0] <= 0
    finally:
        sc.close()


@gpu
def test_refit_and_rebuild_alternate():
    """refit -> rebuild -> refit -> rebuild: every step's bytes are the reference's for its input, so the topology the scene
    keeps follows the new TLAS"""
    tris, offs = many_small_objects(1500, seed=90)
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        pi = sc.download_bvh()[2]
        ts = sc.info()["tlas_start"]
        for step in range(4):
            moved = rigid(tris, offs, 20 + step)
            before = state(sc)
            if step % 2 == 0:
                sc.refit(moved)
                want = refit_two_level(before["nodes"], moved[pi], before["blas"], ts)
                assert np.array_equal(state(sc)["nodes"], want), step
                assert np.array_equal(state(sc)["blas"], before["blas"]), step
            else:
                sc.refit_rebuild_tlas(moved)
                want, blas = rebuild_reference(before["nodes"], moved[pi], before["blas"], ts)
                got = state(sc)
                assert np.array_equal(got["nodes"], want) and np.array_equal(got["blas"], blas), step
                assert got["info"]["n_nodes"] == len(want), step
    finally:
        sc.close()


@gpu
def test_determinism_and_group_replicas():
    tris, offs = many_small_objects(2000, seed=91)
    moved = rigid(tris, offs, 7)
    a = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    b = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    try:
        a.refit_rebuild_tlas(moved)
        b.refit_rebuild_tlas(moved)
        assert same_state(state(a), state(b))
        a.refit_rebuild_tlas(moved)                    # the same input again: the same bytes
        assert same_state(state(a), state(b))
    finally:
        a.close()
        b.close()
    # a group made from the bytes of a two-level build: every replica rebuilt, byte-identical, and the frame of one GPU
    built = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    nodes, rec, pi = built.download_bvh()
    blas, ts = built.download_instances(), built.info()["tlas_start"]
    built.close()
    w, h = 640, 368
    view = host.view_from_camera(host.Camera((0.3, 0.4, 3.0), (0.0, 0.0, 0.0), 60.0), w, h, ts)
    one = cuda.TrayCudaScene(nodes, rec, 48, blas, ts)
    g = cuda.TrayCudaGroup(nodes, rec, 48, blas, ts, devices=list(range(min(cuda.device_count(), 8))))
    try:
        one.refit_rebuild_tlas(moved[pi])
        one.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        want = one.download(rgba=True)["rgba"].copy()
        g.set_frames_in_flight(2)
        g.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        for i in range(len(g.devices)):
            g.scene(i).refit_rebuild_tlas(moved[pi])
        ref = state(one)
        for i in range(len(g.devices)):
            assert same_state(state(g.scene(i)), ref), i
        for _ in range(2):
            g.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        assert (g.frame() == want).all()
        assert (want[..., :3] > 0).any()
    finally:
        g.close()
        one.close()
