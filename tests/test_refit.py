"""Refit (tray_cuda_scene_refit): the same tree re-encoded tight over moved triangles.

The bytes a refit must write are defined without the device: `refit_reference` walks the trees the way tree_walk does and
re-encodes p, the exponents and the q bytes of every used slot of every reachable node from the exact boxes of the new
triangles — the encoding test_build_reference.py's tightness check requires.  CPU tests hold the reference to that check and
to what it must leave alone; the `gpu` tests hold the device to the reference byte for byte, and the refit scene to a scene
created fresh from its bytes and to the oracle, hit for hit and counter for counter."""
import ctypes as C

import numpy as np
import pytest

import cwbvh_bytes as cb
import oracle_binding as ob
from conftest import random_rays
from test_build_reference import (decode, edge_geometry, from_ordered, many_small_objects, ordered, quant_exponent, rays_at, soup,
                                  tight_flat, tight_two_level, tightness_errors, tree_walk, tri_boxes)
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu

BIG, SMALL = np.int32(0x7FFFFFFF), np.int32(-0x7FFFFFFF - 1)


# ---- the reference ---------------------------------------------------------------------------------------------------------


def refit_reference(nodes, roots, slot_lo, slot_hi):
    """(new node bytes, (node min, node max) as ordered ints): every node reachable from `roots` (child = tree root +
    child_base_idx + rank) re-encoded over its exact box — p = the minimum, tight exponents, clamped floor / ceil q bytes of the
    slots with child_meta != 0 — with `slot_lo/hi[k]` the box of leaf entry k.  Nothing else changes; a node with no box under it
    keeps its bytes."""
    nb = np.array(nodes, dtype=np.uint8).reshape(-1, 80)
    f = decode(nb)
    n = nb.shape[0]
    level, child = tree_walk(f, roots)
    lo_o, hi_o = ordered(slot_lo), ordered(slot_hi)
    meta, imask = f["meta"], f["imask"]
    inner = ((imask[:, None] >> np.arange(8)) & 1) == 1
    leaf = (meta != 0) & ~inner
    cnt = np.select([meta >> 5 == 1, meta >> 5 == 3, meta >> 5 == 7], [1, 2, 3], 0)
    first = f["pbase"][:, None] + (meta & 31)
    slo = np.full((n, 8, 3), BIG, np.int32)
    shi = np.full((n, 8, 3), SMALL, np.int32)
    for k in range(3):
        use = leaf & (cnt > k) & (level >= 0)[:, None]           # unreached nodes may index another part's entries
        idx = np.where(use, first + k, 0)
        slo = np.where(use[..., None], np.minimum(slo, lo_o[idx]), slo)
        shi = np.where(use[..., None], np.maximum(shi, hi_o[idx]), shi)
    nlo = np.full((n, 3), BIG, np.int32)
    nhi = np.full((n, 3), SMALL, np.int32)
    for lv in range(int(level.max(initial=-1)), -1, -1):
        at = np.nonzero(level == lv)[0]
        has = child[at] >= 0
        cidx = np.where(has, child[at], 0)
        slo[at] = np.where(has[..., None], nlo[cidx], slo[at])
        shi[at] = np.where(has[..., None], nhi[cidx], shi[at])
        nlo[at] = slo[at].min(axis=1)
        nhi[at] = shi[at].max(axis=1)
    out = nb.copy()
    r = np.nonzero((level >= 0) & (nlo[:, 0] <= nhi[:, 0]))[0]
    mn, mx = from_ordered(nlo[r]), from_ordered(nhi[r])
    k = quant_exponent(mx - mn)
    out[r, 0:12] = np.ascontiguousarray(mn).view(np.uint8).reshape(-1, 12)
    out[r, 12:15] = (k + 127).astype(np.uint8)
    scale = np.ldexp(1.0, k)[:, :, None]
    p = mn.astype(np.float64)[:, :, None]
    with np.errstate(invalid="ignore", over="ignore"):
        ql = np.clip(np.floor((from_ordered(slo[r]).transpose(0, 2, 1).astype(np.float64) - p) / scale), 0, 255)
        qh = np.clip(np.ceil((from_ordered(shi[r]).transpose(0, 2, 1).astype(np.float64) - p) / scale), 0, 255)
    used = meta[r] != 0
    for a in range(3):
        for s in range(8):
            u = used[:, s]
            out[r[u], 32 + 16 * a + s] = ql[u, a, s].astype(np.uint8)
            out[r[u], 40 + 16 * a + s] = qh[u, a, s].astype(np.uint8)
    return out, (nlo, nhi)


def refit_two_level(nodes, slot_tris, blas, tlas_start):
    """every BLAS from its root (the distinct blas_offsets, anywhere in the node array), then the TLAS over the BLAS roots'
    exact boxes (TLAS leaf entry k = instance k)"""
    out, (nlo, nhi) = refit_reference(nodes, np.unique(blas), *tri_boxes(slot_tris))
    top, _ = refit_reference(out[tlas_start:], [0], from_ordered(nlo[blas]), from_ordered(nhi[blas]))
    out[tlas_start:] = top
    return out


def tight_two_level_anywhere(nodes, slot_tris, blas, tlas_start):
    """tight_two_level for BLAS trees on either side of the TLAS"""
    nb = np.asarray(nodes, np.uint8).reshape(-1, 80)
    errs, (nlo, nhi), _ = tightness_errors(nb, np.unique(blas), *tri_boxes(slot_tris))
    end = tlas_start + int(np.nonzero(tree_walk(decode(nb[tlas_start:]), [0])[0] >= 0)[0].max()) + 1     # the TLAS nodes only
    terrs, _, _ = tightness_errors(nb[tlas_start:end], [0], from_ordered(nlo[blas]), from_ordered(nhi[blas]))
    return errs + ["TLAS " + e for e in terrs]


def may_change(nodes, roots_parts):
    """(n, 80) mask of the bytes a refit may write: p, exponents and used q bytes of the nodes reachable in each (sub-array
    offset, roots) part"""
    nb = np.asarray(nodes, np.uint8).reshape(-1, 80)
    mask = np.zeros(nb.shape, bool)
    for off, roots in roots_parts:
        f = decode(nb[off:])
        level, _ = tree_walk(f, roots)
        for j in np.nonzero(level >= 0)[0]:
            mask[off + j, 0:15] = True
            for s in range(8):
                if f["meta"][j, s]:
                    mask[off + j, [32 + 16 * a + s for a in range(3)] + [40 + 16 * a + s for a in range(3)]] = True
    return mask


jitter, rigid = host.jitter, host.rigid


# ---- CPU: the reference on its own -----------------------------------------------------------------------------------------


def test_reference_on_a_reference_build_is_tight_and_touches_only_bounds():
    tris = soup(3000, seed=51)
    r = ob.build_reference(tris)
    slots = tris[r["prim_indices"]]
    same, _ = refit_reference(r["nodes"], [0], *tri_boxes(slots))
    assert np.array_equal(same, r["nodes"].reshape(-1, 80)), "a refit over the unmoved triangles is not the identity"
    moved = jitter(tris, 1)
    out, _ = refit_reference(r["nodes"], [0], *tri_boxes(moved[r["prim_indices"]]))
    assert not tight_flat(out, moved[r["prim_indices"]])
    old = r["nodes"].reshape(-1, 80)
    mask = may_change(old, [(0, [0])])
    assert np.array_equal(out[~mask], old[~mask])
    assert (out[mask] != old[mask]).any()


def test_reference_on_two_level_builds():
    tris, offs = many_small_objects(300, seed=5)
    r = ob.build_reference(tris, object_offsets=offs)
    ts, blas, pi = r["info"]["tlas_start"], r["blas_offsets"], r["prim_indices"]
    assert np.array_equal(refit_two_level(r["nodes"], tris[pi], blas, ts), r["nodes"].reshape(-1, 80))
    moved = rigid(tris, offs, 3)
    out = refit_two_level(r["nodes"], moved[pi], blas, ts)
    assert not tight_two_level(out, moved[pi], blas, ts)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_on_generated_trees(seed):
    """loose exponents, p below the minimum, random empty-slot bytes, gaps, poison nodes: the refit makes every reachable node
    tight and leaves every other byte, the unreachable poison nodes whole"""
    tris = cb.random_tris(400, seed)
    g = cb.random_cwbvh(tris, seed, exact_node=seed == 1)
    rec = g.scene(tris, 48, seed).tris.reshape(-1, 3, 3)
    moved = jitter(rec, seed + 7)
    out, _ = refit_reference(g.nodes, [0], *tri_boxes(moved))
    assert not tightness_errors(out, [0], *tri_boxes(moved))[0]
    mask = may_change(g.nodes, [(0, [0])])
    assert np.array_equal(out[~mask], g.nodes[~mask])
    unreached = tree_walk(decode(g.nodes), [0])[0] < 0
    assert np.array_equal(out[unreached], g.nodes[unreached])


@pytest.mark.parametrize("seed", [0, 3])
def test_reference_on_generated_two_level_trees(seed):
    tris = cb.random_tris(500, seed)
    t, offs = cb.random_objects(tris, 6, seed)
    g = cb.random_tlas(t, offs, seed)
    rec = g.scene(t, 48, seed).tris.reshape(-1, 3, 3)
    moved = jitter(rec, seed + 1)
    out = refit_two_level(g.nodes, moved, g.blas, g.tlas_start)
    assert not tight_two_level_anywhere(out, moved, g.blas, g.tlas_start)
    mask = may_change(g.nodes, [(0, np.unique(g.blas)), (g.tlas_start, [0])])
    assert np.array_equal(out[~mask], g.nodes[~mask])


def test_refit_arguments_without_a_device():
    """NULL scene or triangles are refused before any device is touched; without a device there is no scene to refit"""
    L = cuda.lib()
    t = np.zeros(9, np.float32)
    ms = C.c_float()
    assert L.tray_cuda_scene_refit(None, t.ctypes.data, 1, C.byref(ms)) == -1
    assert L.tray_cuda_scene_refit_device(None, t.ctypes.data, 1, None, None) == -1
    assert L.tray_cuda_scene_refit(None, None, 0, None) == -1
    if cuda.device_count() == 0:
        with pytest.raises(cuda.TrayCudaError, match="no CUDA device"):
            cuda.TrayCudaScene.build(soup(10, 1))


# ---- GPU -------------------------------------------------------------------------------------------------------------------


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def records(stride, tris):
    return host.tri_records(tris, stride).reshape(-1)


def check_against_reference(sc, slot_tris, blas=None, tlas_start=0, validate=True):
    """device node bytes == the reference's, records == the records of the slot triangles; flat trees pass the validator"""
    i = sc.info()
    old = getattr(sc, "_nodes_before")
    nodes, rec, _ = sc.download_bvh(prim_indices=False)
    if blas is None:
        want, _ = refit_reference(old, [0], *tri_boxes(slot_tris))
    else:
        want = refit_two_level(old, slot_tris, blas, tlas_start)
    nodes = nodes.reshape(-1, 80)
    assert np.array_equal(nodes, want), f"{int((nodes != want).any(axis=1).sum())} nodes differ from the reference"
    assert np.array_equal(rec, records(i["tri_stride"], slot_tris)), "triangle records differ"
    if validate and blas is None:
        rc, rep = host.validate_cwbvh(nodes, np.arange(len(slot_tris), dtype=np.uint32), slot_tris.min(axis=1), slot_tris.max(axis=1),
                                      stack_limit=48)
        assert rc == 0, rep
    return nodes, rec


def snapshot(sc):
    sc._nodes_before = sc.download_bvh(prim_indices=False)[0].reshape(-1, 80).copy()
    return sc


def fresh_like(sc, stride, blas=None, tlas_start=0):
    nodes, rec, _ = sc.download_bvh(prim_indices=False)
    return cuda.TrayCudaScene(nodes, rec, stride, blas, tlas_start), nodes, rec


def same_hits(a, b):
    return np.array_equal(a["prim"], b["prim"]) and np.array_equal(bits(a["t"]), bits(b["t"]))


@gpu
@pytest.mark.parametrize("stride,max_leaf", [(24, 1), (48, 2), (64, 3), (48, 3), (24, 3), (64, 1)])
def test_identity_device_built_flat(stride, max_leaf):
    tris = soup(5000, seed=stride + max_leaf)
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, max_prims_per_leaf=max_leaf)
    try:
        nodes, rec, _ = sc.download_bvh()
        before = sc.info()["device_bytes"]
        t = {}
        sc.refit(tris, timings=t)
        n2, r2, _ = sc.download_bvh()
        assert np.array_equal(n2, nodes) and np.array_equal(r2, rec)
        assert t["ms_refit"] > 0 and sc.info()["device_bytes"] > before
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("name", [c[0] for c in edge_geometry()] + ["two_level", "host_flat", "host_tlas"])
def test_identity(cornell, name):
    if name.startswith("host"):
        p = host.PackedScene(cornell, use_tlas=name == "host_tlas")
        sc = cuda.TrayCudaScene.from_packed(p)
        tris = cornell.tris().reshape(-1, 3, 3)[p.prim_to_mesh_tri]
    elif name == "two_level":
        tris, offs = many_small_objects(400, seed=8)
        sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    else:
        tris = dict(edge_geometry())[name]
        sc = cuda.TrayCudaScene.build(tris)
    try:
        nodes, rec, _ = sc.download_bvh(prim_indices=False)
        exact = sc.exact_node_test()
        assert exact == (name == "huge")
        sc.refit(tris)
        n2, r2, _ = sc.download_bvh(prim_indices=False)
        assert np.array_equal(n2, nodes), "nodes changed"
        assert np.array_equal(r2, rec), "records changed"
        assert sc.exact_node_test() == exact
    finally:
        sc.close()


def _moved_cases():
    t = soup(4000, seed=61)
    offs = np.array([0, 900, 1000, 2500, 4000], np.uint64)
    point = t.copy(); point[900:1000] = np.float32(0.3)                             # an object collapsed to a point
    planar = t.copy(); planar[1000:2500, :, 1] = np.float32(-0.2)                   # a planar object
    sz = np.abs(t.copy()); z = np.random.default_rng(2).random(sz.shape) < 0.3
    sz[z] = np.where(np.random.default_rng(3).random(int(z.sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    return t, offs, dict(jitter=jitter(t, 1), rigid=rigid(t, offs, 2), point=point, planar=planar, signed_zero=sz,
                         huge=(t * np.float32(1e15)).astype(np.float32))


@gpu
@pytest.mark.parametrize("two_level", [False, True])
def test_moved_device_built_equal_reference(two_level):
    t, offs, cases = _moved_cases()
    sc = cuda.TrayCudaScene.build(t, object_offsets=offs if two_level else None)
    try:
        pi = sc.download_bvh()[2]
        blas, ts = (sc.download_instances(), sc.info()["tlas_start"]) if two_level else (None, 0)
        rays = random_rays(4000, seed=3)
        for name in ["jitter", "rigid", "point", "planar", "signed_zero", "huge", "jitter"]:      # huge and back: force_exact on, off
            moved = cases[name]
            snapshot(sc).refit(moved)
            nodes, _ = check_against_reference(sc, moved[pi], blas, ts)
            e = nodes[:, 12:15]
            assert bool((e >= 167).any()) == (name == "huge"), name
            assert sc.exact_node_test() == (name == "huge"), name            # on with the scale, and off again
            fresh = cuda.TrayCudaScene(*sc.download_bvh(prim_indices=False)[:2], 48, blas, ts)
            try:
                assert fresh.exact_node_test() == sc.exact_node_test(), name
            finally:
                fresh.close()
            r = rays_at(moved, 3000, seed=4) if name == "huge" else rays
            orc = ob.Oracle(*sc.download_bvh(prim_indices=False)[:2], 48, blas, ts, two_level)
            assert same_hits(sc.traverse(r), orc.trace(r, stack_limit=48)), name
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("stride", [48, 24])
def test_moved_generated_trees(seed, stride):
    tris = cb.random_tris(600, seed)
    g = cb.random_cwbvh(tris, seed, exact_node=seed == 1)
    s = g.scene(tris, stride, seed)
    sc = snapshot(s.cuda())
    try:
        moved = jitter(s.tris, seed + 5)
        sc.refit(moved)
        nodes, _ = check_against_reference(sc, moved, validate=False)
        unreached = tree_walk(decode(g.nodes), [0])[0] < 0
        assert np.array_equal(nodes[unreached], g.nodes[unreached]), "an unreachable node changed"
        rays = random_rays(3000, seed)
        orc = ob.Oracle(nodes, records(stride, moved), stride)
        assert same_hits(sc.traverse(rays), orc.trace(rays, stack_limit=48))
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("seed", [0, 3])
def test_moved_generated_two_level_trees(seed):
    tris = cb.random_tris(700, seed)
    t, offs = cb.random_objects(tris, 7, seed)
    g = cb.random_tlas(t, offs, seed)
    s = g.scene(t, 48, seed)
    sc = snapshot(s.cuda())
    try:
        moved = jitter(s.tris, seed + 2)
        sc.refit(moved)
        nodes, _ = check_against_reference(sc, moved, g.blas, g.tlas_start)
        assert not tight_two_level_anywhere(nodes, moved, g.blas, g.tlas_start)
        rays = random_rays(3000, seed)
        orc = ob.Oracle(nodes, records(48, moved), 48, g.blas, g.tlas_start, True)
        assert same_hits(sc.traverse(rays), orc.trace(rays, stack_limit=48))
    finally:
        sc.close()


FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_COUNTERS


def frame(sc, view, w, h, overlap=False, fc=0):
    sc.set_ray_cost(True)
    sc.render(view, w, h, fc, FLAGS | (cuda.RENDER_OVERLAP if overlap else 0))
    sc.sync()
    out = sc.download(primary=True, bounce=True, rgba=True)
    out["cost"] = sc.download_cost(primary=True, bounce=True)
    out["counters"] = sc.counters()
    return out


def same_frame(a, b):
    return (all(same_hits(a[k], b[k]) for k in ("primary", "bounce")) and np.array_equal(a["rgba"], b["rgba"])
            and all(np.array_equal(a["cost"][k], b["cost"][k]) for k in ("primary", "bounce")) and a["counters"] == b["counters"])


@gpu
@pytest.mark.parametrize("use_tlas", [False, True])
def test_refit_traces_like_a_fresh_scene_and_the_oracle(cornell, use_tlas):
    import torch
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets() if use_tlas else None
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    fresh = None
    try:
        pi = sc.download_bvh()[2]
        blas, ts = (sc.download_instances(), sc.info()["tlas_start"]) if use_tlas else (None, 0)
        moved = rigid(tris, offs, 5) if use_tlas else jitter(tris, 5, frac=0.05)
        sc.refit(moved)
        fresh, nodes, rec = fresh_like(sc, 48, blas, ts)
        orc = ob.Oracle(nodes, rec, 48, blas, ts, use_tlas)
        rays = random_rays(20000, seed=9)
        for any_hit in (False, True):
            a, b, c = sc.traverse(rays, any_hit=any_hit), fresh.traverse(rays, any_hit=any_hit), orc.trace(rays, any_hit=any_hit, stack_limit=48)
            assert same_hits(a, b) and np.array_equal(a["prim"], c["prim"]), any_hit
            if not any_hit:
                assert same_hits(a, c)
            ha, ca = sc.traverse_cost(rays, any_hit=any_hit)
            hb, cbb = fresh.traverse_cost(rays, any_hit=any_hit)
            assert same_hits(ha, hb) and np.array_equal(ca, cbb), any_hit
        # device entry points
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_hits = torch.zeros(rays.size * 8, dtype=torch.uint8, device="cuda")
        sc.traverse_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr(), timed=True)
        got = d_hits.cpu().numpy().view(ob.HIT_DTYPE)
        assert same_hits(got, orc.trace(rays, stack_limit=48))
        # closest hits agree with an exhaustive search over the moved triangles
        brute, _ = orc.brute_force(rays)
        hit = brute["prim"] != ob.INVALID_PRIM
        assert np.array_equal(hit, a["prim"] != ob.INVALID_PRIM) and hit.sum() > 500
        a = sc.traverse(rays)
        assert (np.abs(a["t"][hit] - brute["t"][hit]) <= 1e-5 * np.abs(brute["t"][hit])).all()
        # both frame paths
        w, h = 256, 144
        view = host.view_from_camera(cornell.camera, w, h)
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
def test_frames_before_a_refit_keep_their_results(cornell, in_flight):
    p = host.PackedScene(cornell)
    tris = cornell.tris().reshape(-1, 3, 3)[p.prim_to_mesh_tri]
    w, h = 320, 184
    view = host.view_from_camera(cornell.camera, w, h)
    never = cuda.TrayCudaScene.from_packed(p)
    sc = cuda.TrayCudaScene.from_packed(p)
    fresh = None
    try:
        want_a = frame(never, view, w, h, fc=3)
        sc.set_frames_in_flight(in_flight)
        sc.set_ray_cost(True)
        for fc in range(in_flight):
            sc.render(view, w, h, fc + 3 - (in_flight - 1), FLAGS, timed=False)
        rgba = np.zeros((h, w, 4), np.uint8)
        sc.readback_begin(rgba, 0)
        sc.refit(jitter(tris, 11, frac=0.2))
        sc.readback_wait(0)
        assert np.array_equal(rgba, want_a["rgba"])
        a = sc.download(primary=True, bounce=True, rgba=True)
        a["cost"] = sc.download_cost(primary=True, bounce=True)
        a["counters"] = sc.counters()
        assert same_frame(a, want_a), "a frame rendered before the refit changed"
        b = frame(sc, view, w, h, fc=3)
        fresh, _, _ = fresh_like(sc, 48)
        assert same_frame(b, frame(fresh, view, w, h, fc=3))
        assert not same_hits(b["primary"], want_a["primary"])
    finally:
        for s in (never, sc, fresh):
            if s is not None:
                s.close()


@gpu
def test_refit_device_waits_for_the_callers_stream():
    import torch
    tris = soup(200000, seed=71)
    sc = snapshot(cuda.TrayCudaScene.build(tris))
    try:
        pi = sc.download_bvh()[2]
        moved = jitter(tris, 3, frac=0.5)
        base = torch.from_numpy(tris.reshape(-1)).cuda()
        delta = torch.from_numpy((moved - tris).reshape(-1)).cuda()
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            m = torch.rand(2048, 2048, device="cuda")
            for _ in range(20):                       # keeps the stream busy, so the vertices below are written late
                m = torch.tanh(m @ m)
            d = base + delta + m[0, 0] * 0
        ms = sc.refit_device(d.data_ptr(), tris.shape[0], stream=s.cuda_stream, timed=True)
        assert ms > 0
        check_against_reference(sc, d.cpu().numpy().reshape(-1, 3, 3)[pi])
    finally:
        sc.close()


def _broken(kind):
    """(scene, tris) of a tree the walk must refuse; leaves cover triangles 0 .. 3"""
    tris = soup(4, seed=81)
    lo, hi = tris.min(axis=(0, 1)), tris.max(axis=(0, 1))
    leaf = lambda base: cb.encode_node(lo, hi, [(0, lo, hi, 2), (1, lo, hi, 2)], prim_base=base, leaf_offsets=[0, 2])
    blas = None
    if kind == "twice":          # node 1's child block is node 2, which the root also reaches
        nodes = [cb.encode_node(lo, hi, [(0, lo, hi, "inner"), (1, lo, hi, "inner")], child_base=1),
                 cb.encode_node(lo, hi, [(0, lo, hi, "inner")], child_base=2), leaf(0)]
    elif kind == "child_range":
        nodes = [cb.encode_node(lo, hi, [(0, lo, hi, "inner")], child_base=5), leaf(0)]
    elif kind == "leaf_range":
        nodes = [leaf(2)]
    elif kind == "blas_range":   # a blas_offsets entry outside the node array
        nodes = [leaf(0), cb.encode_node(lo, hi, [(0, lo, hi, 1), (1, lo, hi, 1)], leaf_offsets=[0, 1])]
        blas = np.array([0, 7], np.uint32)
    else:                        # a blas_offsets entry names tlas_start: every node is reachable, and the TLAS root twice
        nodes = [leaf(0), cb.encode_node(lo, hi, [(0, lo, hi, 1), (1, lo, hi, 1)], leaf_offsets=[0, 1])]
        blas = np.array([0, 1], np.uint32)
    nodes = np.stack(nodes)
    return cuda.TrayCudaScene(nodes, host.tri_records(tris), 48, blas, 1 if blas is not None else 0), tris, nodes


@gpu
@pytest.mark.parametrize("kind", ["nan", "inf", "overflow", "count", "null", "twice", "child_range", "leaf_range", "blas_range", "blas_tlas"])
def test_refusals_change_nothing(cornell, kind):
    L = cuda.lib()
    if kind in ("twice", "child_range", "leaf_range", "blas_range", "blas_tlas"):
        sc, tris, _ = _broken(kind)
        traced = kind == "twice"              # the others point outside their arrays: not traced
    else:
        p = host.PackedScene(cornell)
        sc = cuda.TrayCudaScene.from_packed(p)
        tris = cornell.tris().reshape(-1, 3, 3)[p.prim_to_mesh_tri]
        sc.refit(jitter(tris, 1))              # the walk has run: a refusal after it
        traced = True
    try:
        nodes, rec, _ = sc.download_bvh(prim_indices=False)
        rays = random_rays(2000, seed=1)
        before = sc.traverse(rays) if traced else None
        bad = jitter(tris, 2).copy()
        if kind == "nan":
            bad[5, 1, 2] = np.nan
        elif kind == "inf":
            bad[-1, 0, 0] = -np.inf
        elif kind == "overflow":                   # finite, but max - min on y is +inf: no box over them can be encoded
            bad[0, 2, 1] = np.float32(3e38)
            bad[7, 1, 1] = np.float32(-3e38)
        elif kind == "count":
            bad = bad[:-1]
        if kind == "null":
            assert L.tray_cuda_scene_refit(sc._h, None, bad.shape[0], None) == -1
        else:
            with pytest.raises(cuda.TrayCudaError, match="error -1"):
                sc.refit(bad)
        n2, r2, _ = sc.download_bvh(prim_indices=False)
        assert np.array_equal(n2, nodes) and np.array_equal(r2, rec)
        if traced:
            assert same_hits(sc.traverse(rays), before)
    finally:
        sc.close()


@gpu
def test_refused_walks_release_their_device_memory():
    """A topology walk that refuses a tree frees what it allocated: ten refusals of a builder tree of 200k triangles in which a
    node is reached twice take no more free device memory than the buffers of one walk."""
    import torch
    tris = soup(200000, seed=83)
    built = cuda.TrayCudaScene.build(tris)
    nodes, rec, _ = built.download_bvh(prim_indices=False)
    built.close()
    nodes = nodes.reshape(-1, 80).copy()
    assert nodes[1, 15] != 0                      # node 1 (a child of the root) has inner children
    nodes[1, 16:20] = 0                           # ... whose block now starts at node 0: the root is reached twice
    n_nodes, n_tris = nodes.shape[0], tris.shape[0]
    # one walk's buffers: per node its entry (8 B), its box (32 B) and its visited word (4 B); per triangle slot a box (32 B); the
    # flag and check words (28 B) and the walk's tail / error words (8 B); each rounded up to the 2 MiB pages device memory is mapped in
    page = 2 << 20
    walk_bytes = sum(-(-b // page) * page for b in (n_nodes * 8, n_nodes * 32, n_nodes * 4, n_tris * 32, 28, 8))
    sc = cuda.TrayCudaScene(nodes, rec, 48)
    try:
        with pytest.raises(cuda.TrayCudaError, match="error -1"):
            sc.refit(tris)                        # loads the walk's kernels before anything is measured
        torch.cuda.synchronize()
        free = torch.cuda.mem_get_info()[0]
        for _ in range(10):
            with pytest.raises(cuda.TrayCudaError, match="error -1"):
                sc.refit(tris)
        assert free - torch.cuda.mem_get_info()[0] <= walk_bytes
    finally:
        sc.close()


@gpu
def test_large_coordinates_refit_while_every_extent_is_finite(cornell):
    """a coordinate near the top of the f32 range is taken as long as the extent on its axis stays finite"""
    p = host.PackedScene(cornell)
    sc = snapshot(cuda.TrayCudaScene.from_packed(p))
    try:
        moved = jitter(cornell.tris().reshape(-1, 3, 3)[p.prim_to_mesh_tri], 1).copy()
        moved[3, 1, 0] = np.float32(3e38)
        sc.refit(moved)
        check_against_reference(sc, moved)
        assert sc.exact_node_test()
    finally:
        sc.close()


@gpu
def test_empty_scene_refit_does_nothing():
    sc = cuda.TrayCudaScene(np.zeros(0, np.uint8), np.zeros(0, np.uint8))
    try:
        sc.refit(np.zeros((0, 9), np.float32))
        with pytest.raises(cuda.TrayCudaError):
            sc.refit(np.zeros((1, 9), np.float32))
    finally:
        sc.close()


@gpu
def test_group_replicas_refit():
    m = host.Mesh.generate("kitchen", 1, 1.0)
    p = host.PackedScene(m)
    tris = m.tris().reshape(-1, 3, 3)[p.prim_to_mesh_tri]
    moved = jitter(tris, 4, frac=0.1)
    w, h = 640, 368
    view = host.view_from_camera(m.camera, w, h)
    one = cuda.TrayCudaScene.from_packed(p)
    g = cuda.TrayCudaGroup.from_packed(p, devices=list(range(min(cuda.device_count(), 8))))
    try:
        one.refit(moved)
        one.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        want = one.download(rgba=True)["rgba"].copy()
        g.set_frames_in_flight(2)
        g.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        for i in range(len(g.devices)):
            g.scene(i).refit(moved)
        for _ in range(2):
            g.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        assert (g.frame() == want).all()
    finally:
        g.close()
        one.close()
