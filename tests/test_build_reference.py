"""The device CWBVH builder (build_gpu.cu) held to a serial reference of the same rules (oracle/build_ref.c), byte for byte.

The other builder tests check that a device-built tree is valid and traces like the oracle; a builder that is wrong but still
valid (a PLOC tie broken the other way, a reinsertion that stops moving subtrees, a box one quantisation step loose) passes
them.  Here the device bytes must equal the reference's: nodes, prim_indices, triangle records, blas_offsets, tlas_start and
the build statistics.  A check that depends on no builder recomputes every node's exact box from its primitives and requires
each node and child box to be tight: reference trees, device trees and host-producer trees pass it.

CPU tests (unmarked) check the reference itself; the `gpu` tests compare it with the device."""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import load_golden_mesh, random_rays
from tray_racing_b200 import host

gpu = pytest.mark.gpu

# ---- scenes --------------------------------------------------------------------------------------------------------------


def soup(n, seed=0, spread=1.0, size=0.05):
    """n small random triangles in [-spread, spread]^3"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-spread, spread, size=(n, 1, 3)).astype(np.float32)
    return np.ascontiguousarray(c + rng.uniform(-size * spread, size * spread, size=(n, 3, 3)).astype(np.float32))


ONE = np.array([[[0, 0, 0], [1, 0, 0], [0, 1, 0]]], dtype=np.float32)


def signed_zero_soup(n=600, seed=11):
    """triangles in [0, 1]^3 with a third of the coordinates exactly +0.0 or -0.0: node minima land on zeros of both signs"""
    rng = np.random.default_rng(seed)
    t = soup(n, seed, 0.5, 0.2) + np.float32(0.5)
    t = np.abs(t)
    z = rng.random(t.shape) < 0.33
    t[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    return t


def edge_geometry():
    """(name, triangles) of the shapes where a builder's rules are easiest to get wrong"""
    degenerate = np.concatenate([ONE, np.zeros((1, 3, 3), np.float32), ONE + 1, np.array([[[2, 2, 2], [3, 3, 3], [4, 4, 4]]], np.float32)])
    planar = soup(500, 5)
    planar[:, :, 2] = 0.25                                      # ext == 0 on z: every Morton z is 0, every node's z extent hits 1e-20
    return [("coincident37", np.repeat(ONE, 37, axis=0)),       # equal Morton keys, equal merged areas: every tie
            ("degenerate", degenerate),                         # zero-area triangle, a line
            ("planar", planar),
            ("signed_zero", signed_zero_soup()),
            ("huge", soup(400, 7, 1e15, 5e-5))]                 # node extent > 255 * 2^39: exponent byte >= 167, force_exact


def many_small_objects(n_obj=1500, seed=13):
    """a soup split into n_obj objects of 1-4 triangles: the TLAS PLOC starts above the 1024-cluster tail"""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(1, 5, size=n_obj)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    centres = rng.uniform(-1, 1, size=(n_obj, 1, 1, 3)).astype(np.float32)
    tris = [centres[k] + rng.uniform(-0.02, 0.02, size=(int(sizes[k]), 3, 3)).astype(np.float32) for k in range(n_obj)]
    return np.ascontiguousarray(np.concatenate(tris)), offs


def rays_at(tris, n, seed):
    """rays from far outside towards random triangles' centroids, at any scale of the scene"""
    rng = np.random.default_rng(seed)
    t = np.asarray(tris, np.float64).reshape(-1, 3, 3)
    c = t[rng.integers(0, t.shape[0], size=n)].mean(axis=1)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.zeros(n, dtype=ob.RAY_DTYPE)
    rays["o"] = (c - d * 2 * np.abs(t).max()).astype(np.float32)
    rays["d"] = d.astype(np.float32)
    rays["tmax"] = np.float32(3.402823466e+38)
    return rays


# ---- decoding CWBVH nodes ------------------------------------------------------------------------------------------------


def ordered(f):
    """float32 -> int32 whose order is the float order with -0.0 below +0.0 (the device's min / max rule); an involution"""
    i = np.ascontiguousarray(f, dtype=np.float32).view(np.int32)
    return np.where(i >= 0, i, i ^ np.int32(0x7FFFFFFF))


def from_ordered(o):
    o = np.asarray(o, dtype=np.int32)
    return np.where(o >= 0, o, o ^ np.int32(0x7FFFFFFF)).astype(np.int32).view(np.float32)


def tri_boxes(t):
    """per triangle min / max corner under the same order (numpy's min / max do not order -0.0 below +0.0)"""
    o = ordered(np.asarray(t, np.float32).reshape(-1, 3, 3))
    return from_ordered(o.min(axis=1)), from_ordered(o.max(axis=1))


def decode(nodes):
    n = np.ascontiguousarray(nodes, dtype=np.uint8).reshape(-1, 80)
    return dict(p=n[:, 0:12].copy().view(np.float32), e=n[:, 12:15].astype(np.int32), imask=n[:, 15].astype(np.int64),
                cbase=n[:, 16:20].copy().view(np.uint32)[:, 0].astype(np.int64), pbase=n[:, 20:24].copy().view(np.uint32)[:, 0].astype(np.int64),
                meta=n[:, 24:32].astype(np.int64), qlo=np.stack([n[:, 32 + 16 * a:40 + 16 * a] for a in range(3)], 1).astype(np.int64),
                qhi=np.stack([n[:, 40 + 16 * a:48 + 16 * a] for a in range(3)], 1).astype(np.int64))


def quant_exponent(extent):
    """smallest k with 255 * 2^k >= extent (extent at least 1e-20), per element"""
    ext = np.maximum(np.asarray(extent, dtype=np.float32), np.float32(1e-20)).astype(np.float64)
    k = np.ceil(np.log2(ext / 255.0)).astype(np.int64)
    for _ in range(4):
        k = np.where(np.ldexp(255.0, k) < ext, k + 1, k)
    for _ in range(4):
        k = np.where(np.ldexp(255.0, k - 1) >= ext, k - 1, k)
    return k


def tree_walk(f, roots):
    """BFS levels and inner-child node indices of the trees below `roots`; a child's index is its tree root's index +
    child_base_idx + rank (flat trees have the one root 0)"""
    n = f["imask"].shape[0]
    level = np.full(n, -1, np.int64)
    base = np.full(n, -1, np.int64)
    child = np.full((n, 8), -1, np.int64)
    front = np.asarray(roots, np.int64)
    level[front] = 0
    base[front] = front
    lv = 0
    while front.size:
        bits = (f["imask"][front][:, None] >> np.arange(8)) & 1
        rank = np.cumsum(bits, axis=1) - bits
        ci = base[front][:, None] + f["cbase"][front][:, None] + rank
        child[front] = np.where(bits == 1, ci, -1)
        nxt = ci[bits == 1]
        assert ((nxt >= 0) & (nxt < n)).all(), "child index outside the node array"
        assert (level[nxt] == -1).all(), "a node is reached twice"
        lv += 1
        level[nxt] = lv
        base[nxt] = np.repeat(base[front], bits.sum(axis=1))
        front = nxt
    return level, child


def tightness_errors(nodes, roots, slot_lo, slot_hi, limit=5):
    """Recompute the exact union box under every node and every child slot from the primitive boxes (`slot_lo/hi[k]`: box of
    primitive slot k) and require the tight encoding: p = the union minimum bit for bit, e - 127 = quant_exponent(max - min)
    per axis, and every qlo / qhi = the clamped floor / ceil of (child bound - p) / 2^(e - 127).  Returns (messages, node
    boxes as ordered ints, levels)."""
    f = decode(nodes)
    n = f["imask"].shape[0]
    level, child = tree_walk(f, roots)
    lo_o, hi_o = ordered(slot_lo), ordered(slot_hi)
    big, small = np.int32(0x7FFFFFFF), np.int32(-0x7FFFFFFF - 1)
    meta, imask = f["meta"], f["imask"]
    inner = ((imask[:, None] >> np.arange(8)) & 1) == 1
    leaf = (meta != 0) & ~inner
    cnt = np.select([meta >> 5 == 1, meta >> 5 == 3, meta >> 5 == 7], [1, 2, 3], 0)
    first = f["pbase"][:, None] + (meta & 31)
    slo = np.full((n, 8, 3), big, np.int32)
    shi = np.full((n, 8, 3), small, np.int32)
    for k in range(3):
        use = leaf & (cnt > k)
        idx = np.where(use, first + k, 0)
        slo = np.where(use[..., None], np.minimum(slo, lo_o[idx]), slo)
        shi = np.where(use[..., None], np.maximum(shi, hi_o[idx]), shi)
    nlo = np.full((n, 3), big, np.int32)
    nhi = np.full((n, 3), small, np.int32)
    for lv in range(int(level.max()), -1, -1):
        at = np.nonzero(level == lv)[0]
        ch = child[at]
        has = ch >= 0
        cidx = np.where(has, ch, 0)
        slo[at] = np.where(has[..., None], nlo[cidx], slo[at])
        shi[at] = np.where(has[..., None], nhi[cidx], shi[at])
        nlo[at] = slo[at].min(axis=1)
        nhi[at] = shi[at].max(axis=1)
    errs = []
    reached = np.nonzero(level >= 0)[0]
    bad_p = reached[(ordered(f["p"][reached]) != nlo[reached]).any(axis=1)]
    errs += [f"node {i}: p {f['p'][i].tolist()} is not the union minimum {from_ordered(nlo[i]).tolist()}" for i in bad_p[:limit]]
    mn, mx = from_ordered(nlo[reached]), from_ordered(nhi[reached])
    k = quant_exponent(mx - mn)
    bad_e = reached[(f["e"][reached] - 127 != k).any(axis=1)]
    errs += [f"node {i}: exponents {(f['e'][i] - 127).tolist()}, tight ones {k[np.searchsorted(reached, i)].tolist()}" for i in bad_e[:limit]]
    scale = np.ldexp(1.0, k)[:, :, None]
    p = f["p"][reached].astype(np.float64)[:, :, None]
    used = (meta[reached] != 0)[:, None, :]
    cl = from_ordered(slo[reached]).transpose(0, 2, 1).astype(np.float64)
    chh = from_ordered(shi[reached]).transpose(0, 2, 1).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        ql = np.clip(np.floor((cl - p) / scale), 0, 255)
        qh = np.clip(np.ceil((chh - p) / scale), 0, 255)
    bad_q = used & ((f["qlo"][reached] != ql) | (f["qhi"][reached] != qh))
    for i, a, s in list(zip(*np.nonzero(bad_q)))[:limit]:
        j = reached[i]
        errs.append(f"node {j} slot {s} axis {a}: q [{f['qlo'][j, a, s]}, {f['qhi'][j, a, s]}], tight [{int(ql[i, a, s])}, {int(qh[i, a, s])}]")
    return errs, (nlo, nhi), level


def tight_flat(nodes, prim_slots_tris):
    """tightness of a flat tree whose primitive slot k holds triangle prim_slots_tris[k]"""
    return tightness_errors(nodes, [0], *tri_boxes(prim_slots_tris))[0]


def tight_two_level(nodes, prim_slots_tris, blas_offsets, tlas_start):
    """BLAS trees (roots: the blas_offsets, child indices relative to the root) and then the TLAS over their exact boxes"""
    roots = np.unique(blas_offsets)
    nb = np.asarray(nodes, np.uint8).reshape(-1, 80)
    errs, (nlo, nhi), _ = tightness_errors(nb[:tlas_start], roots, *tri_boxes(prim_slots_tris))
    inst_lo, inst_hi = from_ordered(nlo[blas_offsets]), from_ordered(nhi[blas_offsets])
    terrs, _, _ = tightness_errors(nb[tlas_start:], [0], inst_lo, inst_hi)
    return errs + ["TLAS " + e for e in terrs]


def check_reference_tree(tris, r, offs=None):
    """validator (flat), permutation and tightness of a reference build"""
    tris = np.asarray(tris, np.float32).reshape(-1, 3, 3)
    n = tris.shape[0]
    pi = r["prim_indices"]
    assert np.array_equal(np.sort(pi), np.arange(n, dtype=np.uint32)), "prim_indices is not a permutation"
    if offs is None:
        rc, rep = host.validate_cwbvh(r["nodes"], pi, tris.min(axis=1), tris.max(axis=1), stack_limit=48)
        assert rc == 0, rep
        assert rep["prims_reached"] == n and rep["nodes_reached"] == r["nodes"].size // 80
        errs = tight_flat(r["nodes"], tris[pi])
    else:
        obj = np.searchsorted(offs, pi, side="right") - 1
        assert (np.bincount(obj, minlength=offs.size - 1) == np.diff(offs).astype(np.int64)).all()
        assert np.array_equal(np.sort(r["blas_offsets"]), np.arange(offs.size - 1, dtype=np.uint32))
        errs = tight_two_level(r["nodes"], tris[pi], r["blas_offsets"], r["info"]["tlas_start"])
    assert not errs, "\n".join(errs)


def check_bvh2(r, tris, offs=None):
    """the BVH2 the collapse starts from: a binary forest over the same leaves, every inner box the union of its children's
    bit for bit, counts that add up, consistent parents"""
    b, n = r["bvh2"], r["bvh2_leaves"]
    tris = np.asarray(tris, np.float32).reshape(-1, 3, 3)
    assert n == tris.shape[0] and b.size >= n
    leaf, inner = b[:n], b[n:]
    assert (leaf["left"] == -1).all() and (leaf["count"] == 1).all()
    assert np.array_equal(np.sort(leaf["right"]), np.arange(n)), "leaves are not the primitives"
    lo, hi = tri_boxes(tris[leaf["right"]])
    assert np.array_equal(ordered(leaf["lo"]), ordered(lo)) and np.array_equal(ordered(leaf["hi"]), ordered(hi))
    if inner.size:
        l, rr = inner["left"], inner["right"]
        assert (l >= 0).all() and (rr >= 0).all() and (l != rr).all()
        kids = np.concatenate([l, rr])
        assert np.unique(kids).size == kids.size, "a node has two parents"
        idx = np.arange(n, b.size)
        assert (b["parent"][l] == idx).all() and (b["parent"][rr] == idx).all()
        assert (inner["count"] == b["count"][l] + b["count"][rr]).all()
        assert np.array_equal(ordered(inner["lo"]), np.minimum(ordered(b["lo"][l]), ordered(b["lo"][rr])))
        assert np.array_equal(ordered(inner["hi"]), np.maximum(ordered(b["hi"][l]), ordered(b["hi"][rr])))
    roots = np.nonzero(b["parent"] == -1)[0]
    n_obj = 1 if offs is None else offs.size - 1
    assert roots.size == n_obj and b["count"][roots].sum() == n
    if offs is not None:                                        # one tree per object, over that object's triangles
        obj = np.searchsorted(offs, leaf["right"], side="right") - 1
        top = np.arange(b.size)
        for _ in range(64):
            top = np.where(b["parent"][top] >= 0, b["parent"][top], top)
        assert (b["parent"][top] == -1).all()
        assert all(np.unique(top[:n][obj == k]).size == 1 for k in range(n_obj))


# ---- CPU: the reference on its own -------------------------------------------------------------------------------------


@pytest.mark.parametrize("n", [1, 2, 3, 8, 9, 255, 256, 257, 1025, 4097])
def test_reference_soup_validates_and_is_tight(n):
    tris = soup(n, seed=n)
    r = ob.build_reference(tris, bvh2=True)
    check_reference_tree(tris, r)
    check_bvh2(r, tris)
    assert r["build_stats"]["n_nodes"] == r["nodes"].size // 80


@pytest.mark.parametrize("name", [c[0] for c in edge_geometry()])
def test_reference_edge_geometry_validates_and_is_tight(name):
    tris = dict(edge_geometry())[name]
    r = ob.build_reference(tris, bvh2=True)
    check_reference_tree(tris, r)
    check_bvh2(r, tris)
    e = np.asarray(r["nodes"], np.uint8).reshape(-1, 80)[:, 12:15]
    assert r["force_exact"] == bool((e >= 167).any())
    assert r["force_exact"] == (name == "huge")


def test_reference_signed_zero_rule():
    """a node's p takes -0.0 when any primitive below it has -0.0 at the minimum (fminf orders -0.0 below +0.0)"""
    tris = signed_zero_soup()
    r = ob.build_reference(tris)
    p = np.asarray(r["nodes"], np.uint8).reshape(-1, 80)[:, 0:12].copy().view(np.float32)
    assert np.signbit(p[p == 0]).any() and (~np.signbit(p[p == 0])).any()


@pytest.mark.parametrize("max_leaf,radius", [(1, 1), (2, 3), (3, 40), (3, 64), (1, 0)])
def test_reference_parameters(cornell, max_leaf, radius):
    tris = cornell.tris().reshape(-1, 3, 3)
    r = ob.build_reference(tris, max_leaf=max_leaf, radius=radius, bvh2=True)
    check_reference_tree(tris, r)
    check_bvh2(r, tris)


@pytest.mark.parametrize("passes,visits,rounds", [(0, 192, 3), (1, 192, 3), (4, 1, 3), (4, 16, 1), (4, 4096, 5), (8, 192, 3)])
def test_reference_bvh2_after_reinsertion(passes, visits, rounds):
    """the BVH2 stays a correct tree over the same leaves after PLOC alone and after every reinsertion setting; flat and forest"""
    tris = soup(3000, seed=21)
    r = ob.build_reference(tris, passes=passes, visits=visits, rounds=rounds, bvh2=True)
    check_bvh2(r, tris)
    check_reference_tree(tris, r)
    offs = np.array([0, 700, 701, 1900, 3000], np.uint64)
    r = ob.build_reference(tris, object_offsets=offs, passes=passes, visits=visits, rounds=rounds, bvh2=True)
    check_bvh2(r, tris, offs)
    check_reference_tree(tris, r, offs)


def test_reinsertion_statistics():
    """passes=0 moves nothing and reports nothing; the default moves subtrees and lowers the SAH cost on hairball and caldera,
    and its sah_before is the PLOC tree's cost"""
    for name, seed, size in (("hairball", 3, 0.1), ("caldera", 5, 0.02)):
        tris = host.Mesh.generate(name, seed, size).tris()
        r0 = ob.build_reference(tris, passes=0, bvh2=True)
        s0 = r0["build_stats"]
        assert s0["reinsert_moves"] == 0 and s0["reinsert_passes"] == 0 and s0["sah_after"] == s0["sah_before"]
        b = r0["bvh2"][r0["bvh2_leaves"]:]
        d = b["hi"] - b["lo"]
        plo_cost = float(np.sum((d[:, 0] * d[:, 1] + d[:, 1] * d[:, 2] + d[:, 2] * d[:, 0]).astype(np.float64)))
        s = ob.build_reference(tris)["build_stats"]
        assert s["reinsert_passes"] == 4 and s["reinsert_moves"] > 0, (name, s)
        assert s["sah_after"] < s["sah_before"], (name, s)
        assert s["sah_before"] == pytest.approx(plo_cost, rel=1e-12)


def test_reference_bytes_trace_like_brute_force(cornell):
    """the oracle on the reference's own bytes finds what an exhaustive search finds"""
    tris = cornell.tris().reshape(-1, 3, 3)
    r = ob.build_reference(tris)
    orc = ob.Oracle(r["nodes"], r["tri_bytes"], 48)
    rays = random_rays(3000, seed=5)
    got = orc.trace(rays, stack_limit=48)
    brute, _ = orc.brute_force(rays)
    hit = brute["prim"] != ob.INVALID_PRIM
    assert np.array_equal(hit, got["prim"] != ob.INVALID_PRIM) and hit.sum() > 500
    assert (np.abs(got["t"][hit] - brute["t"][hit]) <= 1e-5 * np.abs(brute["t"][hit])).all()
    assert (got["t"][hit].view(np.uint32) == brute["t"][hit].view(np.uint32)).mean() > 0.999


def test_host_producer_trees_are_tight(cornell):
    """the host producer (binned SAH) shares the encoder: its trees must be tight too, flat and two-level"""
    for name, seed, size in (("kitchen", 1, 1.0), ("hairball", 3, 0.02)):
        tris = host.Mesh.generate(name, seed, size).tris().reshape(-1, 3, 3)
        nodes, pi, _ = host.build_cwbvh(tris)
        errs = tight_flat(nodes, tris[pi])
        assert not errs, f"{name}:\n" + "\n".join(errs)
    tris = cornell.tris().reshape(-1, 3, 3)
    p = host.PackedScene(cornell)
    assert not tight_flat(p.bvh_bytes, tris[p.prim_to_mesh_tri])
    p = host.PackedScene(cornell, use_tlas=True)
    errs = tight_two_level(p.bvh_bytes, tris[p.prim_to_mesh_tri], p.blas_offsets, p.tlas_start)
    assert not errs, "\n".join(errs)


def test_tightness_check_sees_a_loose_node():
    """the check is not vacuous: one quantisation step, an exponent or an origin off by one fails it"""
    tris = soup(300, seed=3)
    r = ob.build_reference(tris)
    good = r["nodes"].reshape(-1, 80)
    slots = tris[r["prim_indices"]]
    assert not tight_flat(good, slots)
    for byte, delta in ((40, 1), (13, 1), (0, 1)):       # qhi x of slot 0, exponent y, lowest byte of p.x
        bad = good.copy()
        bad[0, byte] = np.uint8((int(bad[0, byte]) + delta) % 256)
        assert tight_flat(bad, slots), byte


# ---- GPU: device bytes against the reference ---------------------------------------------------------------------------

FIELDS = (("p", 0, 12), ("e", 12, 15), ("imask", 15, 16), ("child base", 16, 20), ("prim base", 20, 24), ("meta", 24, 32), ("q bounds", 32, 80))
STATS = ("n_nodes", "ploc_iterations", "levels", "reinsert_passes", "reinsert_moves")


def device_build(monkeypatch, tris, stride=48, max_leaf=3, radius=0, offs=None, passes=4, visits=192, rounds=3, tail=True):
    """the device build with every knob the reference takes as a parameter set explicitly in the environment"""
    from tray_racing_b200 import cuda
    monkeypatch.setenv("TRAY_CUDA_BUILD_REINSERT", str(passes))
    monkeypatch.setenv("TRAY_CUDA_BUILD_REINSERT_VISITS", str(visits))
    monkeypatch.setenv("TRAY_CUDA_BUILD_REINSERT_ROUNDS", str(rounds))
    monkeypatch.setenv("TRAY_BUILD_PLOC_TAIL", "1" if tail else "0")
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, max_prims_per_leaf=max_leaf, search_radius=radius, object_offsets=offs)
    nodes, tri_bytes, pi = sc.download_bvh()
    out = dict(scene=sc, nodes=nodes, tri_bytes=tri_bytes, prim_indices=pi, blas_offsets=sc.download_instances(),
               info=sc.info(), build_stats=sc.build_stats)
    return out


def mismatch_report(dev, ref):
    """where device and reference part: stats side by side, the first differing wide node with its BFS level and field, the
    first differing prim_indices slot"""
    lines = [f"{k}: device {dev['build_stats'][k]} reference {ref['build_stats'][k]}" for k in STATS + ("sah_before", "sah_after")]
    lines.append(f"tlas_start: device {dev['info']['tlas_start']} reference {ref['info']['tlas_start']}")
    dn, rn = dev["nodes"].reshape(-1, 80), ref["nodes"].reshape(-1, 80)
    m = min(dn.shape[0], rn.shape[0])
    diff = np.nonzero((dn[:m] != rn[:m]).any(axis=1))[0]
    if diff.size:
        i = int(diff[0])
        ts = ref["info"]["tlas_start"]
        roots = np.unique(ref["blas_offsets"]) if ref["info"]["is_tlas"] else [0]
        part, j = ("TLAS", i - ts) if ref["info"]["is_tlas"] and i >= ts else ("BLAS", i)
        sub = rn[ts:] if part == "TLAS" else (rn[:ts] if ref["info"]["is_tlas"] else rn)
        level = tree_walk(decode(sub), [0] if part == "TLAS" else roots)[0][j]
        fields = [name for name, a, b in FIELDS if (dn[i, a:b] != rn[i, a:b]).any()]
        lines.append(f"first differing node {i} ({part} BFS level {level}; {diff.size} nodes differ): fields {', '.join(fields)}")
        lines.append(f"  device    {dn[i].tolist()}\n  reference {rn[i].tolist()}")
    elif dn.shape[0] != rn.shape[0]:
        lines.append(f"node counts differ: device {dn.shape[0]} reference {rn.shape[0]}")
    dp, rp = dev["prim_indices"], ref["prim_indices"]
    if dp.size == rp.size:
        d = np.nonzero(dp != rp)[0]
        if d.size:
            lines.append(f"first differing prim_indices slot {int(d[0])}: device {int(dp[d[0]])} reference {int(rp[d[0]])} ({d.size} slots differ)")
    else:
        lines.append(f"prim_indices sizes differ: {dp.size} / {rp.size}")
    return "\n".join(lines)


def compare(monkeypatch, tris, offs=None, stride=48, max_leaf=3, radius=0, passes=4, visits=192, rounds=3, tail=True, keep=False):
    """device build == reference build: bytes exactly, stats exactly, SAH sums within 1e-5"""
    tris = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 3, 3)
    ref = ob.build_reference(tris, tri_stride=stride, max_leaf=max_leaf, radius=radius, object_offsets=offs,
                             passes=passes, visits=visits, rounds=rounds)
    dev = device_build(monkeypatch, tris, stride, max_leaf, radius, offs, passes, visits, rounds, tail)
    try:
        same = (np.array_equal(dev["nodes"], ref["nodes"]) and np.array_equal(dev["prim_indices"], ref["prim_indices"])
                and np.array_equal(dev["blas_offsets"], ref["blas_offsets"]) and dev["info"]["tlas_start"] == ref["info"]["tlas_start"]
                and all(dev["build_stats"][k] == ref["build_stats"][k] for k in STATS))
        assert same, mismatch_report(dev, ref)
        assert np.array_equal(dev["tri_bytes"], ref["tri_bytes"]), "triangle records differ"
        for k in ("sah_before", "sah_after"):
            assert dev["build_stats"][k] == pytest.approx(ref["build_stats"][k], rel=1e-5, abs=1e-30), mismatch_report(dev, ref)
    finally:
        if not keep:
            dev["scene"].close()
    return dev, ref


SIZES = [0, 1, 2, 3, 8, 9, 255, 256, 257, 1023, 1024, 1025, 4097, 20000]


@gpu
@pytest.mark.parametrize("tail", [True, False])
@pytest.mark.parametrize("n", SIZES)
def test_device_soup_sizes(monkeypatch, n, tail):
    """the 256-thread block halo of the PLOC kernels and the 1024-cluster single-block tail, with and without the tail"""
    tris = soup(n, seed=n + 100)
    compare(monkeypatch, tris, tail=tail, passes=0)
    compare(monkeypatch, tris, tail=tail)


@gpu
@pytest.mark.parametrize("name", [c[0] for c in edge_geometry()])
def test_device_edge_geometry(monkeypatch, name):
    tris = dict(edge_geometry())[name]
    compare(monkeypatch, tris, passes=0)
    compare(monkeypatch, tris, passes=0, tail=False)           # the ties of the multi-kernel PLOC loop, not only the tail's
    dev, ref = compare(monkeypatch, tris, keep=True)
    try:
        if name == "huge":                                      # scale >= 2^40: the device traversal must switch to its exact node test
            assert ref["force_exact"]
            rays = rays_at(tris, 20000, seed=9)
            orc = ob.Oracle(ref["nodes"], ref["tri_bytes"], 48)
            got, want = dev["scene"].traverse(rays), orc.trace(rays, stack_limit=48)
            assert np.array_equal(got["prim"], want["prim"]) and np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32))
            assert (want["prim"] != ob.INVALID_PRIM).sum() > 100
        if name == "signed_zero":                               # both signs of zero reach some p
            p = ref["nodes"].reshape(-1, 80)[:, 0:12].copy().view(np.float32)
            assert np.signbit(p[p == 0]).any() and (~np.signbit(p[p == 0])).any()
    finally:
        dev["scene"].close()


def _scene(name):
    if name in ("cornell_box", "box"):
        return load_golden_mesh(name).tris()
    gen = dict(kitchen=("kitchen", 1, 1.0), hairball=("hairball", 3, 0.1), sanmiguel=("sanmiguel", 4, 0.01), demoscene=("demoscene", 2, 0.01))
    return host.Mesh.generate(*gen[name]).tris()


@gpu
@pytest.mark.parametrize("name", ["cornell_box", "box", "kitchen", "hairball", "sanmiguel", "demoscene"])
def test_device_scenes(monkeypatch, name):
    """PLOC and the collapse first (no reinsertion), so that a disagreement there is told apart from one in the reinsertion"""
    tris = _scene(name)
    compare(monkeypatch, tris, passes=0)
    compare(monkeypatch, tris)


@gpu
@pytest.mark.parametrize("stride,max_leaf,radius", [(24, 1, 0), (48, 2, 1), (64, 3, 3), (48, 1, 40), (24, 3, 64), (64, 2, 0)])
def test_device_parameters(monkeypatch, cornell, stride, max_leaf, radius):
    tris = np.concatenate([cornell.tris().reshape(-1, 3, 3), soup(2000, seed=radius)])
    compare(monkeypatch, tris, stride=stride, max_leaf=max_leaf, radius=radius, passes=0)
    compare(monkeypatch, tris, stride=stride, max_leaf=max_leaf, radius=radius)


@gpu
@pytest.mark.parametrize("passes,visits,rounds", [(1, 192, 3), (4, 1, 3), (4, 16, 1), (8, 4096, 5), (4, 192, 5), (8, 16, 3)])
def test_device_reinsertion_knobs(monkeypatch, passes, visits, rounds):
    tris = _scene("kitchen")
    dev, ref = compare(monkeypatch, tris, passes=passes, visits=visits, rounds=rounds)
    # with one visit a search sees only v's own sibling, the identity move, and stops before it climbs: nothing can move
    assert (ref["build_stats"]["reinsert_moves"] > 0) == (visits > 1)


def _two_level(name):
    if name in ("cornell_box", "box"):
        m = load_golden_mesh(name)
        return m.tris(), m.object_offsets()
    if name == "caldera":
        m = host.Mesh.generate("caldera", 5, 0.02)
        return m.tris(), m.object_offsets()
    if name == "many_small":
        return many_small_objects()
    if name == "single_object":
        t = soup(3000, seed=31)
        return t, np.array([0, t.shape[0]], np.uint64)
    if name == "one_triangle_objects":
        t = soup(300, seed=32)
        return t, np.arange(301, dtype=np.uint64)
    raise KeyError(name)


@gpu
@pytest.mark.parametrize("name", ["cornell_box", "box", "caldera", "many_small", "single_object", "one_triangle_objects"])
def test_device_two_level(monkeypatch, name):
    tris, offs = _two_level(name)
    compare(monkeypatch, tris, offs=offs, passes=0)
    compare(monkeypatch, tris, offs=offs, tail=False, passes=0)
    dev, ref = compare(monkeypatch, tris, offs=offs, keep=True)
    try:
        errs = tight_two_level(dev["nodes"], np.asarray(tris, np.float32).reshape(-1, 3, 3)[dev["prim_indices"]],
                               dev["blas_offsets"], dev["info"]["tlas_start"])
        assert not errs, "\n".join(errs)
    finally:
        dev["scene"].close()


@gpu
def test_device_trees_are_tight(monkeypatch):
    """the builder-independent check on device bytes directly"""
    for tris in (_scene("hairball"), signed_zero_soup(), soup(5000, seed=41)):
        tris = np.asarray(tris, np.float32).reshape(-1, 3, 3)
        dev = device_build(monkeypatch, tris)
        try:
            errs = tight_flat(dev["nodes"], tris[dev["prim_indices"]])
            assert not errs, "\n".join(errs)
        finally:
            dev["scene"].close()
