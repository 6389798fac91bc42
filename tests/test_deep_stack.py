"""The traversal stack beyond shared memory.  `trace_kernel` keeps a lane's stack in three tiers: entries 0-11 in shared memory,
12-47 in a local spill array, and past 47 `push` raises the overflow bit of the error word and drops the entry, which the host
reports as TRAY_ERR_OVERFLOW (error -4).  CWBVHs built from real scenes never push more than 12 entries, so these tests write
deep trees by hand: a LADDER of D levels, where spine node i covers [0, r^i]^3 and holds the next spine node (slot 0) and a
decoy node over [r^(i+1), r^i]^3 (slot 7) with one triangle on the plane x+y+z = r^i + 2 r^(i+1); the last spine node holds
one triangle.  A ray near the diagonal with an all-positive direction descends slot 0 first and pushes the decoy group at every
level: it needs D - 1 entries.  Rays with a tmin past the deepest triangles are closest-hit by a decoy triangle, so the group
that holds it is popped from a known depth and not merely fetched and culled.

Reference: the CPU oracle with a 48-entry stack (Oracle.trace(stack_limit=48)); Oracle.stack_need shows which depths each
batch really reaches.  The CPU tests check the encoder, that need against the independent HLSL transliteration, and the
oracle's capacity; the GPU tests check the kernels bit for bit against it and pin how an overflow is reported."""
import math

import numpy as np
import pytest

import oracle_binding as ob
from tray_racing_b200 import cuda, host

R = 0.93
F32_MAX = np.float32(3.402823466e+38)
KERNEL_STACK = 48                               # STACK_SMEM + STACK_SPILL in traverse.cuh
FLAT_DEPTHS = (12, 13, 32, 33, 48)              # needs D - 1 at the edges of shared memory, of obvhs' 32 and of the kernel's 48
FRAME_FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_KEEP_RAYS | cuda.RENDER_COUNTERS
DIAGONAL_CAMERA = host.Camera((-1.2,) * 3, (0, 0, 0), 10.0)          # pixels span needs 0 .. D - 1
SIDE_CAMERA = host.Camera((-1.2, -1.0, -1.3), (0.3, 0.5, 0.4), 20.0)  # shallow levels only: needs <= 13


# ---- a CWBVH encoder, written the way host/cwbvh_build.cpp's Collapser writes nodes ----------------------------------------
def quant_exponent(extent):
    extent = max(extent, 1e-20)
    k = math.ceil(math.log2(extent / 255.0))
    while math.ldexp(255.0, k) < extent:
        k += 1
    while math.ldexp(255.0, k - 1) >= extent:
        k -= 1
    return k


def encode_node(lo, hi, children, child_base=0, prim_base=0):
    """One 80-byte CwBvhNode over the cube [lo, hi]^3.  children: (slot, child_lo, child_hi, kind), kind "inner" or the
    triangle count of a leaf; inner children are the nodes child_base, child_base + 1, .. in slot order."""
    n = np.zeros(80, np.uint8)
    lo, hi = np.float32(lo), np.float32(hi)
    n[0:12] = np.full(3, lo, np.float32).view(np.uint8)                       # p = box min
    k = quant_exponent(float(hi) - float(lo))
    n[12:15] = k + 127
    scale = math.ldexp(1.0, k)
    n[16:24] = np.array([child_base, prim_base], np.uint32).view(np.uint8)
    tri_offset = 0
    for slot, clo, chi, kind in children:
        for a in range(3):
            n[32 + 16 * a + slot] = min(255, max(0, math.floor((float(np.float32(clo)) - float(lo)) / scale)))
            n[40 + 16 * a + slot] = min(255, max(0, math.ceil((float(np.float32(chi)) - float(lo)) / scale)))
        if kind == "inner":
            n[15] |= 1 << slot
            n[24 + slot] = 0x20 | (24 + slot)
        else:
            n[24 + slot] = (0x20, 0x60, 0xE0)[kind - 1] | tri_offset
            tri_offset += kind
    return n


def ladder_nodes(D, r=R, prim_base=0):
    """2D - 1 nodes; the leaf of decoy i references primitive prim_base + i, the last spine node's prim_base + D - 1"""
    s = [np.float32(r ** i) for i in range(D)]
    nodes = np.zeros((2 * D - 1, 80), np.uint8)
    for i in range(D):
        spine = 0 if i == 0 else 2 * i - 1
        if i < D - 1:
            nodes[spine] = encode_node(0, s[i], [(0, 0, s[i + 1], "inner"), (7, s[i + 1], s[i], "inner")], child_base=2 * i + 1)
            nodes[2 * i + 2] = encode_node(s[i + 1], s[i], [(0, s[i + 1], s[i], 1)], prim_base=prim_base + i)
        else:
            nodes[spine] = encode_node(0, s[i], [(0, 0, s[i], 1)], prim_base=prim_base + i)
    return nodes


def ladder_tris(D, r=R):
    s = [np.float32(r ** i) for i in range(D)]
    t = [[s[i], s[i + 1], s[i + 1], s[i + 1], s[i], s[i + 1], s[i + 1], s[i + 1], s[i]] for i in range(D - 1)]
    t.append([s[-1], 0, 0, 0, s[-1], 0, 0, 0, s[-1]])
    return np.array(t, np.float32)


class Scene:
    """nodes + triangle soup (+ blas_offsets, tlas_start of a two-level scene), as the oracle and the CUDA scene take them"""

    def __init__(self, nodes, tris, blas=None, tlas_start=0, stride=48):
        self.nodes, self.tris, self.blas, self.tlas_start, self.stride = nodes, tris, blas, tlas_start, stride
        self.rec = host.tri_records(tris, stride)

    def oracle(self):
        return ob.Oracle(self.nodes, self.rec, self.stride, self.blas, self.tlas_start, self.blas is not None)

    def cuda(self):
        return cuda.TrayCudaScene(self.nodes, self.rec, self.stride, self.blas, self.tlas_start)


def flat_ladder(D, stride=48):
    return Scene(ladder_nodes(D), ladder_tris(D), stride=stride)


def tlas_ladder(D, stride=48):
    """a D-level ladder as the TLAS: its leaves are instances 0 .. D-1, instance j a one-node BLAS over triangle j"""
    tris = ladder_tris(D)
    t3 = tris.reshape(-1, 3, 3)
    blas = [encode_node(t3[j].min(), t3[j].max(), [(0, t3[j].min(), t3[j].max(), 1)], prim_base=j) for j in range(D)]
    return Scene(np.concatenate([np.stack(blas), ladder_nodes(D)]), tris, np.arange(D, dtype=np.uint32), D, stride)


def blas_ladder(D, stride=48):
    """a shallow TLAS (one root, one leaf of two instances over the unit cube) over a D-level ladder (instance 1, entered first
    with instance 0 on the stack) and an 8-level ladder of another ratio (instance 0): the deep instance needs D entries"""
    deep, shallow = ladder_nodes(D), ladder_nodes(8, 0.8, prim_base=D)
    root = encode_node(0, 1, [(0, 0, 1, 2)], prim_base=0)
    nodes = np.concatenate([shallow, deep, root[None]])
    blas = np.array([0, len(shallow)], np.uint32)
    return Scene(nodes, np.concatenate([ladder_tris(D), ladder_tris(8, 0.8)]), blas, len(nodes) - 1, stride)


def ladder_rays(n, seed, tris, tmin_fraction=0.25, spread=(1e-4, 0.3)):
    """rays from (-1, -1, -1) +- 0.01 along (1, 1, 1), each direction component off by up to a log-uniform `spread`: the
    nearer the diagonal, the deeper the ray goes.  The last `tmin_fraction` get a tmin between the planes of triangles j + 1
    and j (j random): their closest hit is the decoy triangle of level j, behind every deeper one."""
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, ob.RAY_DTYPE)
    rays["o"] = -1 + rng.uniform(-0.01, 0.01, (n, 3))
    jitter = 10 ** rng.uniform(np.log10(spread[0]), np.log10(spread[1]), (n, 1))
    d = 1 + jitter * rng.uniform(-1, 1, (n, 3))
    rays["d"] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays["tmax"] = F32_MAX
    k = int(n * tmin_fraction)
    if k:
        plane = tris[:, 0:3].astype(np.float64).sum(axis=1)                 # x + y + z of each triangle's plane
        j = rng.integers(0, len(tris) - 1, k)
        so, sd = rays["o"][-k:].astype(np.float64).sum(axis=1), rays["d"][-k:].astype(np.float64).sum(axis=1)
        rays["tmin"][-k:] = (((plane[j] + plane[j + 1]) / 2 - so) / sd).astype(np.float32)
    return rays


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_hits_identical(gpu, ref, what=""):
    assert (gpu["prim"] == ref["prim"]).all(), f"{what}: {(gpu['prim'] != ref['prim']).sum()} primitive ids differ"
    assert (bits(gpu["t"]) == bits(ref["t"])).all(), f"{what}: {(bits(gpu['t']) != bits(ref['t'])).sum()} hit t differ"


def assert_reaches(need, depth, what=""):
    """the batch really needs `depth` entries, and needs spread below it (the spill region's boundaries included)"""
    assert need.max() == depth, f"{what}: deepest need {need.max()}, expected {depth}"
    assert len(np.unique(need)) >= min(depth, 10), f"{what}: needs {np.unique(need)}"
    if depth > 12:
        assert ((need >= 12) & (need < depth)).any(), f"{what}: no need between 12 and {depth}"


def hits_from_depth(ref, rays, levels):
    """closest hits on decoy triangles of `levels`, by rays with a tmin past the deeper ones: groups popped from that depth"""
    return int(np.isin(ref["prim"], levels).sum() - np.isin(ref["prim"][rays["tmin"] == 0], levels).sum())


# ---- CPU: the encoder, the oracle's need and capacity ----------------------------------------------------------------------
@pytest.mark.parametrize("D", [2, 13, 14, 33, 34, 49, 50])
def test_ladders_validate_with_the_claimed_depth(D):
    sc = flat_ladder(D)
    t3 = sc.tris.reshape(-1, 3, 3)
    rc, rep = host.validate_cwbvh(sc.nodes, None, t3.min(axis=1), t3.max(axis=1), stack_limit=0)
    assert rc == 0 and rep["nodes_reached"] == 2 * D - 1 and rep["prims_reached"] == D, rep
    assert rep["max_stack"] == D - 1 and rep["max_depth"] == D


def test_two_level_ladders_validate():
    sc = tlas_ladder(48)
    t3 = sc.tris.reshape(-1, 3, 3)
    rc, rep = host.validate_cwbvh(sc.nodes[sc.tlas_start:], None, t3.min(axis=1), t3.max(axis=1), stack_limit=0)
    assert rc == 0 and rep["max_stack"] == 47, rep
    for j in range(0, 48, 7):                                           # the one-node BLASes, each over its own triangle
        blas = sc.nodes[j].copy()
        blas[20:24] = 0
        rc, rep = host.validate_cwbvh(blas[None], None, t3[j:j + 1].min(axis=1), t3[j:j + 1].max(axis=1), stack_limit=0)
        assert rc == 0, rep
    sc = blas_ladder(47)
    t3 = sc.tris.reshape(-1, 3, 3)[:47]
    rc, rep = host.validate_cwbvh(sc.nodes[sc.blas[1]:sc.tlas_start], None, t3.min(axis=1), t3.max(axis=1), stack_limit=0)
    assert rc == 0 and rep["max_stack"] == 46, rep


def test_oracle_need_equals_the_transliteration_peak():
    import hlsl_transliteration as hl
    for D, seed in ((14, 1), (34, 2), (50, 3)):
        sc = flat_ladder(D)
        rays = ladder_rays(48, seed, sc.tris, tmin_fraction=0)
        need = sc.oracle().stack_need(rays)
        hs = hl.Scene(sc.nodes.tobytes(), sc.rec.tobytes(), 48)
        peak = [hl.traverse_bvh(hs, rays["o"][i], rays["d"][i], stack_peak=True)[-1] for i in range(len(rays))]
        assert need.tolist() == peak
        assert need.max() == D - 1
    sc = tlas_ladder(20)
    rays = ladder_rays(32, 4, sc.tris, tmin_fraction=0)
    need = sc.oracle().stack_need(rays)
    hs = hl.Scene(sc.nodes.tobytes(), sc.rec.tobytes(), 48, sc.blas, sc.tlas_start)
    assert need.tolist() == [hl.traverse_bvh_tlas(hs, rays["o"][i], rays["d"][i], stack_peak=True)[-1] for i in range(len(rays))]
    assert need.max() == 19


def test_validator_bounds_the_need(cornell):
    for D in (13, 34, 50):
        sc = flat_ladder(D)
        t3 = sc.tris.reshape(-1, 3, 3)
        _, rep = host.validate_cwbvh(sc.nodes, None, t3.min(axis=1), t3.max(axis=1), stack_limit=0)
        assert sc.oracle().stack_need(ladder_rays(2000, D, sc.tris)).max() <= rep["max_stack"]
    from conftest import random_rays
    tris = cornell.tris()
    nodes, pidx, _ = host.build_cwbvh(tris)
    t3 = tris.reshape(-1, 3, 3)[pidx]
    _, rep = host.validate_cwbvh(nodes, None, t3.min(axis=1), t3.max(axis=1), stack_limit=0)
    need = ob.Oracle(nodes, host.tri_records(tris[pidx])).stack_need(random_rays(20000, 5))
    assert 0 < need.max() <= rep["max_stack"]


def test_oracle_stack_capacity():
    rays = ladder_rays(500, 6, ladder_tris(50), tmin_fraction=0, spread=(1e-5, 1e-3))     # all near the diagonal
    for D, ok, too_small in ((33, ob.STACK_DEFAULT, None), (34, 48, ob.STACK_DEFAULT), (49, 48, None), (50, 64, 48)):
        orc = flat_ladder(D).oracle()
        assert orc.stack_need(rays).max() == D - 1
        orc.trace(rays, stack_limit=ok)
        if too_small:
            with pytest.raises(RuntimeError, match="overflow"):
                orc.trace(rays, stack_limit=too_small)
    flat_ladder(33).oracle().trace(rays)                                   # default 32: a need of 32 passes ..
    with pytest.raises(RuntimeError, match="overflow"):
        flat_ladder(34).oracle().trace(rays)                               # .. and 33 does not
    with pytest.raises(RuntimeError, match="overflow"):
        flat_ladder(34).oracle().render(host.view_from_camera(DIAGONAL_CAMERA, 64, 64), 64, 64, 0)
    with pytest.raises(ValueError):
        flat_ladder(13).oracle().trace(rays, stack_limit=ob.STACK_MAX + 1)
    assert ob.lib().orc_stack_limit() == ob.STACK_DEFAULT                  # every call leaves the default in place
    with pytest.raises(RuntimeError):
        flat_ladder(66).oracle().stack_need(rays)


def deep_batches():
    """the ray batches of the GPU parity cases below (flat and two-level ladders, any-hit), by case: (scene, rays, any_hit)"""
    out = {}
    for d in FLAT_DEPTHS:
        sc = flat_ladder(d + 1)
        out[f"flat {d}"] = (sc, ladder_rays(4096, d, sc.tris), False)
        out[f"flat {d} large"] = (sc, ladder_rays((1 << 18) + 1234, 100 + d, sc.tris), False)
    sc = flat_ladder(49)
    out["any-hit"] = (sc, mixed_rays(sc), True)
    sc = tlas_ladder(48)
    out["tlas ladder"] = (sc, ladder_rays(8192, 48, sc.tris, tmin_fraction=0.5), False)
    sc = blas_ladder(48)
    out["blas ladder"] = (sc, ladder_rays(8192, 49, sc.tris, tmin_fraction=0.5), False)
    return out


def mixed_rays(sc):
    """deep rays and shallow ones interleaved, so that lanes retiring from the spill region are refilled with short rays"""
    deep = ladder_rays(20000, 7, sc.tris, spread=(1e-5, 3e-3))
    shallow = ladder_rays(20000, 8, sc.tris, spread=(0.05, 0.5))
    rays = np.empty(40000, ob.RAY_DTYPE)
    rays[0::2], rays[1::2] = deep, shallow
    return rays


def test_the_deep_cases_reach_every_stack_boundary():
    """The GPU cases' batches, taken together, need 12, 13, 32, 33, 47 and 48 entries (the printed histogram is the oracle's)."""
    hist = np.zeros(ob.STACK_MAX + 1, np.int64)
    for name, (sc, rays, any_hit) in deep_batches().items():
        need = sc.oracle().stack_need(rays, any_hit=any_hit)
        assert need.max() <= KERNEL_STACK, name
        hist += np.bincount(need, minlength=hist.size)
    print("stack need histogram:", {k: int(v) for k, v in enumerate(hist) if v})
    for need in (12, 13, 32, 33, 47, 48):
        assert hist[need] > 0, need


# ---- GPU: the kernels equal the 48-entry oracle through the spill region ----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("stride", [48, 64, 24])
@pytest.mark.parametrize("depth", FLAT_DEPTHS)
def test_flat_ladder_matches_the_48_entry_oracle(depth, stride):
    sc = flat_ladder(depth + 1, stride)
    orc = sc.oracle()
    batches = [ladder_rays(4096, depth, sc.tris)]
    if stride == 48:
        batches.append(ladder_rays((1 << 18) + 1234, 100 + depth, sc.tris))          # the chunked copy pipeline
    g = sc.cuda()
    try:
        for rays in batches:
            assert_reaches(orc.stack_need(rays), depth, f"{len(rays)} rays")
            ref, _, tot = orc.trace(rays, counts=True, stack_limit=KERNEL_STACK)
            if depth > 12:                                                              # closest hits popped from the spill region
                assert hits_from_depth(ref, rays, np.arange(12, depth)) > 0
            g.set_counting(False)
            assert_hits_identical(g.traverse(rays), ref, f"{len(rays)} rays")
            g.set_counting(True)
            assert_hits_identical(g.traverse(rays), ref, f"{len(rays)} rays, counting")
            cp, _ = g.counters()
            assert (cp["rays"], cp["nodes"], cp["tris"], cp["instances"], cp["hits"]) == \
                (len(rays), tot["nodes"], tot["tris"], tot["insts"], tot["hits"])
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("refill_min", [1, 32])
def test_any_hit_refills_lanes_retired_from_the_spill_region(monkeypatch, refill_min):
    monkeypatch.setenv("TRAY_CUDA_REFILL_MIN", str(refill_min))
    sc = flat_ladder(49)
    rays = mixed_rays(sc)
    orc = sc.oracle()
    assert_reaches(orc.stack_need(rays, any_hit=True), 48)
    ref = orc.trace(rays, any_hit=True, stack_limit=KERNEL_STACK)
    g = sc.cuda()
    try:
        assert_hits_identical(g.traverse(rays, any_hit=True), ref, "any-hit")
        assert_hits_identical(g.traverse(rays), orc.trace(rays, stack_limit=KERNEL_STACK), "closest hit")
        big = np.tile(rays, 7)                                                          # 280000 rays: the copy pipeline
        assert_hits_identical(g.traverse(big, any_hit=True), np.tile(ref, 7), "any-hit, pipelined")
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [cuda.VARIANT_TIE_LAST | cuda.VARIANT_BOX_TMIN_RAY,
                                   cuda.VARIANT_BOX_DIVIDE | cuda.VARIANT_ZERODIR_BOX_ONLY])
def test_semantic_variants_through_the_spill_region(flags):
    g = None
    try:
        for depth in (33, 48):
            sc = flat_ladder(depth + 1)
            rays = ladder_rays(8192, depth, sc.tris)
            ob.set_variant(flags)
            orc = sc.oracle()
            assert orc.stack_need(rays).max() == depth
            ref = orc.trace(rays, stack_limit=KERNEL_STACK)
            g = sc.cuda()
            g.set_variant(flags)
            assert_hits_identical(g.traverse(rays), ref, f"variant {flags:#x}, need {depth}")
            g.close()
            g = None
    finally:
        ob.set_variant(0)
        if g is not None:
            g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,stride", [("tlas ladder", 48), ("tlas ladder", 64), ("blas ladder", 48)])
def test_two_level_ladders_return_to_the_tlas_in_the_spill_region(shape, stride):
    """tlas ladder: instances are entered with the TLAS stack 0 .. 47 entries deep, so `sp == tlas_sp` ends an instance in
    the spill region.  blas ladder: a 48-deep BLAS below an instance entry that pushed the other instance."""
    sc = tlas_ladder(48, stride) if shape == "tlas ladder" else blas_ladder(48, stride)
    rays = ladder_rays(8192, 48 if shape == "tlas ladder" else 49, sc.tris, tmin_fraction=0.5)
    orc = sc.oracle()
    assert_reaches(orc.stack_need(rays), 47 if shape == "tlas ladder" else 48, shape)
    ref, _, tot = orc.trace(rays, counts=True, stack_limit=KERNEL_STACK)
    assert hits_from_depth(ref, rays, np.arange(12, 46)) > 0
    g = sc.cuda()
    try:
        assert_hits_identical(g.traverse(rays), ref, shape)
        g.set_counting(True)
        assert_hits_identical(g.traverse(rays), ref, shape + ", counting")
        cp, _ = g.counters()
        assert (cp["nodes"], cp["tris"], cp["instances"]) == (tot["nodes"], tot["tris"], tot["insts"]) and tot["insts"] > len(rays)
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
def test_frames_down_the_ladder(overlap):
    """A camera looking down the diagonal of a 48-deep ladder: both frame paths, against Oracle.render with 48 entries."""
    w, h = 256, 192
    sc = flat_ladder(49)
    view = host.view_from_camera(DIAGONAL_CAMERA, w, h)
    orc = sc.oracle()
    assert_reaches(orc.stack_need(ob.primary_rays(view, w, h)), 48, "primary rays")
    ref = orc.render(view, w, h, 0, rgba=True, stack_limit=KERNEL_STACK)
    g = sc.cuda()
    try:
        g.render(view, w, h, 0, FRAME_FLAGS | (cuda.RENDER_OVERLAP if overlap else 0))
        g.sync()
        out = g.download(primary=True, bounce=True, bounce_rays=True, rgba=True)
        assert_hits_identical(out["primary"], ref["primary"], "primary")
        assert (out["bounce_rays"].view(np.uint32) == ref["bounce_rays"].view(np.uint32)).all(), "bounce rays differ"
        assert_hits_identical(out["bounce"], ref["bounce"], "bounce")
        assert np.abs(out["rgba"].reshape(-1, 4).astype(int) - ref["rgba"].astype(int)).max() <= 1
        cp, cb = g.counters()
        for got, want in ((cp, ref["primary_totals"]), (cb, ref["bounce_totals"])):
            assert (got["rays"], got["hits"], got["nodes"], got["tris"]) == (want["rays"], want["hits"], want["nodes"], want["tris"])
    finally:
        g.close()


# ---- GPU: the overflow status -----------------------------------------------------------------------------------------------
def overflow_case(D):
    """a ladder of D levels, a batch with rays that need D - 1 entries and a clean batch (needs <= 48) for it"""
    sc = flat_ladder(D)
    orc = sc.oracle()
    rays = ladder_rays(4096, 11, sc.tris)
    need = orc.stack_need(rays)
    assert need.max() == D - 1
    clean = rays[need <= KERNEL_STACK]
    return sc, orc, rays, clean


def expect(overflows):
    """the call raises TRAY_ERR_OVERFLOW when `overflows`, and nothing otherwise"""
    import contextlib
    return pytest.raises(cuda.TrayCudaError, match=r"error -4\b") if overflows else contextlib.nullcontext()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [49, 50])
def test_batch_overflow_is_reported_once_by_the_call_that_covers_it(D):
    import torch
    over = D - 1 > KERNEL_STACK
    sc, orc, rays, clean = overflow_case(D)
    ref_clean = orc.trace(clean, stack_limit=KERNEL_STACK)
    big = ladder_rays((1 << 18) + 99, 12, sc.tris)
    big_clean = big[orc.stack_need(big) <= KERNEL_STACK]
    assert over == (len(big_clean) < len(big))
    g = sc.cuda()
    try:
        for any_hit in (False, True):
            assert (orc.stack_need(rays, any_hit=any_hit).max() > KERNEL_STACK) == over
            with expect(over):
                g.traverse(rays, any_hit=any_hit)
            assert_hits_identical(g.traverse(clean, any_hit=any_hit), orc.trace(clean, any_hit=any_hit, stack_limit=KERNEL_STACK),
                                  f"clean batch after the overflow, any_hit={any_hit}")
        with expect(over):
            g.traverse(big)                                                  # the pipelined path
        assert_hits_identical(g.traverse(big_clean), orc.trace(big_clean, stack_limit=KERNEL_STACK), "pipelined clean batch")

        def device(r):
            return torch.from_numpy(r.view(np.uint8).copy()).cuda(), torch.empty(len(r) * 8, dtype=torch.uint8, device="cuda")
        d_rays, d_hits = device(rays)
        g.traverse_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr())   # asynchronous: nothing to report yet ..
        with expect(over):
            g.sync()                                                         # .. the synchronising call reports it
        g.sync()                                                             # once
        with expect(over):
            g.traverse_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr(), timed=True)
        g.sync()
        assert_hits_identical(g.traverse(clean), ref_clean, "clean batch after traverse_device")
        c_rays, c_hits = device(clean)
        g.traverse_device(c_rays.data_ptr(), len(clean), c_hits.data_ptr(), timed=True)
        assert_hits_identical(c_hits.cpu().numpy().view(ob.HIT_DTYPE), ref_clean, "clean traverse_device")
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [49, 50])
def test_frame_overflow_is_reported_for_its_own_frame(D):
    import torch
    over = D - 1 > KERNEL_STACK
    w, h = 128, 128
    sc, orc, _, _ = overflow_case(D)
    deep = host.view_from_camera(DIAGONAL_CAMERA, w, h)
    side = host.view_from_camera(SIDE_CAMERA, w, h)
    assert (orc.stack_need(ob.primary_rays(deep, w, h)).max() > KERNEL_STACK) == over
    ref_side = orc.render(side, w, h, 0, rgba=True, stack_limit=KERNEL_STACK)
    ref_deep = orc.render(deep, w, h, 0, stack_limit=ob.STACK_MAX)
    flags = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA

    def clean_frame(g, timed=True):
        g.render(side, w, h, 0, flags, timed=timed)
        out = g.download(primary=True, rgba=True)
        assert_hits_identical(out["primary"], ref_side["primary"], "clean frame")
        assert np.abs(out["rgba"].reshape(-1, 4).astype(int) - ref_side["rgba"].astype(int)).max() <= 1

    g = sc.cuda()
    bufs = [torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)]
    try:
        for overlap in (0, cuda.RENDER_OVERLAP):
            clean_frame(g)                                                   # (the wrapper learns the frame size of a call that returns)
            with expect(over):
                g.render(deep, w, h, 0, flags | overlap)                     # timed: synchronises, reports
            # the frame kernel finished (no watchdog) and every primary hit was published, the overflowing ray's too
            out = g.download(primary=True)
            fine = orc.stack_need(ob.primary_rays(deep, w, h)) <= KERNEL_STACK
            assert_hits_identical(out["primary"][fine], ref_deep["primary"][fine], "pixels that fit")
            assert not np.isnan(out["primary"]["t"]).any() and (bits(out["primary"]["t"]) != 0xFFFFFFFF).all()
            clean_frame(g)
            with expect(over):
                g.render_frame_ms(deep, w, h, 0, flags | overlap)
            clean_frame(g)
            g.render(deep, w, h, 0, flags | overlap, timed=False)
            with expect(over):
                g.download(rgba=True)
            g.sync()
            clean_frame(g, timed=False)
            # one frame in flight through the asynchronous readback
            g.render(deep, w, h, 0, flags | overlap, timed=False)
            g.readback_begin(bufs[0], 0)
            with expect(over):
                g.readback_wait(0)
            g.sync()
            g.render(side, w, h, 0, flags | overlap, timed=False)
            g.readback_begin(bufs[1], 1)
            g.readback_wait(1)
            assert np.abs(bufs[1].reshape(-1, 4).astype(int) - ref_side["rgba"].astype(int)).max() <= 1
        # two frames in flight: A overflows, B is clean; each wait reports its own frame
        g.set_frames_in_flight(2)
        for overlap in (0, cuda.RENDER_OVERLAP):
            g.render(deep, w, h, 0, flags | overlap, timed=False)
            g.readback_begin(bufs[0], 0)
            g.render(side, w, h, 0, flags | overlap, timed=False)
            g.readback_begin(bufs[1], 1)
            with expect(over):
                g.readback_wait(0)
            g.readback_wait(1)
            assert np.abs(bufs[1].reshape(-1, 4).astype(int) - ref_side["rgba"].astype(int)).max() <= 1
            g.sync()
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [49, 50])
def test_start_and_group_report_the_overflow(D):
    over = D - 1 > KERNEL_STACK
    w, h = 128, 128
    sc, orc, _, _ = overflow_case(D)
    deep = host.view_from_camera(DIAGONAL_CAMERA, w, h)
    side = host.view_from_camera(SIDE_CAMERA, w, h)
    with expect(over):
        mn, _, frames = cuda.start(sc.nodes, np.zeros(0, np.uint8), sc.rec, 0, deep, w, h, render_time=0.05)
        assert frames >= 1 and mn > 0
    grp = cuda.TrayCudaGroup(sc.nodes, sc.rec, devices=[0])
    try:
        with expect(over):
            grp.render(deep, w, h, timed=True)
        grp.render(side, w, h, timed=True)
        ref = orc.render(side, w, h, 0, rgba=True, stack_limit=KERNEL_STACK)
        assert np.abs(grp.frame().reshape(-1, 4).astype(int) - ref["rgba"].astype(int)).max() <= 1
        grp.sync()
    finally:
        grp.close()
