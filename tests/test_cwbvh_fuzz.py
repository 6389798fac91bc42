"""Every trace_kernel instantiation on CWBVH layouts that neither of the project's builders writes.

A scene handed to tray_cuda_scene_create is somebody else's bytes (obvhs writes them in the reference).  The host and device
builders both write one way: octant slots, inner children in BFS order, leaf triangles packed from offset 0, tight
quantisation, zeroed empty slots, no holes.  tests/cwbvh_bytes.py generates trees the validator accepts but that use what the
format allows beyond that: children in any slots, child blocks anywhere in the node array, leaf ranges in any order with
gaps, loose exponents and q bytes, random bytes in empty slots, nodes with 24 triangles, overlapping boxes, and in two-level
scenes permuted blas_offsets, a BLAS shared by two instances and BLAS nodes on both sides of the TLAS.  Bytes a correct
traversal never reads hold poison (see cwbvh_bytes.py); a kernel that reads them returns a poison id.

CPU: the validator accepts every generated tree, the knobs do what they say, the oracle equals exhaustive search and the
independent HLSL transliteration on them.  GPU: each of the 42 instantiations (pick_kernel in tray_cuda.cu) is bit-identical
to the oracle on them — hits, bounce rays, counters — and never returns a poison id."""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import random_rays
from cwbvh_bytes import (EXACT_EXP_BYTE, KNOBS, POISON_BOX, decode, random_cwbvh, random_objects, random_tlas, random_tris, tri_bounds)
from tray_racing_b200 import cuda, host

KERNEL_STACK = 48
F32_MAX = np.float32(3.402823466e+38)
STRIDES = (24, 48, 64)
# the 42 trace_kernel instantiations: MODE 0 {flat, TLAS} x {COUNT off, on} x {stride} x {closest hit, any hit, FRAME},
# MODE 1 {flat, TLAS} x {stride} (no counters, closest hit)
KERNELS = [(tlas, count, stride, kind, 0) for tlas in (False, True) for count in (False, True) for stride in STRIDES
           for kind in ("closest", "any", "frame")] + [(tlas, False, stride, "closest", 1) for tlas in (False, True) for stride in STRIDES]


def kernel_id(k):
    tlas, count, stride, kind, mode = k
    return f"{'tlas' if tlas else 'flat'}-{'count' if count else 'nocount'}-{stride}-{kind}-mode{mode}"


def case_knobs(seed):
    """a different mix of the generator's freedoms per seed; every one appears in several cases"""
    return dict(split=("random", "median", "mix")[seed % 3], slots=("random", "octant", "low", "high", "mix")[seed % 5],
                order=("random", "dfs", "bfs", "random")[seed % 4], leaf_order=("random", "slot")[seed % 2],
                exact_node=seed % 6 == 5)


def make_case(tlas, stride, seed, n_tris=1200):
    """(triangle soup, Generated, Scene) of one GPU case"""
    tris = random_tris(n_tris, seed)
    if tlas:
        tris, off = random_objects(tris, 4 + seed % 6, seed)
        g = random_tlas(tris, off, seed, **case_knobs(seed))
    else:
        g = random_cwbvh(tris, seed, **case_knobs(seed))
    return tris, g, g.scene(tris, stride, seed)


def case_seed(k):
    return KERNELS.index(k) + 1


CAMERA = host.Camera((1.5, 1.1, 1.9), (0.0, 0.0, 0.0), 50.0)              # just outside the scene box [-1, 1]^3, looking at it


def case_rays(seed, n=20000):
    """rays at the scene box from a shell around it: 5 % axis-parallel, 15 % with a bounded [tmin, tmax]"""
    return random_rays(n, seed, axis_fraction=0.05, bounded_fraction=0.15)


def report_ok(rep, unreached, missing):
    bad = {k: v for k, v in rep.items() if v and k in ("prim_seen_twice", "node_visited_twice", "bad_child_index",
                                                        "bad_prim_index", "bad_meta", "bad_quant", "box_violations")}
    return not bad and rep["nodes_unreached"] == unreached and rep["prims_missing"] == missing


def validate(tris, g, sc):
    """every tree of the scene passes the validator with exactly the poison the generator reports"""
    rl, rh = tri_bounds(sc.tris)
    for base, size, unreached, missing in g.regions:
        if g.blas is not None and base == g.tlas_start:
            _, rep = host.validate_cwbvh(g.nodes[base:base + size], None, g.inst_lo, g.inst_hi, stack_limit=0)
        else:
            _, rep = host.validate_cwbvh(g.nodes[base:base + size], None, rl, rh, stack_limit=0)
        assert report_ok(rep, unreached, missing), (base, size, unreached, missing, rep)
        assert rep["prim_seen_twice"] == 0


def full_node(n):
    """8 leaves of 3 triangles (tri_y = 0xFFFFFF), not a poison node"""
    return not is_poison(n) and decode(n)[0] == 0 and [m >> 5 for _, m in decode(n)[3]] == [7] * 8


def is_poison(n):
    return n[0:12].view(np.float32)[0] == -POISON_BOX


def poison_free(hits, g, what=""):
    n = int(np.isin(hits["prim"], g.poison_ids()).sum())
    assert n == 0, f"{what}: {n} rays returned a poison record"


def zeroed_oracle(g, sc):
    """the oracle on the records with every poison record zeroed (a zero record is never hit)"""
    rec = sc.rec.reshape(len(g.rec_tri), -1).copy()
    rec[g.rec_tri < 0] = 0
    return ob.Oracle(g.nodes, rec.reshape(-1), sc.stride, g.blas, g.tlas_start, g.blas is not None)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_the_kernel_table_names_42_distinct_instantiations():
    assert len(KERNELS) == 42 and len(set(KERNELS)) == 42 and len({kernel_id(k) for k in KERNELS}) == 42
    assert sum(k[4] == 1 for k in KERNELS) == 6


def test_the_generator_is_deterministic():
    tris = random_tris(400, 3)
    a, b = random_cwbvh(tris, 11, slots="mix"), random_cwbvh(tris, 11, slots="mix")
    assert np.array_equal(a.nodes, b.nodes) and np.array_equal(a.rec_tri, b.rec_tri)
    assert not np.array_equal(a.nodes, random_cwbvh(tris, 12, slots="mix").nodes)
    t, off = random_objects(tris, 5, 3)
    a, b = random_tlas(t, off, 4), random_tlas(t, off, 4)
    assert np.array_equal(a.nodes, b.nodes) and np.array_equal(a.blas, b.blas) and a.tlas_start == b.tlas_start


@pytest.mark.parametrize("k", KERNELS, ids=kernel_id)
def test_every_gpu_case_is_valid_and_within_the_kernel_stack(k):
    tlas, _, stride, kind, _ = k
    tris, g, sc = make_case(tlas, stride, case_seed(k))
    validate(tris, g, sc)
    need = sc.oracle().stack_need(case_rays(case_seed(k)), any_hit=kind == "any")
    assert 0 < need.max() <= KERNEL_STACK


def special_scenes():
    """the shapes the case mix does not reach by chance: an empty scene, a root that is one leaf, flat sheets only, 24-triangle
    nodes everywhere, single-child chains, every node on the unfused path"""
    out = {"empty": (np.zeros((0, 9), np.float32), random_cwbvh(np.zeros((0, 9), np.float32), 1))}
    for n in (1, 2, 3):
        t = random_tris(n, 40 + n, flat_fraction=0)
        out[f"root leaf {n}"] = (t, random_cwbvh(t, n, root_leaf=True))
    t = random_tris(800, 44, flat_fraction=1.0)
    out["flat sheets"] = (t, random_cwbvh(t, 44, slots="mix", split="median"))
    t = random_tris(24 * 40, 45)
    out["24-triangle nodes"] = (t, random_cwbvh(t, 45, full=1.0, split="median"))
    t = random_tris(600, 46)
    out["chains"] = (t, random_cwbvh(t, 46, chain=0.6))
    out["exact path"] = (t, random_cwbvh(t, 47, exact_node=True, exp_raise=0.8, slack=0.8, loose_p=0.8))
    return out


@pytest.mark.parametrize("name", list(special_scenes()))
def test_special_scenes_are_valid(name):
    tris, g = special_scenes()[name]
    sc = g.scene(tris, 48)
    if len(tris):
        validate(tris, g, sc)
    if name.startswith("root leaf"):
        _, _, _, used = decode(g.nodes[0])
        assert len(g.nodes) - g.regions[0][2] == 1 and len(used) == 1
    if name == "24-triangle nodes":
        assert any(full_node(n) for n in g.nodes)


def test_knobs_do_what_they_say():
    tris = random_tris(1500, 5)

    def used_slots(g):
        return [[s for s, _ in decode(n)[3]] for n in g.nodes if decode(n)[3]]

    for how, check in (("low", lambda s: s == list(range(len(s)))), ("high", lambda s: s == list(range(8 - len(s), 8)))):
        assert all(check(sorted(s)) for s in used_slots(random_cwbvh(tris, 1, slots=how, node_gaps=0)))
    hist = np.bincount([s for ss in used_slots(random_cwbvh(tris, 1, slots="random")) for s in ss if len(ss) < 8], minlength=8)
    assert hist.min() > 0.5 * hist.mean()                                  # no slot preferred
    g = random_cwbvh(tris, 2)
    assert g.regions[0][2] > 0 and (g.rec_tri < 0).sum() > 24             # poison nodes and gap records
    # leaf ranges: gaps, ranges ending at 24, offsets out of slot order
    gaps = end24 = unordered = 0
    for n in g.nodes:
        leaves = [(s, m & 31, {1: 1, 3: 2, 7: 3}[m >> 5]) for s, m in decode(n)[3] if m != 0x20 | (24 + s)]
        by_off = sorted(leaves, key=lambda x: x[1])
        gaps += bool(by_off) and (any(b[1] > a[1] + a[2] for a, b in zip(by_off, by_off[1:])) or by_off[0][1] > 0)
        end24 += bool(by_off) and by_off[-1][1] + by_off[-1][2] == 24
        unordered += [x[0] for x in by_off] != sorted(x[0] for x in by_off)
    assert gaps and end24 and unordered
    # quantisation: exponents above the tight one, q bytes widened, p below the box minimum, bytes in empty slots
    tight = random_cwbvh(tris, 3, exp_raise=0, loose_p=0, slack=0, empty_fill=False, node_gaps=0)
    loose = random_cwbvh(tris, 3, exp_raise=1.0, loose_p=0, slack=0, empty_fill=False, node_gaps=0)
    assert (loose.nodes[:, 12:15].astype(int) > tight.nodes[:, 12:15]).any(axis=1).mean() > 0.9
    assert ((loose.nodes[:, 12:15].astype(int) - tight.nodes[:, 12:15]) <= 8).all()
    empty = [n for n in g.nodes if len(decode(n)[3]) < 8 and not is_poison(n)]
    assert any(n[32:80].reshape(3, 2, 8)[:, :, [s for s in range(8) if not n[24 + s]]].any() for n in empty)
    assert not random_cwbvh(tris, 2, exact_node=False).nodes[:, 12:15].max() >= EXACT_EXP_BYTE
    assert random_cwbvh(tris, 2, exact_node=True).nodes[:, 12:15].max() >= EXACT_EXP_BYTE
    # node order: child blocks out of BFS order (BFS: child_base grows with the node index)
    for order, want in (("bfs", False), ("dfs", True), ("random", True)):
        g = random_cwbvh(tris, 4, order=order, node_gaps=0)
        bases = [decode(n)[1] for n in g.nodes if decode(n)[0]]
        assert (bases != sorted(bases)) == want, order
    # 24-triangle nodes and single-child chains
    g = random_cwbvh(tris, 6, full=1.0, chain=0.3)
    assert any(full_node(n) for n in g.nodes)
    assert any(decode(n)[0] and len(decode(n)[3]) == 1 for n in g.nodes)
    assert set(KNOBS) >= set(case_knobs(0))


@pytest.mark.parametrize("tlas", [False, True])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_oracle_equals_exhaustive_search(tlas, seed):
    """closest hit over the generated tree == brute force over the records with the poison zeroed (test_oracle's bar), and no
    poison id, on random rays (axis-parallel and bounded ones among them)"""
    from test_oracle import assert_matches_brute_force
    tris, g, sc = make_case(tlas, 48, 100 + seed)
    rays = random_rays(30000, seed, axis_fraction=0.05, bounded_fraction=0.2)
    hits = sc.oracle().trace(rays, stack_limit=KERNEL_STACK)
    poison_free(hits, g, "oracle")
    assert np.array_equal(zeroed_oracle(g, sc).trace(rays, stack_limit=KERNEL_STACK), hits)
    bf, ties = zeroed_oracle(g, sc).brute_force(rays)
    assert_matches_brute_force(hits, bf, ties)
    assert (hits["prim"] != ob.INVALID_PRIM).mean() > 0.2


@pytest.mark.parametrize("tlas", [False, True])
def test_oracle_equals_the_transliteration(tlas):
    """the C oracle and the line-by-line Python reading of the shader (test_oracle.py) on the generated layouts: primitive,
    t bit for bit, and node / triangle / instance visits per ray, with the CPU-vs-HLSL switches set to the shader's side"""
    import hlsl_transliteration as hl
    ob.set_variant(ob.VARIANT_BOX_DIVIDE | ob.VARIANT_TIE_LAST)
    try:
        for seed in (7, 8):
            tris, g, sc = make_case(tlas, 48, seed, n_tris=1000)
            rays = random_rays(150, seed, axis_fraction=0.1, bounded_fraction=0.0)
            hits, cnt, _ = sc.oracle().trace(rays, counts=True)
            hs = hl.Scene(sc.nodes.tobytes(), sc.rec.tobytes(), 48, g.blas, g.tlas_start)
            n_hit = 0
            for i in range(len(rays)):
                if tlas:
                    t, prim, nn, nt, ni = hl.traverse_bvh_tlas(hs, rays["o"][i], rays["d"][i])
                    assert cnt["insts"][i] == ni, i
                else:
                    t, prim, nn, nt = hl.traverse_bvh(hs, rays["o"][i], rays["d"][i])
                assert cnt["nodes"][i] == nn and cnt["tris"][i] == nt, (i, cnt[i], nn, nt)
                if prim < 0:
                    assert hits["prim"][i] == ob.INVALID_PRIM, i
                else:
                    n_hit += 1
                    assert hits["prim"][i] == prim and np.float32(hits["t"][i]).view(np.uint32) == np.float32(t).view(np.uint32), i
            assert n_hit > len(rays) // 10
    finally:
        ob.set_variant(0)


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_hits_identical(gpu, ref, g, what=""):
    poison_free(gpu, g, what)
    assert (gpu["prim"] == ref["prim"]).all(), f"{what}: {(gpu['prim'] != ref['prim']).sum()} primitive ids differ"
    assert (bits(gpu["t"]) == bits(ref["t"])).all(), f"{what}: {(bits(gpu['t']) != bits(ref['t'])).sum()} hit t differ"


def assert_counters(cp, tot, n_rays, what=""):
    assert (cp["rays"], cp["nodes"], cp["tris"], cp["instances"], cp["hits"]) == \
        (n_rays, tot["nodes"], tot["tris"], tot["insts"], tot["hits"]), (what, cp, tot)


def device_trace(sc_gpu, rays, any_hit, timed):
    """tray_cuda_trace_device / _trace_any_device on a caller's torch stream; `timed`: the synchronising form, which also
    publishes the batch's counters"""
    import torch
    d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
    d_hits = torch.empty(len(rays) * 8, dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())                      # the uploads above ran on the current stream
    with torch.cuda.stream(s):
        sc_gpu.traverse_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr(), stream=s.cuda_stream, timed=timed, any_hit=any_hit)
    s.synchronize()
    sc_gpu.sync()
    return d_hits.cpu().numpy().view(ob.HIT_DTYPE)


def check_batch(sc_gpu, orc, g, rays, any_hit, count):
    """the device entry point (on a caller's stream, asynchronous and then timed) and the host entry point; the timed device call
    comes first, so counters left over from an earlier batch (other rays) cannot pass for its own"""
    ref, _, tot = orc.trace(rays, counts=True, any_hit=any_hit, stack_limit=KERNEL_STACK)
    what = "any hit" if any_hit else "closest hit"
    sc_gpu.set_counting(count)
    assert_hits_identical(device_trace(sc_gpu, rays, any_hit, timed=False), ref, g, what + ", device entry point")
    for where, run in (("device entry point", lambda: device_trace(sc_gpu, rays, any_hit, timed=True)),
                       ("host entry point", lambda: sc_gpu.traverse(rays, any_hit=any_hit))):
        assert_hits_identical(run(), ref, g, f"{what}, {where}")
        if count:
            assert_counters(sc_gpu.counters()[0], tot, len(rays), f"{what}, {where}")


def check_frames(sc_gpu, orc, g, tlas_start, count, w=192, h=128):
    view = host.view_from_camera(CAMERA, w, h, tlas_start)
    assert orc.stack_need(ob.primary_rays(view, w, h)).max() <= KERNEL_STACK
    ref = orc.render(view, w, h, 3, rgba=True, stack_limit=KERNEL_STACK)
    assert (ref["primary"]["prim"] != ob.INVALID_PRIM).mean() > 0.05
    flags = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_KEEP_RAYS | (cuda.RENDER_COUNTERS if count else 0)
    for overlap in (0, cuda.RENDER_OVERLAP):
        what = "one-launch frame" if overlap else "two-launch frame"
        sc_gpu.render(view, w, h, 3, flags | overlap)
        sc_gpu.sync()
        out = sc_gpu.download(primary=True, bounce=True, bounce_rays=True, rgba=True)
        assert_hits_identical(out["primary"], ref["primary"], g, what + ", primary")
        assert (out["bounce_rays"].view(np.uint32) == ref["bounce_rays"].view(np.uint32)).all(), what + ": bounce rays differ"
        assert_hits_identical(out["bounce"], ref["bounce"], g, what + ", bounce")
        assert np.abs(out["rgba"].reshape(-1, 4).astype(int) - ref["rgba"].astype(int)).max() <= 1
        if count:
            cp, cb = sc_gpu.counters()
            for got, want in ((cp, ref["primary_totals"]), (cb, ref["bounce_totals"])):
                assert (got["rays"], got["hits"], got["nodes"], got["tris"], got["instances"]) == \
                    (want["rays"], want["hits"], want["nodes"], want["tris"], want["insts"]), (what, got, want)


VARIANTS = list(range(1, 16))                                          # every combination of the four TRAY_VARIANT_* switches


@pytest.mark.gpu
@pytest.mark.parametrize("k", KERNELS, ids=kernel_id)
def test_instantiation_matches_the_oracle_on_generated_trees(k):
    tlas, count, stride, kind, mode = k
    seed = case_seed(k)
    tris, g, sc = make_case(tlas, stride, seed)
    rays = case_rays(seed)
    orc = sc.oracle()
    assert orc.stack_need(rays, any_hit=kind == "any").max() <= KERNEL_STACK
    gpu = sc.cuda()
    try:
        if mode == 1:
            try:
                for v in VARIANTS:
                    ob.set_variant(v)
                    gpu.set_variant(v)
                    assert_hits_identical(gpu.traverse(rays), orc.trace(rays, stack_limit=KERNEL_STACK), g, f"variant {v:#x}")
            finally:
                ob.set_variant(0)
        elif kind == "frame":
            check_frames(gpu, orc, g, g.tlas_start, count)
        else:
            check_batch(gpu, orc, g, rays, kind == "any", count)
            check_batch(gpu, orc, g, case_rays(seed + 1000, (1 << 18) + 77), kind == "any", count)    # the copy pipeline
        gpu.sync()
    finally:
        gpu.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(special_scenes()))
@pytest.mark.parametrize("stride", [48, 24])
def test_special_scenes_match_the_oracle(name, stride):
    tris, g = special_scenes()[name]
    sc = g.scene(tris, stride)
    orc = sc.oracle()
    rays = case_rays(7)
    gpu = sc.cuda()
    try:
        for any_hit in (False, True):
            check_batch(gpu, orc, g, rays, any_hit, count=not any_hit)
        if len(tris) > 3:
            check_frames(gpu, orc, g, 0, True)
    finally:
        gpu.close()


@pytest.mark.gpu
@pytest.mark.parametrize("knob,value", [("TRAY_CUDA_TRI_WEIGHT", 1), ("TRAY_CUDA_TRI_WEIGHT", 64), ("TRAY_CUDA_REFILL_MIN", 1),
                                        ("TRAY_CUDA_REFILL_MIN", 32), ("TRAY_CUDA_GEN_MIN", 1), ("TRAY_CUDA_GEN_MIN", 32)])
@pytest.mark.parametrize("tlas", [False, True])
def test_scheduler_extremes_on_a_generated_tree(monkeypatch, knob, value, tlas):
    monkeypatch.setenv(knob, str(value))
    tris, g, sc = make_case(tlas, 48, 77)
    orc = sc.oracle()
    gpu = sc.cuda()
    try:
        check_batch(gpu, orc, g, case_rays(78), False, True)
        check_batch(gpu, orc, g, case_rays(79), True, False)
        check_frames(gpu, orc, g, g.tlas_start, True)
    finally:
        gpu.close()


@pytest.mark.gpu
def test_a_batch_beyond_one_launch_keeps_its_hits_and_counters():
    """trace_device splits a batch into launches of 2^30 rays (the kernel keeps two tag bits above the ray index); the counters
    of one batch accumulate over its launches.  2^16 distinct rays tiled to 2^30 + 2^16 + 5 rays (34 GB of rays, 8.6 GB of hits),
    compared on the device with the tiled oracle result."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < (48 << 30):
        pytest.skip(f"needs about 48 GB of free device memory, {free / 2**30:.1f} GB free")
    tris = random_tris(300, 90)
    g = random_cwbvh(tris, 90, slots="mix")
    sc = g.scene(tris, 48)
    base = case_rays(91, 1 << 16)
    ref, _, tot = sc.oracle().trace(base, counts=True, stack_limit=KERNEL_STACK)
    _, _, tail_tot = sc.oracle().trace(base[:5], counts=True, stack_limit=KERNEL_STACK)
    reps, n = (1 << 14) + 1, (1 << 30) + (1 << 16) + 5
    gpu = sc.cuda()
    d_rays = d_hits = None
    try:
        d_base = torch.from_numpy(base.view(np.uint8).copy()).cuda().view(1 << 16, 32)
        d_rays = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
        d_rays[:reps << 16].view(reps, 1 << 16, 32).copy_(d_base.expand(reps, -1, -1))
        d_rays[reps << 16:].copy_(d_base[:5])
        d_hits = torch.full((n, 8), 0xFF, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()                                     # the fills ran on torch's stream, the trace runs on the scene's
        gpu.set_counting(True)
        gpu.traverse_device(d_rays.data_ptr(), n, d_hits.data_ptr(), timed=True)
        want = torch.from_numpy(ref.view(np.int64).copy()).cuda()
        got = d_hits.view(torch.int64).view(-1)
        assert bool((got[:reps << 16].view(reps, 1 << 16) == want).all())
        assert bool((got[reps << 16:] == want[:5]).all())
        cp, _ = gpu.counters()
        assert_counters(cp, {k: v * reps + tail_tot[k] for k, v in tot.items()}, n)
    finally:
        del d_rays, d_hits
        gpu.close()
        torch.cuda.empty_cache()
