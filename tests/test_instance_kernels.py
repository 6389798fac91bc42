"""The 12 instanced trace_kernel instantiations (INST: two-level, MODE 0, closest or any hit x counting x stride 24 / 48 / 64)
where they can go wrong, and the instanced bounce normal at the exponent edges of f32.

1. Generated trees (tests/cwbvh_bytes.py, TLAS moved to the tail of the node array): BLAS layouts neither builder writes, poison
   in the bytes a correct traversal never reads, exact-node exponents, hundreds of instances over them, the scheduler's extremes.
2. Deep BLAS inside instances (the ladders of test_deep_stack.py): an instance entered with TLAS entries on the stack, whose
   descent reaches the spill region, the last stack entry and the overflow status.
3. Objects of size 2^k, k in +-{8, 16, 24, 32}, placed at world size ~1 by powers of two, rotations, signed axis permutations, an
   ill-conditioned diagonal, strong shear and far translations.  Hits and bounce rays are held to tests/instance_ref.c bit for
   bit, and both to a float64 evaluation in world space.

Every kernel result is compared with instance_ref.c (`Reference` of test_instances.py) bit for bit; the float64 checks hold that
reference, and so the kernels, to the geometry itself."""
import os
import re

import numpy as np
import pytest

import cwbvh_bytes as cb
import oracle_binding as ob
from conftest import ROOT, random_rays
from test_build_reference import many_small_objects
from test_cwbvh_fuzz import KERNELS as PLAIN_KERNELS, case_knobs
from test_deep_stack import DIAGONAL_CAMERA, blas_ladder, ladder_rays
from test_device_primitives import hash_noise_np
from test_hit_attributes import reference as attr_reference, same_bytes
from test_instances import (FLAGS, F32_MAX, INVALID, KERNEL_STACK, Reference, brute_force, check_frame, instance_boxes,
                            reference_frame, rotation, same_hits, xforms)
from test_refit_tlas import tlas_at_the_tail, tlas_reference
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu
STRIDES = (24, 48, 64)
# (TLAS, COUNT, STRIDE, ANYHIT, FRAME, MODE, INST): the template arguments of every INST instantiation of trace_kernel
INST_KERNELS = [(True, count, stride, any_hit, False, 0, True) for count in (False, True) for stride in STRIDES for any_hit in (False, True)]


def kernel_id(k):
    return f"{'count' if k[1] else 'nocount'}-{k[2]}-{'any' if k[3] else 'closest'}"


# ---- CPU: the kernel table ---------------------------------------------------------------------------------------------------


def test_the_inst_table_is_what_pick_kernel_selects():
    """12 distinct instantiations, none of them among the 42 of test_cwbvh_fuzz.py, and exactly the ones pick_kernel's INST
    branch names for COUNT in {false, true} and STRIDE in {24, 48, 64}"""
    assert len(INST_KERNELS) == 12 and len(set(INST_KERNELS)) == 12 and len({kernel_id(k) for k in INST_KERNELS}) == 12
    plain = {(t, c, s, kind == "any", kind == "frame", m, False) for t, c, s, kind, m in PLAIN_KERNELS}
    assert len(plain) == 42 and not plain & set(INST_KERNELS)
    src = open(os.path.join(ROOT, "tray_racing_b200", "csrc", "tray_cuda.cu")).read()
    body = re.search(r"kernel_fn pick_kernel\(bool anyhit, bool frame, bool variant, bool inst\) \{(.*?)\n\}", src, re.S).group(1)
    branch = re.search(r"if \(inst\) return anyhit \? (.*?) : (.*?);", body, re.S)
    args = [re.sub(r"\s+", "", re.search(r"trace_kernel<(.*?)>", b).group(1)).split(",") for b in branch.groups()]
    assert args == [["true", "COUNT", "STRIDE", "true", "false", "0", "true"], ["true", "COUNT", "STRIDE", "false", "false", "0", "true"]]
    assert "if constexpr (TLAS)" in body                                      # only two-level launches reach it
    for s in STRIDES:
        assert f"pick_kernel<TLAS, COUNT, {s}>(anyhit, frame, variant, inst)" in src
    for c in ("true", "false"):
        assert f"pick_kernel<true, {c}>(stride, anyhit, frame, variant, inst)" in src
    picked = {(True, c, s, a, False, 0, True) for c in (False, True) for s in STRIDES for a in (True, False)}
    assert picked == set(INST_KERNELS)


# ---- shared pieces -----------------------------------------------------------------------------------------------------------


def inverse_f32(xf):
    """world_to_object as set_instances computes it: adjugate over determinant in double, rounded to f32"""
    m = np.asarray(xf, np.float32).astype(np.float64)
    A = m[:, :, :3]
    adj = np.stack([np.cross(A[:, 1], A[:, 2]), np.cross(A[:, 2], A[:, 0]), np.cross(A[:, 0], A[:, 1])], axis=2)
    W = adj / np.einsum("ni,ni->n", A[:, 0], adj[:, :, 0])[:, None, None]
    return np.concatenate([W, -np.einsum("nij,nj->ni", W, m[:, :, 3])[:, :, None]], axis=2).astype(np.float32)


def cpu_reference(nodes, rec, stride, ts, roots, xf, max_leaf=3):
    """the Reference of a scene after set_instances(roots, xf), built on the CPU: the TLAS of tlas_reference over the box rule of
    include/tray_cuda.h, written at ts (test_instances.check_tlas holds the device to exactly this TLAS)"""
    nodes = np.asarray(nodes, np.uint8).reshape(-1, 80)[:ts]
    lo, hi = instance_boxes(nodes, roots, xf)
    top, perm, _ = tlas_reference(lo, hi, max_leaf)
    return Reference(np.concatenate([nodes, top]), rec, stride, np.asarray(roots, np.uint32)[perm], ts, inverse_f32(xf), perm)


def device_trace(sc, rays, any_hit, timed=True):
    """traverse_instance_device on device buffers: (hits, ids)"""
    import torch
    d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
    d_hits = torch.zeros(rays.size * 8, dtype=torch.uint8, device="cuda")
    d_ids = torch.zeros(rays.size, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    sc.traverse_instance_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr(), d_ids.data_ptr(), timed=timed, any_hit=any_hit)
    sc.sync()
    return d_hits.cpu().numpy().view(ob.HIT_DTYPE), d_ids.cpu().numpy().view(np.uint32)


def check_costs(costs, cnt, peak, what=""):
    for a, b in (("nodes", "nodes"), ("tris", "tris"), ("instances", "insts")):
        assert np.array_equal(costs[a], cnt[b]), f"{what}: per-ray {a} differ on {(costs[a] != cnt[b]).sum()} rays"
    assert np.array_equal(costs["stack"], peak), f"{what}: per-ray stack peaks differ on {(costs['stack'] != peak).sum()} rays"


def check_counters(tot, cnt, n, hits, what=""):
    assert (tot["rays"], tot["nodes"], tot["tris"], tot["instances"], tot["hits"]) == \
        (n, int(cnt["nodes"].sum()), int(cnt["tris"].sum()), int(cnt["insts"].sum()), int((hits["prim"] != INVALID).sum())), (what, tot)


def run_kernel(sc, ref, rays, count, any_hit, what="", device=True, poison=None):
    """one INST kernel (count, any_hit) on `rays` through the host path (and the device path): hits and ids equal to the
    reference, no poison id, and for the counting kernel per-ray costs and counters equal to the reference's"""
    want, wid, cnt, peak = ref.trace(rays, any_hit, cap=KERNEL_STACK)
    if poison is not None:
        assert not np.isin(want["prim"], poison).any(), "the reference read a poison record"
    sc.set_counting(count)
    runs = [("host", lambda: sc.traverse_instance(rays, any_hit=any_hit))]
    if device:
        runs.append(("device", lambda: device_trace(sc, rays, any_hit)))
    for where, run in runs:
        hits, ids = run()
        if poison is not None:
            assert not np.isin(hits["prim"], poison).any(), f"{what}, {where}: a poison id came back"
        assert same_hits(hits, want), f"{what}, {where}: {(hits['prim'] != want['prim']).sum()} hits differ"
        assert np.array_equal(ids, wid), f"{what}, {where}: {(ids != wid).sum()} instance ids differ"
        if count:
            check_counters(sc.counters()[0], cnt, rays.size, want, f"{what}, {where}")
    if count:
        h2, costs = sc.traverse_cost(rays, any_hit=any_hit)
        assert same_hits(h2, want), what
        check_costs(costs, cnt, peak, what)
    sc.set_counting(False)
    return want, wid, peak


# ---- 1. generated trees ------------------------------------------------------------------------------------------------------


def generated_instances(stride, seed, n_inst=300):
    """(Generated, Scene, node bytes with the TLAS at the tail, blas_offsets, tlas_start, the object roots, roots and transforms
    of n_inst instances): shared BLAS, every transform kind of test_instances.xforms"""
    tris = cb.random_tris(1200, seed)
    tris, off = cb.random_objects(tris, 4 + seed % 6, seed)
    g = cb.random_tlas(tris, off, seed, **case_knobs(seed))
    s = g.scene(tris, stride, seed)
    nodes, blas, ts = tlas_at_the_tail(g)
    m = g.regions[-1][1]
    objects = np.array([b if b < g.tlas_start else b - m for b, _, _, _ in g.regions[:-1]], np.uint32)
    rng = np.random.default_rng(seed)
    roots = rng.choice(objects, n_inst).astype(np.uint32)
    kinds = ["identity", "translation", "rotation", "uniform", "nonuniform", "mirror", "shear", "mixed"]
    xf = np.concatenate([xforms(k, n, seed + i) for i, (k, n) in enumerate(zip(kinds, np.diff(np.linspace(0, n_inst, len(kinds) + 1).astype(int))))])
    return g, s, nodes, blas, ts, objects, roots, xf


def instance_rays(tris, offs, roots, xf, n, seed):
    """rays aimed at instances through their world-space triangles, rays from inside instances, random rays with axis-parallel
    and bounded [tmin, tmax] ones"""
    rng = np.random.default_rng(seed)
    m = xf.astype(np.float64)
    k = rng.integers(0, roots.size, n)
    t3 = np.asarray(tris, np.float64).reshape(-1, 3, 3)
    lo, hi = offs[roots[k]].astype(np.int64), offs[roots[k] + 1].astype(np.int64)
    j = lo + (rng.random(n) * (hi - lo)).astype(np.int64)
    c = np.einsum("nij,nj->ni", m[k, :, :3], t3[j].mean(axis=1)) + m[k, :, 3]
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    at = np.zeros(n, ob.RAY_DTYPE)
    at["o"] = (c - 3 * d).astype(np.float32); at["d"] = d.astype(np.float32); at["tmax"] = F32_MAX
    inside = at.copy(); inside["o"] = c.astype(np.float32)
    return np.concatenate([at, inside, random_rays(n, seed, lo=-3.0, hi=3.0, axis_fraction=0.05, bounded_fraction=0.15)])


@gpu
@pytest.mark.parametrize("k", INST_KERNELS, ids=kernel_id)
def test_inst_kernel_on_generated_trees(k):
    _, count, stride, any_hit, _, _, _ = k
    seed = INST_KERNELS.index(k) + 201
    g, s, nodes, blas, ts, objects, roots, xf = generated_instances(stride, seed)
    sc = cuda.TrayCudaScene(nodes, s.rec, stride, blas, ts)
    try:
        sc.set_instances(roots, xf, max_prims_per_leaf=1 if seed % 2 else 3)
        assert sc.exact_node_test() == case_knobs(seed)["exact_node"]
        ref = Reference.of(sc)
        # rays at instances need each BLAS's triangles: the records it reaches
        per_root = [s.tris.reshape(-1, 9)[reachable_records(nodes, int(r), g)] for r in objects]
        offs = np.concatenate([[0], np.cumsum([len(t) for t in per_root])]).astype(np.int64)
        obj_of = np.array([objects.tolist().index(r) for r in roots.tolist()])
        rays = instance_rays(np.concatenate(per_root), offs, obj_of, xf, 4000, seed)
        want, wid, peak = run_kernel(sc, ref, rays, count, any_hit, kernel_id(k), poison=g.poison_ids())
        assert (want["prim"] != INVALID).sum() > 3000 and np.unique(wid[wid != INVALID]).size > 100
        big = np.concatenate([rays, random_rays((1 << 18) - rays.size + 77, seed + 1, lo=-3.0, hi=3.0, axis_fraction=0.05,
                                                bounded_fraction=0.15)])
        run_kernel(sc, ref, big, count, any_hit, kernel_id(k) + ", pipelined", device=False, poison=g.poison_ids())
    finally:
        sc.close()


def reachable_records(nodes, root, g):
    """the triangle records a BLAS reaches from `root` (node indices relative to it), poison records excluded"""
    nodes = np.asarray(nodes, np.uint8).reshape(-1, 80)
    out, todo = [], [0]
    while todo:
        j = todo.pop()
        imask, cb_, pb, used = cb.decode(nodes[root + j])
        for slot, meta in used:
            if imask >> slot & 1:
                todo.append(cb_ + bin(imask & ((1 << slot) - 1)).count("1"))
            else:
                n = {1: 1, 3: 2, 7: 3}[meta >> 5]
                out.extend(range(pb + (meta & 31), pb + (meta & 31) + n))
    out = np.array(sorted(set(out)), np.int64)
    return out[g.rec_tri[out] >= 0]


@gpu
@pytest.mark.parametrize("knob,value", [("TRAY_CUDA_TRI_WEIGHT", 1), ("TRAY_CUDA_TRI_WEIGHT", 64), ("TRAY_CUDA_REFILL_MIN", 1),
                                        ("TRAY_CUDA_REFILL_MIN", 32)])
def test_inst_kernels_at_scheduler_extremes(monkeypatch, knob, value):
    monkeypatch.setenv(knob, str(value))                                      # read when the scene is created
    seed = 251 + value
    g, s, nodes, blas, ts, objects, roots, xf = generated_instances(48, seed)
    sc = cuda.TrayCudaScene(nodes, s.rec, 48, blas, ts)
    try:
        sc.set_instances(roots, xf)
        ref = Reference.of(sc)
        rays = random_rays(30000, seed, lo=-3.0, hi=3.0, axis_fraction=0.05, bounded_fraction=0.15)
        for count, any_hit in ((True, False), (False, True)):
            run_kernel(sc, ref, rays, count, any_hit, f"{knob}={value}", poison=g.poison_ids())
    finally:
        sc.close()


def test_generated_instance_cases_are_valid():
    """the generated scenes the GPU tests instance: every object root is a BLAS root of the tail layout, the CPU-built reference
    of the instanced scene reads no poison record and hits often, and exact_node where the knobs ask for it"""
    for k in INST_KERNELS[:4]:
        seed = INST_KERNELS.index(k) + 201
        g, s, nodes, blas, ts, objects, roots, xf = generated_instances(k[2], seed)
        assert set(objects.tolist()) <= set(blas.tolist()) and np.unique(roots).size == objects.size
        assert (nodes[:ts, 12:15].max() >= cb.EXACT_EXP_BYTE) == case_knobs(seed)["exact_node"]
        ref = cpu_reference(nodes, s.rec, k[2], ts, roots, xf, 1 if seed % 2 else 3)
        rays = random_rays(20000, seed, lo=-3.0, hi=3.0, axis_fraction=0.05, bounded_fraction=0.15)
        hits, ids, _, peak = ref.trace(rays, k[3])
        assert not np.isin(hits["prim"], g.poison_ids()).any()
        assert (hits["prim"] != INVALID).mean() > 0.2 and peak.max() <= KERNEL_STACK


# ---- 2. deep BLAS inside instances -------------------------------------------------------------------------------------------


def ladder_instances(D, stride=48):
    """blas_ladder(D)'s nodes and records (the D-level ladder at root blas[1], an 8-level one at blas[0], TLAS at the tail)
    with the deep ladder placed five times, overlapping along the diagonal, and the shallow one twice"""
    sc = blas_ladder(D, stride)
    deep, shallow = int(sc.blas[1]), int(sc.blas[0])
    roots = np.array([deep] * 5 + [shallow] * 2, np.uint32)
    xf = np.tile(np.eye(3, 4), (roots.size, 1, 1))
    xf[1, :, 3] = 0.004; xf[2, :, 3] = -0.003                                  # along the diagonal
    xf[3, :, :3] *= 1.01; xf[4, :, :3] *= 0.995                                # scaled about the ladder's apex
    xf[5, :, 3] = (0.002, -0.001, 0.0); xf[6, :, :3] *= 0.99
    return sc, roots, xf.astype(np.float32)


LADDER_DEPTHS = {"spill": 13, "last entry": 48}      # D of the clean cases (the rays peak at D: D - 1 ladder entries, one TLAS entry)
OVERFLOW_D = 50


def ladder_batch(sc, seed, n=8192):
    return ladder_rays(n, seed, sc.tris, tmin_fraction=0.3)


def test_instanced_ladders_reach_every_stack_boundary():
    """the reference peaks of the GPU cases below: 12 and 13 (shared memory to the spill array), 47 and 48 (the last entries)
    in the clean batches, and more than 48 in the overflow batch"""
    peaks = []
    for name, D in LADDER_DEPTHS.items():
        sc, roots, xf = ladder_instances(D)
        ref = cpu_reference(sc.nodes, sc.rec, 48, sc.tlas_start, roots, xf)
        _, ids, _, peak = ref.trace(ladder_batch(sc, D), cap=KERNEL_STACK)
        assert np.unique(ids).size >= 6, name
        peaks.append(peak)
    peaks = np.concatenate(peaks)
    for need in (12, 13, 47, 48):
        assert (peaks == need).any(), (need, np.unique(peaks))
    sc, roots, xf = ladder_instances(OVERFLOW_D)
    ref = cpu_reference(sc.nodes, sc.rec, 48, sc.tlas_start, roots, xf)
    peak = ref.trace(ladder_batch(sc, OVERFLOW_D), cap=ob.STACK_MAX)[3]
    assert peak.max() > KERNEL_STACK and (peak <= KERNEL_STACK).mean() > 0.5
    with pytest.raises(RuntimeError):
        ref.trace(ladder_batch(sc, OVERFLOW_D), cap=KERNEL_STACK)


@gpu
@pytest.mark.parametrize("stride", STRIDES)
def test_deep_blas_inside_instances(stride):
    for name, D in LADDER_DEPTHS.items():
        sc, roots, xf = ladder_instances(D, stride)
        g = sc.cuda()
        try:
            g.set_instances(roots, xf)
            ref = Reference.of(g)
            rays = ladder_batch(sc, D)
            for count in (False, True):
                for any_hit in (False, True):
                    _, _, peak = run_kernel(g, ref, rays, count, any_hit, f"{name}, count={count}, any_hit={any_hit}")
                    assert peak.max() == D
        finally:
            g.close()


def expect_overflow():
    return pytest.raises(cuda.TrayCudaError, match=r"error -4\b")


@gpu
def test_deep_blas_overflow_is_reported_once():
    import torch
    sc, roots, xf = ladder_instances(OVERFLOW_D)
    g = sc.cuda()
    try:
        g.set_instances(roots, xf)
        ref = Reference.of(g)
        rays = ladder_batch(sc, OVERFLOW_D)
        peak = ref.trace(rays, cap=ob.STACK_MAX)[3]
        clean = rays[peak <= KERNEL_STACK]
        assert peak.max() > KERNEL_STACK and clean.size > rays.size // 2
        want, wid, _, _ = ref.trace(clean)
        for any_hit in (False, True):
            if ref.trace(rays, any_hit, cap=ob.STACK_MAX)[3].max() > KERNEL_STACK:
                with expect_overflow():
                    g.traverse_instance(rays, any_hit=any_hit)
            w2, i2, _, _ = ref.trace(clean, any_hit)
            h, i = g.traverse_instance(clean, any_hit=any_hit)
            assert same_hits(h, w2) and np.array_equal(i, i2), f"clean batch after the overflow, any_hit={any_hit}"
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_hits = torch.empty(rays.size * 8, dtype=torch.uint8, device="cuda")
        d_ids = torch.empty(rays.size, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        g.traverse_instance_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr(), d_ids.data_ptr())    # nothing to report yet ..
        with expect_overflow():
            g.sync()                                                         # .. the synchronising call reports it
        g.sync()                                                             # once
        h, i = device_trace(g, clean, False)
        assert same_hits(h, want) and np.array_equal(i, wid), "clean device batch after the overflow"
    finally:
        g.close()


@gpu
@pytest.mark.parametrize("refill_min", [1, 32])
def test_any_hit_refill_from_the_spill_region_inside_instances(monkeypatch, refill_min):
    monkeypatch.setenv("TRAY_CUDA_REFILL_MIN", str(refill_min))
    sc, roots, xf = ladder_instances(LADDER_DEPTHS["last entry"])
    deep = ladder_rays(20000, 7, sc.tris, spread=(1e-5, 3e-3))
    shallow = ladder_rays(20000, 8, sc.tris, spread=(0.05, 0.5))
    rays = np.empty(40000, ob.RAY_DTYPE)
    rays[0::2], rays[1::2] = deep, shallow
    g = sc.cuda()
    try:
        g.set_instances(roots, xf)
        ref = Reference.of(g)
        _, _, peak = run_kernel(g, ref, rays, False, True, "any hit", device=False)
        assert peak.max() >= 40 and (peak < 12).sum() > 1000
        run_kernel(g, ref, np.tile(rays, 7), False, True, "any hit, pipelined", device=False)
    finally:
        g.close()


@gpu
@pytest.mark.parametrize("stride", STRIDES)
def test_frame_down_an_instanced_ladder(stride):
    w, h = 192, 128
    sc, roots, xf = ladder_instances(LADDER_DEPTHS["last entry"], stride)
    g = sc.cuda()
    try:
        g.set_instances(roots, xf)
        view = host.view_from_camera(DIAGONAL_CAMERA, w, h)
        want = reference_frame(Reference.of(g), view, w, h)
        assert want["pcost"][1].max() >= 40 and want["shoot"].sum() > 1000
        g.set_ray_cost(True)
        g.render(view, w, h, 0, FLAGS)
        g.sync()
        check_frame(g, want)
    finally:
        g.close()


# ---- 3. extreme but accepted transforms -------------------------------------------------------------------------------------

SCALES = (-32, -24, -16, -8, 8, 16, 24, 32)
KINDS = ("pow2", "pow2 rotated", "permutation", "ill-conditioned", "shear", "far")
PER_KIND = 8
# relative bound on t of unique, non-grazing hits against float64, by kind: 1e-5 for the well-conditioned kinds; the others
# multiply it by the condition number of the 3x3 part (shear; the ill-conditioned diagonal is exact in f32 both ways, its bound
# is stated at its condition number all the same) or by |translation| / object world size (far: the f32 origin and the
# cancellation in o' = W o + W_3 carry an absolute error of ~2^-24 |translation|)
T_REL = 1e-5


def extreme_case(k, n_obj=12, seed=0):
    """(object-space triangles (n, 9) of objects of size ~2^k, object offsets, roots, object_to_world (f32), kind of each
    instance, t bound of each instance): every object placed at world size ~1 by every kind of KINDS"""
    tris, offs = many_small_objects(n_obj, seed=seed + 5)
    t3 = tris.reshape(-1, 3, 3).astype(np.float64)
    obj = np.empty_like(t3)
    s = np.ldexp(1.0, k)
    for o in range(n_obj):
        a, b = int(offs[o]), int(offs[o + 1])
        c = t3[a:b].reshape(-1, 3).mean(axis=0)
        obj[a:b] = (t3[a:b] - c) * 25.0 * s                                    # 0.04 wide: ~2^k in object space
    rng = np.random.default_rng(seed + k + 100)
    roots, xf, kinds, bound = [], [], [], []
    grid = np.stack(np.meshgrid(*[np.arange(4)] * 3, indexing="ij"), -1).reshape(-1, 3) * 1.25 - 1.875
    cells = rng.permutation(len(grid))
    for ki, kind in enumerate(KINDS):
        for i in range(PER_KIND):
            A = np.eye(3)
            if kind == "pow2 rotated":
                A = rotation(rng)
            elif kind == "permutation":
                A = np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]
            elif kind == "ill-conditioned":
                A = np.diag([2.0 ** -12, 1.0, 2.0 ** 12])[rng.permutation(3)] * 2.0 ** int(rng.integers(-2, 3))
            elif kind == "shear":
                A = np.eye(3) + np.triu(rng.choice([-4.0, 4.0], (3, 3)), 1)
            else:
                A = np.diag(2.0 ** rng.integers(-1, 2, 3).astype(float))
            M = np.zeros((3, 4))
            M[:, :3] = A / s
            t = grid[cells[ki * PER_KIND + i]]
            cond = np.linalg.cond(A)
            b = T_REL * (cond if kind in ("ill-conditioned", "shear") else 1.0)
            if kind == "far":
                t = t + rng.choice([-1.0, 1.0], 3) * 1e4 * rng.uniform(1, 2, 3)
                b = T_REL * (1 + np.abs(t).max())
            M[:, 3] = t
            roots.append(int(rng.integers(0, n_obj))); xf.append(M); kinds.append(kind); bound.append(b)
    return obj.reshape(-1, 9).astype(np.float32), offs, np.array(roots, np.uint32), np.array(xf).astype(np.float32), np.array(kinds), np.array(bound)


def extreme_rays(tris, offs, roots, xf, kinds, n, seed):
    """rays at points inside the world-space triangles of random instances (from 5 world units away, or 5 % of that for the
    far kind: f32 origins near 1e4), and axis-parallel rays at the permuted instances (exact zero object-space components)"""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, roots.size, n)
    perm = np.flatnonzero(kinds == "permutation")
    k[: n // 5] = perm[rng.integers(0, perm.size, n // 5)]
    lo, hi = offs[roots[k]].astype(np.int64), offs[roots[k] + 1].astype(np.int64)
    j = lo + (rng.random(n) * (hi - lo)).astype(np.int64)
    b = rng.uniform(0.1, 0.8, (n, 2)); b[b.sum(1) > 0.9] *= 0.45
    t3 = np.asarray(tris, np.float32).reshape(-1, 3, 3).astype(np.float64)[j]
    p = t3[:, 0] + b[:, :1] * (t3[:, 1] - t3[:, 0]) + b[:, 1:] * (t3[:, 2] - t3[:, 0])
    m = xf.astype(np.float64)
    target = np.einsum("nij,nj->ni", m[k, :, :3], p) + m[k, :, 3]
    d = rng.normal(size=(n, 3))
    ax = rng.integers(0, 3, n // 5)
    d[: n // 5] = 0; d[np.arange(n // 5), ax] = rng.choice([-1.0, 1.0], n // 5)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    dist = np.where(kinds[k] == "far", 0.25, 5.0)[:, None]
    rays = np.zeros(n, ob.RAY_DTYPE)
    rays["o"] = (target - dist * d).astype(np.float32); rays["d"] = d.astype(np.float32); rays["tmax"] = F32_MAX
    return rays


def check_hits_float64(hits, ids, rays, case, pi=None):
    """unique non-grazing hits: instance and triangle of a float64 world-space brute force, t within the kind's bound"""
    tris, offs, roots, xf, kinds, bound = case
    t, inst, tri, second, cos = brute_force(tris, offs, roots, xf, rays)
    unique = np.isfinite(t) & (second > t * (1 + 1e-5) + 1e-12) & (cos > 0.1)
    assert unique.sum() > rays.size // 3
    assert np.array_equal(ids[unique], inst[unique]), f"{(ids[unique] != inst[unique]).sum()} instances differ from float64"
    prim = hits["prim"][unique] if pi is None else pi[hits["prim"][unique]]
    assert np.array_equal(prim, tri[unique]), "triangles differ from float64"
    err = np.abs(hits["t"][unique].astype(np.float64) - t[unique]) / t[unique]
    lim = bound[inst[unique]]
    worst = np.argmax(err / lim)
    assert (err <= lim).all(), f"t off by {err[worst]:.3g} relative on a {kinds[inst[unique]][worst]} instance (bound {lim[worst]:.3g})"
    for kind in KINDS:
        assert (kinds[inst[unique]] == kind).sum() > 20, kind


def world_normals(tris, roots, xf, prim, ids, pi=None):
    """float64 world-space normal of hit triangle prim in instance ids: M^-T cross(e1, e2), unit length"""
    t3 = np.asarray(tris, np.float32).reshape(-1, 3, 3).astype(np.float64)
    j = prim if pi is None else pi[prim]
    e1, e2 = t3[j, 0] - t3[j, 1], t3[j, 2] - t3[j, 0]
    n = np.cross(e1, e2)
    A = xf.astype(np.float64)[ids, :, :3]
    n = np.einsum("nji,nj->ni", np.linalg.inv(A), n)                          # inverse transpose of object_to_world
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def check_ng(attrs, hits, ids, case, pi=None):
    """the attribute normal is finite, nonzero and parallel to the float64 world normal"""
    tris, offs, roots, xf, kinds, bound = case
    hit = hits["prim"] != INVALID
    ng = attrs["ng"][hit].astype(np.float64)
    assert np.isfinite(ng).all() and (np.abs(ng).max(axis=1) > 0).all()
    want = world_normals(tris, roots, xf, hits["prim"][hit], ids[hit], pi)
    cos = np.abs((ng / np.linalg.norm(ng, axis=1, keepdims=True) * want).sum(1))
    assert cos.min() >= 1 - 1e-6, f"ng off the float64 normal by 1 - cos = {1 - cos.min():.3g}"


def check_bounce_float64(brays, prays, hits, ids, view, w, case, pi=None, fc=0):
    """bounce directions of primary hits: finite, unit length within 1e-6, in the hemisphere of the float64 world normal facing
    the primary ray, within 2e-6 of a float64 evaluation of the same sampler (test_device_primitives' formula) — scaled by the
    condition number for the ill-conditioned and shear kinds"""
    tris, offs, roots, xf, kinds, bound = case
    hit = np.flatnonzero(hits["prim"] != INVALID)
    assert hit.size > 500
    d = brays["d"][hit].astype(np.float64)
    assert np.isfinite(d).all(), f"{(~np.isfinite(d).all(axis=1)).sum()} bounce directions are not finite"
    assert np.abs(np.linalg.norm(d, axis=1) - 1).max() <= 1e-6
    nf = world_normals(tris, roots, xf, hits["prim"][hit], ids[hit], pi)
    pd = prays["d"][hit].astype(np.float64)
    nf *= np.where((nf * -pd).sum(1) >= 0, 1.0, -1.0)[:, None]
    keep = np.abs(nf[:, 2] + 1) > 1e-3                                         # away from the basis singularity nz = -1
    px, py = (hit % w).astype(np.uint32), (hit // w).astype(np.uint32)
    f = np.full(hit.size, fc, np.uint32)
    u0, u1 = hash_noise_np(px, py, f).astype(np.float64), hash_noise_np(px, py, f + np.uint32(1024)).astype(np.float64)
    l = np.stack([np.sqrt(u0) * np.cos(2 * np.pi * u1), np.sqrt(u0) * np.sin(2 * np.pi * u1), np.sqrt(np.maximum(0, 1 - u0))], 1)
    sign = np.where(nf[:, 2] >= 0, 1.0, -1.0)
    a = -1.0 / (sign + nf[:, 2])
    b = nf[:, 0] * nf[:, 1] * a
    b1 = np.stack([1 + sign * nf[:, 0] ** 2 * a, sign * b, -sign * nf[:, 0]], 1)
    b2 = np.stack([b, sign + nf[:, 1] ** 2 * a, -nf[:, 1]], 1)
    want = b1 * l[:, :1] + b2 * l[:, 1:2] + nf * l[:, 2:3]
    want /= np.linalg.norm(want, axis=1, keepdims=True)
    k = kinds[ids[hit]]
    cond = np.array([np.linalg.cond(xf[i, :, :3].astype(np.float64)) for i in range(len(xf))])[ids[hit]]
    lim = 2e-6 * np.where(np.isin(k, ("ill-conditioned", "shear")), cond, 1.0)
    err = np.abs(d - want).max(axis=1)
    assert (err[keep] <= lim[keep]).all(), f"bounce direction off float64 by {err[keep].max():.3g} ({k[keep][np.argmax(err[keep] / lim[keep])]})"
    assert ((d * nf).sum(1) >= -1e-6).all(), "a bounce direction leaves the hemisphere"


EXTREME_CAMERA = host.Camera((5.0, 4.0, 6.5), (0.0, 0.0, 0.0), 45.0)


@pytest.mark.parametrize("k", SCALES)
def test_reference_against_float64_at_extreme_scales(k):
    """instance_ref (traversal, attributes and bounce rays, built on the CPU) against float64 in world space"""
    tris, offs, roots, xf, kinds, bound = case = extreme_case(k)
    r = ob.build_reference(tris, tri_stride=48, object_offsets=offs)
    ts, pi = r["info"]["tlas_start"], r["prim_indices"]
    ref = cpu_reference(r["nodes"], r["tri_bytes"], 48, ts, roots, xf)
    rays = extreme_rays(tris, offs, roots, xf, kinds, 4000, seed=k + 100)
    hits, ids, _, _ = ref.trace(rays)
    check_hits_float64(hits, ids, rays, case, pi)
    attrs, at = attr_reference(r["tri_bytes"], 48, rays, hits, inverse_f32(xf), ids)
    assert np.array_equal(at[hits["prim"] != INVALID].view(np.uint32), hits["t"][hits["prim"] != INVALID].view(np.uint32))
    check_ng(attrs, hits, ids, case, pi)
    w, h = 160, 120
    view = host.view_from_camera(EXTREME_CAMERA, w, h)
    prays = ob.primary_rays(view, w, h)
    ph, pid, _, _ = ref.trace(prays)
    brays = ref.bounce_rays(view, w, h, prays, ph, pid)
    check_bounce_float64(brays, prays, ph, pid, view, w, case, pi)


@gpu
@pytest.mark.parametrize("stride,k", [(s, k) for s in (48, 64) for k in SCALES] + [(24, -8), (24, 8)])
def test_extreme_transforms(stride, k):
    """kernels == instance_ref bit for bit (hits, ids, costs, attributes, frames), and the float64 checks on the device results.
    Stride 24 keeps its edges in f16 (normal for 2^-14 .. 2^15): only k = +-8 fits it."""
    tris, offs, roots, xf, kinds, bound = case = extreme_case(k)
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=offs)
    try:
        sc.set_instances(roots, xf)
        ref = Reference.of(sc)
        pi = sc.download_bvh()[2]
        rays = extreme_rays(tris, offs, roots, xf, kinds, 4000, seed=k + 100)
        for count in (False, True):
            for any_hit in (False, True):
                run_kernel(sc, ref, rays, count, any_hit, f"count={count}, any_hit={any_hit}", device=False)
        hits, ids = sc.traverse_instance(rays)
        rec = sc.download_bvh(prim_indices=False)[1]
        want_attrs, _ = attr_reference(rec, stride, rays, hits, sc.download_instance_xforms()[1], ids)
        got = sc.hit_attributes(rays, hits, ids)
        assert same_bytes(got, want_attrs)
        if stride != 24:
            check_hits_float64(hits, ids, rays, case, pi)
            check_ng(got, hits, ids, case, pi)
        w, h = 160, 120
        view = host.view_from_camera(EXTREME_CAMERA, w, h)
        want = reference_frame(ref, view, w, h)
        sc.set_ray_cost(True)
        sc.render(view, w, h, 0, FLAGS)
        sc.sync()
        check_frame(sc, want)
        if stride != 24:
            out = sc.download(primary=True, bounce_rays=True)
            pid = sc.download_instance(primary=True)["primary"]
            check_bounce_float64(out["bounce_rays"], ob.primary_rays(view, w, h), out["primary"], pid, view, w, case, pi)
    finally:
        sc.close()
