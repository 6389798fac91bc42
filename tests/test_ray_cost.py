"""Per-ray cost records: what each ray cost the counting kernels (nodes fetched, triangles tested, TLAS leaf entries, peak
stack entries), through tray_cuda_trace_cost / _device for batches and tray_cuda_scene_set_ray_cost +
tray_cuda_frame_download_cost for frames.

The oracle keeps the same numbers per ray: Oracle.trace(counts=True) fills {nodes, tris, insts} and Oracle.stack_need the peak
stack, counted as the kernels count them.  Every GPU comparison below is bit for bit against those, and the records of a
call sum to the tray_counters of the same call with counting on."""
import os
import re

import numpy as np
import pytest

import oracle_binding as ob
from conftest import ROOT, random_rays
from tray_racing_b200 import cuda, host

KERNEL_STACK = 48
PIPE_MIN = 1 << 18                                  # tray_cuda_trace: batches from here on take the chunked copy pipeline
FRAME = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_COUNTERS
COST_FIELDS = ("nodes", "tris", "instances", "stack")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_hits_identical(gpu, ref, what=""):
    assert (gpu["prim"] == ref["prim"]).all(), f"{what}: {(gpu['prim'] != ref['prim']).sum()} primitive ids differ"
    assert (bits(gpu["t"]) == bits(ref["t"])).all(), f"{what}: {(bits(gpu['t']) != bits(ref['t'])).sum()} hit t differ"


def assert_costs_equal(got, want, what=""):
    for f in COST_FIELDS:
        bad = got[f] != want[f]
        assert not bad.any(), f"{what}: {int(bad.sum())} rays differ in {f} (first at {int(np.flatnonzero(bad)[0])}: " \
                              f"{got[np.flatnonzero(bad)[0]]} vs {want[np.flatnonzero(bad)[0]]})"


def expected(orc, rays, any_hit=False):
    """(hits, cost records) of the oracle for `rays`"""
    hits, cnt, _ = orc.trace(rays, counts=True, any_hit=any_hit, stack_limit=KERNEL_STACK)
    c = np.zeros(len(rays), cuda.COST_DTYPE)
    c["nodes"], c["tris"], c["instances"] = cnt["nodes"], cnt["tris"], cnt["insts"]
    c["stack"] = orc.stack_need(rays, any_hit=any_hit)
    return hits, c


def sums(c):
    return {"nodes": int(c["nodes"].sum(dtype=np.uint64)), "tris": int(c["tris"].sum(dtype=np.uint64)),
            "instances": int(c["instances"].sum(dtype=np.uint64))}


def picked(counters):
    return {k: counters[k] for k in ("nodes", "tris", "instances")}


def cornell_rays(mesh, n, seed):
    t = mesh.tris().reshape(-1, 3)
    return random_rays(n, seed, lo=float(t.min()), hi=float(t.max()))


def frame_expected(orc, view, w, h, fc, ao=False):
    """the oracle's frame and the cost records its primary and bounce rays must report (zero where no bounce ray is shot)"""
    ref = orc.render(view, w, h, fc)
    _, prim = expected(orc, ob.primary_rays(view, w, h))
    shoot = ref["bounce_rays"]["tmax"] > 0
    bounce = np.zeros(w * h, cuda.COST_DTYPE)
    brays = np.ascontiguousarray(ref["bounce_rays"][shoot])
    bhits, bounce[shoot] = expected(orc, brays, any_hit=ao)
    return ref, prim, bounce, shoot, bhits


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_cost_record_layout_agrees_between_header_python_and_rust():
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "tray_cuda.h")).read(), flags=re.S)
    body = re.search(r"typedef struct tray_ray_cost \{(.*?)\} tray_ray_cost;", header, flags=re.S).group(1)
    fields = re.findall(r"uint32_t\s+(\w+);", body)
    assert fields == list(COST_FIELDS)                                  # four u32: offsets 0, 4, 8, 12, 16 bytes
    assert cuda.COST_DTYPE.itemsize == 16 and list(cuda.COST_DTYPE.names) == fields
    assert [cuda.COST_DTYPE.fields[f][1] for f in fields] == [0, 4, 8, 12]
    assert all(cuda.COST_DTYPE.fields[f][0] == np.dtype("<u4") for f in fields)
    rust = open(os.path.join(ROOT, "tray_cuda", "src", "lib.rs")).read()
    m = re.search(r"#\[repr\(C\)\]\s*#\[derive\([^)]*\)\]\s*pub struct TrayRayCost \{(.*?)\}", rust, flags=re.S)
    assert m and re.findall(r"pub (\w+): u32", m.group(1)) == fields


def test_cost_entry_points_reject_null_arguments_without_a_device():
    L = cuda.lib()
    assert L.tray_cuda_trace_cost(None, None, 0, 0, None, None, None, None) == -1
    assert L.tray_cuda_trace_cost(None, None, 4, 1, None, None, None, None) == -1
    assert L.tray_cuda_trace_cost_device(None, None, 0, 0, None, None, None, None) == -1
    assert L.tray_cuda_trace_cost_device(None, None, 4, 0, None, None, None, None) == -1
    assert L.tray_cuda_scene_set_ray_cost(None, 1) == -1
    assert L.tray_cuda_frame_download_cost(None, None, None) == -1
    assert b"NULL" in L.tray_cuda_last_error()


# ---- GPU: batches -------------------------------------------------------------------------------------------------------------
def device_copy(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda()


def device_cost_trace(g, rays, any_hit, stream=0, timed=True):
    import torch
    d_rays = device_copy(rays)
    d_hits = torch.empty(len(rays) * 8, dtype=torch.uint8, device="cuda")
    d_cost = torch.zeros(len(rays) * 16, dtype=torch.uint8, device="cuda")
    torch.cuda.current_stream().synchronize()                           # the buffers are ready before a caller's stream uses them
    g.traverse_cost_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr(), d_cost.data_ptr(), stream=stream, timed=timed, any_hit=any_hit)
    return d_hits, d_cost


@pytest.mark.gpu
@pytest.mark.parametrize("any_hit", [False, True], ids=["closest", "any"])
@pytest.mark.parametrize("stride", [24, 48, 64])
@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
def test_batch_costs_match_the_oracle(cornell, use_tlas, stride, any_hit):
    import torch
    p = host.PackedScene(cornell, use_tlas=use_tlas, tri_stride=stride)
    orc = ob.Oracle.from_packed(p)
    g = cuda.TrayCudaScene.from_packed(p)
    batches = [cornell_rays(cornell, 20000, 1 + stride)]
    if stride == 48:
        batches.append(cornell_rays(cornell, PIPE_MIN + 1234, 2 + stride))          # the chunked copy pipeline
    try:
        for rays in batches:
            what = f"{len(rays)} rays"
            ref, want = expected(orc, rays, any_hit)
            assert want["nodes"].min() > 0 and (want["tris"] > 0).mean() > 0.2 and want["stack"].max() > 0
            if use_tlas:
                assert (want["instances"] > 0).mean() > 0.2
            hits, costs = g.traverse_cost(rays, any_hit=any_hit)
            assert_hits_identical(hits, ref, what)
            assert_hits_identical(hits, g.traverse(rays, any_hit=any_hit), what + " vs tray_cuda_trace")
            assert_costs_equal(costs, want, what)
        # the device entry point on a caller's stream: asynchronous, then timed
        rays = batches[0]
        _, want = expected(orc, rays, any_hit)
        s = torch.cuda.Stream()
        for timed in (False, True):
            d_hits, d_cost = device_cost_trace(g, rays, any_hit, stream=s.cuda_stream, timed=timed)
            s.synchronize()
            assert_hits_identical(d_hits.cpu().numpy().view(ob.HIT_DTYPE), expected(orc, rays, any_hit)[0], "device entry point")
            assert_costs_equal(d_cost.cpu().numpy().view(cuda.COST_DTYPE), want, f"device entry point, timed={timed}")
        g.sync()
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
def test_batch_costs_sum_to_the_counters_and_leave_them_to_set_counting(cornell, use_tlas):
    p = host.PackedScene(cornell, use_tlas=use_tlas)
    g = cuda.TrayCudaScene.from_packed(p)
    try:
        for n, seed in ((30000, 5), (PIPE_MIN + 99, 6)):
            rays = cornell_rays(cornell, n, seed)
            for any_hit in (False, True):
                g.set_counting(True)
                g.traverse(rays, any_hit=any_hit)
                counted = g.counters()[0]
                _, costs = g.traverse_cost(rays, any_hit=any_hit)
                assert sums(costs) == picked(counted)
                assert g.counters()[0] == counted                             # counting on: the cost call counts the same rays
                g.set_counting(False)
                other = cornell_rays(cornell, 5000, seed + 10)
                g.traverse_cost(other, any_hit=any_hit)
                assert g.counters()[0] == counted                             # counting off: the counters stay as they were
                device_cost_trace(g, other, any_hit, timed=True)
                assert g.counters()[0] == counted
    finally:
        g.close()


# ---- GPU: frames --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ao", [False, True], ids=["bounce", "anyhit_ao"])
@pytest.mark.parametrize("overlap", [False, True], ids=["two_launch", "one_launch"])
@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
def test_frame_costs_match_the_oracle(cornell, use_tlas, overlap, ao):
    w, h, fc = 100, 37, 2
    p = host.PackedScene(cornell, use_tlas=use_tlas)
    view = host.view_from_camera(cornell.camera, w, h, p.tlas_start)
    orc = ob.Oracle.from_packed(p)
    ref, want_p, want_b, shoot, bhits = frame_expected(orc, view, w, h, fc, ao)
    assert shoot.mean() > 0.3 and (~shoot).any()
    flags = FRAME | (cuda.RENDER_OVERLAP if overlap else 0) | (cuda.RENDER_ANYHIT_AO if ao else 0)
    g = cuda.TrayCudaScene.from_packed(p)
    try:
        g.set_ray_cost(False)
        g.render(view, w, h, fc, flags)
        off = g.download(primary=True, bounce=True, rgba=True)
        g.set_ray_cost(True)
        g.render(view, w, h, fc, flags)
        on = g.download(primary=True, bounce=True, rgba=True)
        for k in ("primary", "bounce", "rgba"):
            assert np.ascontiguousarray(on[k]).tobytes() == np.ascontiguousarray(off[k]).tobytes(), f"{k} changes with ray costs on"
        assert_hits_identical(on["primary"], ref["primary"], "primary")
        assert_hits_identical(on["bounce"][shoot], bhits, "bounce")
        c = g.download_cost(primary=True, bounce=True)
        assert_costs_equal(c["primary"], want_p, "primary")
        assert_costs_equal(c["bounce"], want_b, "bounce")
        assert not bits(c["bounce"][~shoot]).any()
        cp, cb = g.counters()
        assert sums(c["primary"]) == picked(cp) and sums(c["bounce"]) == picked(cb)
        assert g.download_cost(primary=False, bounce=True).keys() == {"bounce"}
        g.render(view, w, h, fc, flags & ~cuda.RENDER_BOUNCE)
        assert_costs_equal(g.download_cost()["primary"], want_p, "primary of a frame without bounce rays")
        with pytest.raises(cuda.TrayCudaError, match="BOUNCE"):
            g.download_cost(bounce=True)
    finally:
        g.close()


@pytest.mark.gpu
def test_frame_costs_of_three_shards_merge_to_the_whole_frame(cornell):
    w, h = 100, 37
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, w, h)
    g = cuda.TrayCudaScene.from_packed(p)
    try:
        g.set_ray_cost(True)
        g.render(view, w, h, 1, FRAME)
        whole = g.download_cost(primary=True, bounce=True)
        merged = None
        for shard in range(3):
            g.render(view, w, h, 1, FRAME, shard=shard, shards=3)
            part = g.download_cost(primary=True, bounce=True)
            own = cuda.shard_mask(w, h, shard, 3)
            for k in ("primary", "bounce"):
                assert not bits(part[k][~own]).any(), f"shard {shard}: {k} records outside its tiles"
                assert (part[k][own] == whole[k][own]).all()
            cp, cb = g.counters()
            assert sums(part["primary"]) == picked(cp) and sums(part["bounce"]) == picked(cb)
            merged = g.download_cost(primary=True, bounce=True, into=merged, merge=True) if merged is not None else part
        for k in ("primary", "bounce"):
            assert merged[k].tobytes() == whole[k].tobytes()
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_in_flight", [2, 3])
def test_frame_costs_follow_the_last_frame(cornell, n_in_flight):
    w, h = 100, 37
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, w, h)
    orc = ob.Oracle.from_packed(p)
    want = {fc: frame_expected(orc, view, w, h, fc)[1:3] for fc in range(n_in_flight + 1)}
    g = cuda.TrayCudaScene.from_packed(p)

    def check(fc, what):
        c = g.download_cost(primary=True, bounce=True)
        assert_costs_equal(c["primary"], want[fc][0], f"{what}: primary")
        assert_costs_equal(c["bounce"], want[fc][1], f"{what}: bounce")

    try:
        g.set_ray_cost(True)
        g.set_frames_in_flight(n_in_flight)
        for fc in range(n_in_flight + 1):
            g.render(view, w, h, fc, FRAME, timed=False)
            check(fc, f"frame {fc} of {n_in_flight} in flight")
        # the last frame's slot does not survive the switch: its records move with the frame
        g.render(view, w, h, n_in_flight - 1, FRAME, timed=False)
        g.set_frames_in_flight(1)
        check(n_in_flight - 1, "after set_frames_in_flight(1)")
        # a refused render changes nothing
        with pytest.raises(cuda.TrayCudaError):
            g.render(view, w, h, 0, FRAME, shard=3, shards=3)
        g.set_variant(cuda.VARIANT_TIE_LAST)
        with pytest.raises(cuda.TrayCudaError, match="semantic variants"):
            g.render(view, w, h, 0, FRAME)
        g.set_variant(0)
        check(n_in_flight - 1, "after refused renders")
        # a later frame without counters, or with ray costs off, keeps no records: the download refuses
        g.set_frames_in_flight(n_in_flight)
        g.render(view, w, h, 0, FRAME & ~cuda.RENDER_COUNTERS, timed=False)
        with pytest.raises(cuda.TrayCudaError, match="no ray costs"):
            g.download_cost()
        g.render(view, w, h, 0, FRAME, timed=False)
        check(0, "counted again")
        g.set_ray_cost(False)
        g.render(view, w, h, 1, FRAME, timed=False)
        with pytest.raises(cuda.TrayCudaError, match="no ray costs"):
            g.download_cost()
        g.sync()
    finally:
        g.close()


# ---- GPU: the stack column ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("depth", [12, 13, 32, 33, 48])
@pytest.mark.parametrize("shape", ["flat", "tlas"])
def test_stack_equals_stack_need_down_the_ladders(shape, depth):
    from test_deep_stack import assert_reaches, flat_ladder, ladder_rays, tlas_ladder
    sc = flat_ladder(depth + 1) if shape == "flat" else tlas_ladder(depth + 1)
    rays = ladder_rays(4096, depth, sc.tris)
    orc = sc.oracle()
    ref, want = expected(orc, rays)
    assert_reaches(want["stack"], depth, shape)
    g = sc.cuda()
    try:
        hits, costs = g.traverse_cost(rays)
        assert_hits_identical(hits, ref, shape)
        assert_costs_equal(costs, want, f"{shape} ladder, need {depth}")
        _, costs = g.traverse_cost(rays, any_hit=True)
        assert_costs_equal(costs, expected(orc, rays, any_hit=True)[1], f"{shape} ladder, need {depth}, any hit")
    finally:
        g.close()


@pytest.mark.gpu
def test_a_need_of_49_reports_48_and_the_overflow():
    import torch
    from test_deep_stack import flat_ladder, ladder_rays
    sc = flat_ladder(50)
    rays = ladder_rays(4096, 11, sc.tris)
    need = sc.oracle().stack_need(rays)
    assert need.max() == 49
    g = sc.cuda()
    try:
        d_hits, d_cost = device_cost_trace(g, rays, False, timed=False)      # asynchronous: the next sync reports
        with pytest.raises(cuda.TrayCudaError, match=r"error -4\b"):
            g.sync()
        stack = d_cost.cpu().numpy().view(cuda.COST_DTYPE)["stack"]
        assert (stack[need > KERNEL_STACK] == KERNEL_STACK).all()
        assert (stack[need <= KERNEL_STACK] == need[need <= KERNEL_STACK]).all()
        with pytest.raises(cuda.TrayCudaError, match=r"error -4\b"):
            g.traverse_cost(rays)
        clean = rays[need <= KERNEL_STACK]
        _, costs = g.traverse_cost(clean)
        assert_costs_equal(costs, expected(sc.oracle(), clean)[1], "clean batch after the overflow")
        torch.cuda.synchronize()
    finally:
        g.close()


# ---- GPU: every counting instantiation on generated trees --------------------------------------------------------------------
COUNT_KERNELS = [(tlas, stride, kind) for tlas in (False, True) for stride in (24, 48, 64) for kind in ("closest", "any", "frame")]


@pytest.mark.gpu
@pytest.mark.parametrize("k", COUNT_KERNELS, ids=lambda k: f"{'tlas' if k[0] else 'flat'}-{k[1]}-{k[2]}")
def test_counting_instantiation_costs_on_generated_trees(k):
    from test_cwbvh_fuzz import CAMERA, KERNELS, case_rays, case_seed, make_case, zeroed_oracle
    tlas, stride, kind = k
    seed = case_seed((tlas, True, stride, kind, 0))
    assert (tlas, True, stride, kind, 0) in KERNELS
    tris, gen, sc = make_case(tlas, stride, seed)
    orc = zeroed_oracle(gen, sc)
    g = sc.cuda()
    try:
        if kind == "frame":
            w, h = 192, 128
            view = host.view_from_camera(CAMERA, w, h, gen.tlas_start)
            _, want_p, want_b, shoot, _ = frame_expected(orc, view, w, h, 3)
            assert shoot.mean() > 0.05
            g.set_ray_cost(True)
            for overlap in (cuda.RENDER_OVERLAP, 0):                        # the FRAME kernel, then the two launches
                g.render(view, w, h, 3, FRAME | overlap)
                c = g.download_cost(primary=True, bounce=True)
                assert_costs_equal(c["primary"], want_p, f"primary, overlap={bool(overlap)}")
                assert_costs_equal(c["bounce"], want_b, f"bounce, overlap={bool(overlap)}")
        else:
            rays = case_rays(seed)
            ref, want = expected(orc, rays, kind == "any")
            hits, costs = g.traverse_cost(rays, any_hit=kind == "any")
            assert_hits_identical(hits, ref, kind)
            assert_costs_equal(costs, want, kind)
        g.sync()
    finally:
        g.close()


# ---- GPU: edges ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_empty_scene_costs_are_zero():
    from cwbvh_bytes import random_cwbvh
    tris = np.zeros((0, 9), np.float32)
    sc = random_cwbvh(tris, 1).scene(tris, 48)
    g = sc.cuda()
    try:
        for n in (1000, PIPE_MIN + 5):
            rays = random_rays(n, 3)
            for any_hit in (False, True):
                hits, costs = g.traverse_cost(rays, any_hit=any_hit)
                assert (hits["prim"] == ob.INVALID_PRIM).all()
                assert not bits(costs).any()
        g.set_ray_cost(True)
        view = host.view_from_camera(host.Camera((1.5, 1.1, 1.9), (0, 0, 0), 50.0), 64, 40)
        g.render(view, 64, 40, 0, FRAME)
        c = g.download_cost(primary=True, bounce=True)
        assert not bits(c["primary"]).any() and not bits(c["bounce"]).any()
        assert g.counters()[0]["nodes"] == 0
    finally:
        g.close()


@pytest.mark.gpu
def test_variant_scene_refuses_the_cost_calls_and_changes_nothing(cornell):
    import torch
    p = host.PackedScene(cornell)
    w, h = 100, 37
    view = host.view_from_camera(cornell.camera, w, h)
    g = cuda.TrayCudaScene.from_packed(p)
    try:
        g.set_ray_cost(True)
        g.set_counting(True)
        rays = cornell_rays(cornell, 4000, 9)
        g.traverse(rays)
        g.render(view, w, h, 0, FRAME)
        before = g.download_cost(primary=True, bounce=True)
        counted = g.counters()                                               # the frame's
        g.set_variant(cuda.VARIANT_BOX_DIVIDE)
        with pytest.raises(cuda.TrayCudaError, match="semantic variants"):
            g.traverse_cost(rays)
        d_rays = device_copy(rays)
        d_out = torch.full((len(rays) * 16,), 7, dtype=torch.uint8, device="cuda")
        with pytest.raises(cuda.TrayCudaError, match="semantic variants"):
            g.traverse_cost_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), d_out.data_ptr(), timed=True)
        assert (d_out.cpu().numpy() == 7).all()
        assert g.counters() == counted
        after = g.download_cost(primary=True, bounce=True)
        assert after["primary"].tobytes() == before["primary"].tobytes() and after["bounce"].tobytes() == before["bounce"].tobytes()
        g.set_variant(0)
        _, costs = g.traverse_cost(rays)
        assert sums(costs) == picked(g.counters()[0])
    finally:
        g.close()


# ---- GPU: one process, several GPUs -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_group_shard_costs_sum_to_the_single_gpu_frame(cornell):
    if cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    w, h = 160, 90
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, w, h)
    one = cuda.TrayCudaScene.from_packed(p)
    try:
        one.set_ray_cost(True)
        one.render(view, w, h, 0, FRAME)
        want = one.download_cost(primary=True, bounce=True)
    finally:
        one.close()
    n = min(cuda.device_count(), 4)
    grp = cuda.TrayCudaGroup.from_packed(p, devices=list(range(n)))
    try:
        for i in range(n):
            grp.scene(i).set_ray_cost(True)
        grp.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_COUNTERS, timed=True)
        grp.sync()
        total = {k: np.zeros(w * h, cuda.COST_DTYPE) for k in ("primary", "bounce")}
        for i in range(n):
            part = grp.scene(i).download_cost(primary=True, bounce=True)
            for k in total:
                for f in COST_FIELDS:
                    total[k][f] += part[k][f]
        for k in total:
            assert total[k].tobytes() == want[k].tobytes(), k
    finally:
        grp.close()
