"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same inputs.
Bar (BASELINE.json north_star): primitive ids bit-identical except genuine ties, t within 1e-5 relative.
Because each lane runs the reference's per-ray state machine unchanged, the kernel actually meets the
stronger bar asserted here: ids AND t bit-identical, and identical node / triangle visit counts."""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import load_golden_mesh, random_rays
from tray_racing_b200 import cuda, host

pytestmark = pytest.mark.gpu
F32_MAX = np.float32(3.402823466e+38)
FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_KEEP_RAYS


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_hits_identical(gpu, ref, what=""):
    assert (gpu["prim"] == ref["prim"]).all(), f"{what}: {(gpu['prim'] != ref['prim']).sum()} primitive ids differ"
    assert (bits(gpu["t"]) == bits(ref["t"])).all(), f"{what}: {(bits(gpu['t']) != bits(ref['t'])).sum()} hit t differ"
    # and therefore also the stated tolerance: |t_gpu - t_ref| <= 1e-5 * |t_ref|
    hit = ref["prim"] != ob.INVALID_PRIM
    assert (np.abs(gpu["t"][hit] - ref["t"][hit]) <= 1e-5 * np.abs(ref["t"][hit])).all()


def render_and_compare(mesh, w, h, use_tlas=False, stride=48, frame=0, counters=True, overlap=False):
    p = host.PackedScene(mesh, use_tlas=use_tlas, tri_stride=stride)
    view = host.view_from_camera(mesh.camera, w, h, p.tlas_start)
    ref = ob.Oracle.from_packed(p).render(view, w, h, frame_count=frame, rgba=True)
    sc = cuda.TrayCudaScene.from_packed(p)
    try:
        sc.render(view, w, h, frame, FLAGS | (cuda.RENDER_COUNTERS if counters else 0) | (cuda.RENDER_OVERLAP if overlap else 0))
        sc.sync()                                                            # raises if a kernel flagged an overflow / watchdog
        out = sc.download(primary=True, bounce=True, bounce_rays=True, rgba=True)
        assert_hits_identical(out["primary"], ref["primary"], "primary")
        assert (out["bounce_rays"].view(np.uint32) == ref["bounce_rays"].view(np.uint32)).all(), "bounce rays differ"
        assert_hits_identical(out["bounce"], ref["bounce"], "bounce")
        # shading uses powf, which is not bit-portable: +-1 grey level (not a parity item, SURVEY.md §8a a15)
        assert np.abs(out["rgba"].reshape(-1, 4).astype(int) - ref["rgba"].astype(int)).max() <= 1
        if counters:
            cp, cb = sc.counters()
            for got, want in ((cp, ref["primary_totals"]), (cb, ref["bounce_totals"])):
                assert got["rays"] == want["rays"] and got["hits"] == want["hits"]
                assert got["nodes"] == want["nodes"] and got["tris"] == want["tris"] and got["instances"] == want["insts"]
    finally:
        sc.close()
    return p, ref


@pytest.mark.parametrize("use_tlas,stride", [(False, 48), (False, 64), (True, 48), (True, 64)])
def test_cornell_box_frame(cornell, use_tlas, stride):
    p, ref = render_and_compare(cornell, 640, 360, use_tlas, stride)
    assert ref["primary_totals"]["hits"] > 100000


@pytest.mark.parametrize("use_tlas", [False, True])
def test_box_scene_tiny_blas(box, use_tlas):
    render_and_compare(box, 320, 200, use_tlas)


def test_odd_resolution_and_other_frame(cornell):
    """W, H not multiples of the 32x8 tile (the reference drops the tail, rt_gpu_software.rs:298; we render it),
    and a non-zero frame_count (--animate, rt_cpu.rs:95-97)."""
    render_and_compare(cornell, 101, 37, frame=5)
    render_and_compare(cornell, 33, 9, use_tlas=True, frame=1029)


@pytest.mark.parametrize("name,seed,size,tlas", [("kitchen", 1, 1.0, False), ("hairball", 3, 0.1, False),
                                                 ("demoscene", 2, 0.1, False), ("sanmiguel", 4, 0.05, False),
                                                 ("caldera", 5, 0.02, True), ("caldera", 5, 0.02, False)])
def test_synthetic_scenes_frame(name, seed, size, tlas):
    render_and_compare(host.Mesh.generate(name, seed, size), 480, 270, use_tlas=tlas)


@pytest.mark.parametrize("use_tlas,stride", [(False, 48), (False, 64), (True, 48), (True, 64), (False, 24)])
def test_one_launch_frame_kernel_is_bit_identical(cornell, use_tlas, stride):
    """TRAY_RENDER_OVERLAP: one launch per frame; bounce rays of finished tiles are generated and traced while the primary
    pass drains.  Primary hits, bounce rays, bounce hits, image and the per-kind node / triangle / instance counters are those
    of the oracle (and so of the two-launch path)."""
    render_and_compare(cornell, 640, 360, use_tlas, stride, overlap=True)
    render_and_compare(cornell, 101, 37, use_tlas, stride, frame=5, overlap=True)
    render_and_compare(cornell, 640, 360, use_tlas, stride, counters=False, overlap=True)


@pytest.mark.parametrize("gen_min", [1, 32])
@pytest.mark.parametrize("name,seed,size,tlas", [("hairball", 3, 0.1, False), ("caldera", 5, 0.02, True), ("kitchen", 1, 1.0, False)])
def test_one_launch_frame_kernel_on_synthetic_scenes(monkeypatch, name, seed, size, tlas, gen_min):
    monkeypatch.setenv("TRAY_CUDA_GEN_MIN", str(gen_min))
    render_and_compare(host.Mesh.generate(name, seed, size), 480, 270, use_tlas=tlas, overlap=True)


def test_one_launch_frame_kernel_edge_frames(cornell, box):
    """The frame kernel on frames where its hand-shake has little to chew on: a camera that sees nothing (every group of
    32 pixels is all misses), a frame smaller than one tile, tile shards (each shard a frame of its own), two frames in a row."""
    away = host.Camera((0.0, 1.0, 50.0), (0.0, 1.0, 100.0), 40.0)            # looks away from the box
    p = host.PackedScene(cornell)
    sc = cuda.TrayCudaScene.from_packed(p)
    orc = ob.Oracle.from_packed(p)
    try:
        for cam, w, h in ((away, 320, 184), (cornell.camera, 7, 3), (cornell.camera, 33, 9)):
            view = host.view_from_camera(cam, w, h)
            ref = orc.render(view, w, h, 0)
            for _ in range(2):
                sc.render(view, w, h, 0, FLAGS | cuda.RENDER_OVERLAP)
                sc.sync()
                out = sc.download(primary=True, bounce=True)
                for k in ("primary", "bounce"):
                    assert_hits_identical(out[k], ref[k], f"{k} {w}x{h}")
        w, h = 200, 120
        view = host.view_from_camera(cornell.camera, w, h)
        ref = orc.render(view, w, h, 0)
        acc = {}
        for s in range(3):
            sc.render(view, w, h, 0, FLAGS | cuda.RENDER_OVERLAP, shard=s, shards=3)
            sc.download(primary=True, bounce=True, into=acc, merge=True)
        for k in ("primary", "bounce"):
            assert_hits_identical(acc[k], ref[k], f"{k} shards")
    finally:
        sc.close()


def test_traverse_random_rays(cornell):
    """Batch operator (Traversable::traverse at batch grain) on rays with exact-zero direction components
    (zero-direction fix-up, query.hlsl:334) and finite [tmin, tmax] windows; ragged batch sizes."""
    p = host.PackedScene(cornell)
    orc = ob.Oracle.from_packed(p)
    sc = cuda.TrayCudaScene.from_packed(p)
    try:
        for n, seed in [(1, 1), (31, 2), (33, 3), (1000, 4), (100003, 5)]:
            rays = random_rays(n, seed, axis_fraction=0.1, bounded_fraction=0.3)
            t = {}
            assert_hits_identical(sc.traverse(rays, t), orc.trace(rays), f"n={n}")
            assert t["ms_total"] >= t["ms_kernel"] >= 0
        assert len(sc.traverse(np.zeros(0, dtype=host.RAY_DTYPE))) == 0            # empty batch
        # rays that cannot hit anything
        away = random_rays(500, 6)
        away["o"] += 100; away["d"] = np.float32([0, 1, 0])
        h = sc.traverse(away)
        assert (h["prim"] == ob.INVALID_PRIM).all() and np.isinf(h["t"]).all()
    finally:
        sc.close()


@pytest.mark.parametrize("any_hit", [False, True])
def test_large_host_batches_take_the_copy_pipeline(cornell, any_hit):
    """Batches of >= 2^18 rays go through the chunked upload / trace / read-back pipeline of tray_cuda_trace (pinned staging
    slots, three streams): ragged last chunk, exactly one chunk, several chunks; hits and counters as the oracle's."""
    p = host.PackedScene(cornell)
    orc = ob.Oracle.from_packed(p)
    sc = cuda.TrayCudaScene.from_packed(p)
    try:
        for n, seed in [((1 << 18), 7), ((1 << 20), 8), (3 * (1 << 20) + 12345, 9)]:
            rays = random_rays(n, seed, axis_fraction=0.05, bounded_fraction=0.2)
            assert_hits_identical(sc.traverse(rays, any_hit=any_hit), orc.trace(rays, any_hit=any_hit), f"n={n}")
        if not any_hit:
            sc.set_counting(True)
            rays = random_rays(2 * (1 << 20) + 77, 10)
            got = sc.traverse(rays)
            ref, _, tot = orc.trace(rays, counts=True)
            assert_hits_identical(got, ref)
            cp, _ = sc.counters()
            assert cp["rays"] == len(rays) and cp["nodes"] == tot["nodes"] and cp["tris"] == tot["tris"]
    finally:
        sc.close()


def test_two_devices_in_one_process_assemble_the_frame(cornell):
    """INTEGRATION.md §4 without torchrun: one scene per device in ONE process (uploads through the shared pinned slots with
    per-device events), each renders its tile shard, the shards assemble to the single-GPU frame.  Needs two GPUs."""
    if cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    p = host.PackedScene(host.Mesh.generate("kitchen", 1, 1.0))      # > 8 MiB of triangles: takes the pipelined upload
    w, h = 640, 360
    view = host.view_from_camera(cornell.camera, w, h)
    ref = ob.Oracle.from_packed(p).render(view, w, h, 0)
    scenes = [cuda.TrayCudaScene.from_packed(p, device=d) for d in (0, 1)]
    try:
        acc = {}
        for d, sc in enumerate(scenes):
            sc.render(view, w, h, 0, cuda.RENDER_BOUNCE, shard=d, shards=2)
            sc.download(primary=True, bounce=True, into=acc, merge=True)
        for k in ("primary", "bounce"):
            assert_hits_identical(acc[k], ref[k], k)
        rays = random_rays(400000, 5)
        assert_hits_identical(scenes[1].traverse(rays), ob.Oracle.from_packed(p).trace(rays), "device 1 batch")
    finally:
        for sc in scenes:
            sc.close()


def test_two_host_threads_trace_concurrently(cornell, box):
    """Two scenes driven from two host threads at once (ctypes drops the GIL): the copy threads and the pinned upload slots
    are shared by the process, the pipeline slots are per scene — results stay those of the oracle."""
    import threading
    jobs = []
    for mesh, use_tlas, stride, seed in ((cornell, False, 48, 31), (cornell, True, 64, 32), (box, False, 24, 33)):
        p = host.PackedScene(mesh, use_tlas=use_tlas, tri_stride=stride)
        rays = random_rays(700001, seed)
        jobs.append((p, rays, ob.Oracle.from_packed(p).trace(rays)))
    out, errs = [None] * len(jobs), []

    def work(i):
        try:
            p, rays, _ = jobs[i]
            sc = cuda.TrayCudaScene.from_packed(p)
            try:
                for _ in range(3):
                    out[i] = sc.traverse(rays)
            finally:
                sc.close()
        except Exception as e:          # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(jobs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for i, (_, _, ref) in enumerate(jobs):
        assert_hits_identical(out[i], ref, f"job {i}")


def test_tiny_direction_components_take_the_unfused_node_test(cornell, monkeypatch):
    """The fused node test (fma(2^23 + q, A, -2^23 A) == fl(q A)) needs 2^23 * A finite.  Rays with |1/d| >= 2^64 on an
    axis, and scenes with node scales >= 2^40, fall back to the unfused test; both paths must match the oracle, and
    forcing the unfused path everywhere must not change a single bit."""
    p = host.PackedScene(cornell)
    orc = ob.Oracle.from_packed(p)
    rays = random_rays(60000, 21, axis_fraction=0.0)
    rng = np.random.default_rng(3)
    tiny = rng.choice([1e-20, -1e-20, 1e-25, -3e-30, 1e-37, -1e-38, 1e-42], size=len(rays)).astype(np.float32)
    ax = rng.integers(0, 3, size=len(rays))
    rays["d"][np.arange(len(rays)), ax] = tiny                       # not renormalised on purpose: t scales, parity must hold
    ref = orc.trace(rays)
    assert (ref["prim"] != ob.INVALID_PRIM).sum() > 1000
    results = []
    for force in ("0", "1"):
        monkeypatch.setenv("TRAY_CUDA_FORCE_EXACT", force)
        sc = cuda.TrayCudaScene.from_packed(p)
        try:
            results.append(sc.traverse(rays))
            plain = random_rays(50000, 22)
            assert_hits_identical(sc.traverse(plain), orc.trace(plain), f"force_exact={force}")
        finally:
            sc.close()
    assert_hits_identical(results[0], ref, "tiny components")
    assert_hits_identical(results[1], ref, "tiny components, unfused everywhere")


def test_huge_scene_scale_falls_back_to_unfused_test():
    """A scene 2^50 units across has node scales >= 2^40 and is traversed with the unfused test.  (At that size the
    triangle test itself overflows f32 in the reference arithmetic, so nothing is hit — what matters is that the
    kernel agrees with the oracle and produces no spurious hit out of an overflowed 2^23 * A.)"""
    m = host.Mesh.generate("soup", 5, 0.002)
    tris = (m.tris() * np.float32(2.0 ** 50)).astype(np.float32)
    nodes, pidx, _ = host.build_cwbvh(tris)
    assert nodes[:, 12:15].max() >= 167
    rec = host.tri_records(tris[pidx])
    rays = random_rays(20000, 23, lo=-1, hi=1)
    rays["o"] *= np.float32(2.0 ** 50)
    sc = cuda.TrayCudaScene(nodes, rec)
    try:
        got = sc.traverse(rays)
    finally:
        sc.close()
    ref = ob.Oracle(nodes, rec).trace(rays)
    assert_hits_identical(got, ref)
    # a merely large scene (2^30 units, node scales ~2^23) still uses the fused test and still matches
    tris = (m.tris() * np.float32(2.0 ** 30)).astype(np.float32)
    nodes, pidx, _ = host.build_cwbvh(tris)
    assert nodes[:, 12:15].max() < 167
    rec = host.tri_records(tris[pidx])
    rays = random_rays(20000, 24, lo=-1, hi=1)
    rays["o"] *= np.float32(2.0 ** 30)
    sc = cuda.TrayCudaScene(nodes, rec)
    try:
        got = sc.traverse(rays)
    finally:
        sc.close()
    ref = ob.Oracle(nodes, rec).trace(rays)
    assert (ref["prim"] != ob.INVALID_PRIM).sum() > 100
    assert_hits_identical(got, ref)


def test_degenerate_scenes():
    """One triangle (root with a single leaf child), coincident triangles (tie rule), empty scene."""
    one = np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], dtype=np.float32)
    for tris in (one, np.repeat(one, 5, axis=0)):
        nodes, pidx, _ = host.build_cwbvh(tris)
        rec = host.tri_records(tris[pidx])
        rays = random_rays(4000, 7, lo=-0.2, hi=1.2)
        sc = cuda.TrayCudaScene(nodes, rec)
        try:
            assert_hits_identical(sc.traverse(rays), ob.Oracle(nodes, rec).trace(rays))
        finally:
            sc.close()
    sc = cuda.TrayCudaScene(np.zeros(0, np.uint8), np.zeros(0, np.uint8))
    try:
        h = sc.traverse(random_rays(100, 8))
        assert (h["prim"] == ob.INVALID_PRIM).all() and np.isinf(h["t"]).all()
    finally:
        sc.close()


def test_tile_shards_reassemble_the_frame(cornell):
    """N-way interleaved-tile sharding (the multi-GPU partition) reproduces the single-shard frame bit for bit."""
    p = host.PackedScene(cornell)
    w, h = 200, 120
    view = host.view_from_camera(cornell.camera, w, h)
    sc = cuda.TrayCudaScene.from_packed(p)
    try:
        sc.render(view, w, h, 0, FLAGS)
        full = sc.download(primary=True, bounce=True, rgba=True)
        for shards in (2, 3, 8):
            acc = {}
            for s in range(shards):
                sc.render(view, w, h, 0, FLAGS, shard=s, shards=shards)
                sc.download(primary=True, bounce=True, rgba=True, into=acc, merge=True)
            for k in ("primary", "bounce"):
                assert (acc[k]["prim"] == full[k]["prim"]).all() and (bits(acc[k]["t"]) == bits(full[k]["t"])).all()
            assert (acc["rgba"] == full["rgba"]).all()
    finally:
        sc.close()


def test_deterministic_across_runs_and_scheduler_knobs(cornell, monkeypatch):
    """The warp-level schedule (refill threshold, phase vote) never changes a ray's own traversal order."""
    p = host.PackedScene(host.Mesh.generate("hairball", 3, 0.05))
    rays = random_rays(200000, 12, lo=-5, hi=5)
    results = []
    for tw, rm in [(4, 8), (1, 1), (64, 24), (2, 32)]:
        monkeypatch.setenv("TRAY_CUDA_TRI_WEIGHT", str(tw))
        monkeypatch.setenv("TRAY_CUDA_REFILL_MIN", str(rm))
        sc = cuda.TrayCudaScene.from_packed(p)
        try:
            results.append(sc.traverse(rays))
        finally:
            sc.close()
    for r in results[1:]:
        assert (r["prim"] == results[0]["prim"]).all() and (bits(r["t"]) == bits(results[0]["t"])).all()
    assert_hits_identical(results[0], ob.Oracle.from_packed(p).trace(rays))


def test_start_slot_runs_the_reference_protocol(cornell):
    """tray_cuda_start == rt_gpu_software::start: returns min frame ms (rt_gpu_software.rs:376) after rendering
    for render_time seconds, with the warm-up dispatch when benchmark is set (:289-295)."""
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, 640, 360)
    mn, mean, frames = cuda.start(p.bvh_bytes, p.instance_bytes, p.tri_bytes, p.tlas_start, view, 640, 360,
                                  render_time=0.2, benchmark=True)
    assert frames >= 2 and 0 < mn <= mean < 50
    from tray_racing_b200.runner import Options, Scene, cwbvh_cuda_runner
    st = cwbvh_cuda_runner(cornell, Options(width=320, height=184, render_time=0.1, tlas=True), Scene(camera=cornell.camera))
    assert st.frames >= 1 and st.traversal_ms > 0


@pytest.mark.parametrize("w,h,shards", [(640, 360, 1), (101, 37, 1), (333, 130, 3)])
def test_frame_target_receives_the_same_pixels(cornell, w, h, shards):
    """Fused framebuffer exchange (include/tray_cuda.h, tray_cuda_scene_set_frame_target): the kernels store RGBA
    straight into a row-major frame (here on the same GPU; a peer mapping in a multi-GPU run) — same bytes as the
    compact buffer + untile path, for whole frames and for interleaved tile shards writing into ONE frame."""
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, w, h)
    sc = cuda.TrayCudaScene.from_packed(p)
    frame = cuda.frame_alloc(w * h * 4)
    try:
        sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
        want = sc.download(rgba=True)["rgba"].copy()
        sc.set_frame_target(frame)
        for s in range(shards):
            sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA, shard=s, shards=shards)
        sc.sync()
        import torch
        got = torch.as_tensor(cuda.DeviceArray(frame, (h, w, 4), "|u1", sc), device="cuda").cpu().numpy()
        assert (got.reshape(want.shape) == want).all()
        with pytest.raises(cuda.TrayCudaError):
            sc.download(rgba=True)                       # the compact RGBA buffer was not written for this frame
        sc.set_frame_target(None)
        sc.render(view, w, h, 0, cuda.RENDER_RGBA)       # primary-only shading goes through the same switch
        sc.download(rgba=True)
        # an IPC handle can be exported for the allocation (opening it needs a second process: bench.py --gpus 2)
        assert len(cuda.ipc_export(frame)) == 64
    finally:
        sc.close()
        cuda.frame_free(frame)


def test_async_readback_matches_synchronous_download(cornell):
    """tray_cuda_frame_readback_begin / _wait (double-buffered, copy stream) deliver the same bytes as
    tray_cuda_frame_download for a run of different frames, whatever the interleaving with the next render."""
    import torch
    w, h = 333, 187
    p = host.PackedScene(cornell)
    view = host.view_from_camera(cornell.camera, w, h)
    sc = cuda.TrayCudaScene.from_packed(p)
    try:
        want = []
        for f in range(5):
            sc.render(view, w, h, f, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA)
            want.append(sc.download(rgba=True)["rgba"].copy())
        assert any((want[0] != want[k]).any() for k in range(1, 5))        # the frames really differ (bounce directions)
        bufs = [torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)]
        got = []
        for f in range(5):
            slot = f & 1
            sc.render(view, w, h, f, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA, timed=False)
            sc.readback_begin(bufs[slot], slot)
            if f > 0:
                sc.readback_wait(slot ^ 1)
                got.append(bufs[slot ^ 1].copy())
        sc.readback_wait(0)
        got.append(bufs[0].copy())
        for f in range(5):
            assert np.array_equal(got[f], want[f]), f"frame {f}"
    finally:
        sc.close()


@pytest.mark.gpu
def test_roofline_probes_measure_something_sane():
    """bench.py's denominators: L2-resident streaming reads run faster than HBM-sized ones, and the L1 gather probe (every lane
    its own 16-byte record of an L1-resident table) lands between 10 and 128 bytes per clock per SM."""
    l2 = cuda.bandwidth_probe(32 << 20, 10)
    hbm = cuda.bandwidth_probe(1024 << 20, 2)
    assert l2 > hbm > 500.0
    g = cuda.l1_gather_probe(32 << 10, 50)
    sms = 148
    per_clk = g * 1e9 / (sms * 1.9e9)
    assert 10.0 < per_clk < 128.0, g
