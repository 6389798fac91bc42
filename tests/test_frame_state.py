"""The frame operator across call sequences: the state the host layer of tray_cuda.cu keeps between calls (frame slots and
"the last frame", the counting switch, the variant, the frame target, the readback slots, the scene stream), checked against
the oracle and against what include/tray_cuda.h promises.

Part A aims one test at each piece of that state: the last frame across frames-in-flight switches, refused renders, the scope
of TRAY_RENDER_COUNTERS, per-shard counters, and caller-owned streams.  Downloads whose size a library bug could change go
through ctypes into host buffers sized for the largest frame of the test plus a canary tail, so that a call that returns the
wrong frame is reported as such instead of writing past a buffer sized for the right one.

Part B drives one scene with seeded sequences of about 40 calls and checks every call against a small model of the header's
promises.  Each op is printed as it runs, so a failing case reads as its own reproduction; replay one with
`-k "flat-s48-seed2"`."""
import numpy as np
import pytest

import oracle_binding as ob
from conftest import random_rays
from tray_racing_b200 import cuda, host

pytestmark = pytest.mark.gpu

BOUNCE, RGBA, COUNTERS = cuda.RENDER_BOUNCE, cuda.RENDER_RGBA, cuda.RENDER_COUNTERS
KEEP_RAYS, ANYHIT_AO, OVERLAP = cuda.RENDER_KEEP_RAYS, cuda.RENDER_ANYHIT_AO, cuda.RENDER_OVERLAP
HIT, RAY, INVALID = ob.HIT_DTYPE, ob.RAY_DTYPE, ob.INVALID_PRIM
ITEMSIZE = {"primary": HIT.itemsize, "bounce": HIT.itemsize, "bounce_rays": RAY.itemsize, "rgba": 4}
DOWNLOAD_ORDER = ("primary", "bounce", "bounce_rays", "rgba")      # tray_cuda_frame_download's arguments

BIG = (320, 184)                                   # the largest frame any test here renders
CAP = cuda.local_items(*BIG)                       # >= its pixels and its compact entries
TAIL = 4096                                        # canary bytes behind a buffer sized for the largest frame
PATTERN = 0xA5
NO_COUNTS = dict(rays=0, nodes=0, tris=0, instances=0, hits=0)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def last_error():
    return cuda.lib().tray_cuda_last_error().decode(errors="replace")


# ---- the oracle, memoized per scene and frame ---------------------------------------------------------------------------

class Ref:
    """One packed scene, its oracle, and the oracle's frames memoized per (size, frame_count, variant, kind).
    kind: "primary" (no TRAY_RENDER_BOUNCE), "bounce", or "ao" (bounce rays traced as any-hit queries)."""

    def __init__(self, mesh, use_tlas, stride):
        self.p = host.PackedScene(mesh, use_tlas=use_tlas, tri_stride=stride)
        self.cam = mesh.camera
        self.orc = ob.Oracle.from_packed(self.p)
        self.memo = {}

    def view(self, w, h):
        return host.view_from_camera(self.cam, w, h, self.p.tlas_start)

    def scene(self):
        return cuda.TrayCudaScene.from_packed(self.p)

    def trace(self, rays, any_hit=False, variant=0):
        ob.set_variant(variant)
        try:
            return self.orc.trace(rays, counts=True, any_hit=any_hit)
        finally:
            ob.set_variant(0)

    def frame(self, w, h, fc=0, variant=0, kind="bounce"):
        key = (w, h, fc if kind != "primary" else 0, variant, kind)
        if key in self.memo:
            return self.memo[key]
        view = self.view(w, h)
        ob.set_variant(variant)
        try:
            r = self.orc.render(view, w, h, fc, flags=0 if kind == "primary" else ob.RENDER_BOUNCE, rgba=True)
            hit = r["primary"]["prim"] != INVALID
            fr = dict(kind=kind, primary=r["primary"], bounce=r["bounce"], bounce_rays=r["bounce_rays"], rgba=r["rgba"])
            # per-pixel visit counts: the primary ray of every pixel, the bounce ray of every hit pixel
            _, fr["pc"], fr["primary_totals"] = self.orc.trace(ob.primary_rays(view, w, h), counts=True)
            fr["bc"] = np.zeros(w * h, dtype=ob.COUNT_DTYPE)
            if kind != "primary":
                bh, fr["bc"][hit], fr["bounce_totals"] = self.orc.trace(r["bounce_rays"][hit], counts=True, any_hit=kind == "ao")
                if kind == "ao":                   # the bounce buffer holds the AO rays' first hits, the image their visibility
                    fr["bounce"] = r["bounce"].copy()
                    fr["bounce"][hit] = bh
                    fr["rgba"] = r["rgba"].copy()
                    fr["rgba"][hit, :3] = np.where(bh["prim"] != INVALID, 0, 255)[:, None]
        finally:
            ob.set_variant(0)
        self.memo[key] = fr
        return fr


@pytest.fixture(scope="module")
def refs(cornell):
    cache = {}

    def get(use_tlas=False, stride=48):
        if (use_tlas, stride) not in cache:
            cache[(use_tlas, stride)] = Ref(cornell, use_tlas, stride)
        return cache[(use_tlas, stride)]
    return get


@pytest.fixture(autouse=True)
def _oracle_variant_reset():
    yield
    ob.set_variant(0)


def kind_of(flags):
    return "primary" if not flags & BOUNCE else "ao" if flags & ANYHIT_AO else "bounce"


def counts(c, sel, rays, hits):
    return dict(rays=int(rays), nodes=int(c["nodes"][sel].sum()), tris=int(c["tris"][sel].sum()),
                instances=int(c["insts"][sel].sum()), hits=int(hits))


def expect_counters(fr, w, h, shard, shards):
    """(primary, bounce) counters of a counting render of `shard`: the oracle's per-ray counts over the shard's pixels"""
    own = cuda.shard_mask(w, h, shard, shards)
    hit = fr["primary"]["prim"] != INVALID
    cp = counts(fr["pc"], own, own.sum(), (hit & own).sum())
    if fr["kind"] == "primary":
        return cp, dict(NO_COUNTS)
    sel = hit & own
    return cp, counts(fr["bc"], sel, sel.sum(), (fr["bounce"]["prim"][sel] != INVALID).sum())


def trace_counters(tot, n):
    return dict(rays=n, nodes=tot["nodes"], tris=tot["tris"], instances=tot["insts"], hits=tot["hits"]), dict(NO_COUNTS)


def check_frame(got, fr, w, h, shard, shards, what):
    """`got`: row-major arrays of a frame (any of primary / bounce / bounce_rays / rgba as (w*h, 4)); the shard's pixels are the
    oracle's — hits and rays bit for bit, RGBA within one grey level (powf) — and every other pixel is zero"""
    own = cuda.shard_mask(w, h, shard, shards)
    for k in ("primary", "bounce", "bounce_rays"):
        if k in got:
            g, want = bits(got[k]).reshape(w * h, -1), bits(fr[k]).reshape(w * h, -1)
            bad = np.flatnonzero((g[own] != want[own]).any(axis=1))
            assert bad.size == 0, f"{what}: {bad.size} of {int(own.sum())} {k} records differ from the oracle's {w}x{h} frame"
            assert (g[~own] == 0).all(), f"{what}: {k} of other shards' pixels are not zero"
    if "rgba" in got:
        g = np.asarray(got["rgba"]).reshape(w * h, 4).astype(int)
        d = np.abs(g[own] - fr["rgba"][own].astype(int))
        assert d.size == 0 or d.max() <= 1, f"{what}: rgba of {int((d > 1).any(axis=1).sum())} pixels differs from the oracle's by > 1"
        assert (g[~own] == 0).all(), f"{what}: rgba of other shards' pixels is not zero"


# ---- host buffers with a canary tail, device buffers read through torch ----------------------------------------------------

def canary(itemsize, n=CAP):
    return np.full(n * itemsize + TAIL, PATTERN, dtype=np.uint8)


def canary_take(buf, itemsize, n, what):
    """the first n records of `buf`; every byte after them must still hold the pattern"""
    used = n * itemsize
    bad = np.flatnonzero(buf[used:] != PATTERN)
    if bad.size:
        tail = " and into the canary tail" if used + bad[-1] >= buf.size - TAIL else ""
        raise AssertionError(f"{what}: the call wrote {bad[-1] + 1} bytes past the {n} entries of the latest frame{tail}: "
                             "it returned an older, larger frame")
    return buf[:used]


def raw_download(sc, w, h, what, keys=DOWNLOAD_ORDER):
    """tray_cuda_frame_download through ctypes, into canary buffers sized for the largest frame"""
    bufs = {k: canary(ITEMSIZE[k]) for k in keys}
    rc = cuda.lib().tray_cuda_frame_download(sc._h, *(bufs[k].ctypes.data if k in bufs else None for k in DOWNLOAD_ORDER))
    assert rc == 0, f"{what}: tray_cuda_frame_download failed: {last_error()}"
    out = {k: canary_take(bufs[k], ITEMSIZE[k], w * h, f"{what}: download of {k}") for k in keys}
    for k, dt in (("primary", HIT), ("bounce", HIT), ("bounce_rays", RAY)):
        if k in out:
            out[k] = out[k].view(dt)
    if "rgba" in out:
        out["rgba"] = out["rgba"].reshape(-1, 4)
    return out


def raw_readback(sc, w, h, slot, what):
    """tray_cuda_frame_readback_begin / _wait through ctypes, into a canary buffer sized for the largest frame"""
    buf = canary(4)
    L = cuda.lib()
    assert L.tray_cuda_frame_readback_begin(sc._h, buf.ctypes.data, slot) == 0, f"{what}: readback_begin failed: {last_error()}"
    assert L.tray_cuda_frame_readback_wait(sc._h, slot) == 0, f"{what}: readback_wait failed: {last_error()}"
    return canary_take(buf, 4, w * h, f"{what}: readback").reshape(-1, 4)


def device_bytes(ptr, nbytes):
    import torch
    return torch.as_tensor(cuda.DeviceArray(ptr, (nbytes,), "|u1"), device="cuda").cpu().numpy()


def item_pixels(w, h, shard, shards):
    """row-major pixel of each compact work item of the shard, -1 outside the frame (traverse.cuh item_to_pixel)"""
    j = np.arange(cuda.local_items(w, h, shard, shards))
    k = shard + (j >> 8) * shards
    sub, lane = (j & 255) >> 5, j & 31
    tx = (w + 31) // 32
    px = (k % tx) * 32 + (sub & 3) * 8 + (lane & 7)
    py = (k // tx) * 8 + (sub >> 2) * 4 + (lane >> 3)
    return np.where((px < w) & (py < h), py * w + px, -1)


def untile(compact, w, h, shard, shards):
    pix = item_pixels(w, h, shard, shards)
    ok = pix >= 0
    out = np.zeros(w * h, dtype=compact.dtype)
    out[pix[ok]] = compact[:pix.size][ok]
    return out


def check_last_frame(sc, ref, w, h, fc, what, readback_slot=1):
    """download, readback, push and frame_device_ptrs all return the frame of the latest render (w x h, frame_count fc)"""
    import torch
    fr = ref.frame(w, h, fc)
    check_frame(raw_download(sc, w, h, what), fr, w, h, 0, 1, what + ", download")
    check_frame({"rgba": raw_readback(sc, w, h, readback_slot, what)}, fr, w, h, 0, 1, what + ", readback")
    items = cuda.local_items(w, h)
    dst = torch.full((CAP * 4 + TAIL,), PATTERN, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()                       # filled before the frame's stream copies into it
    sc.push(dst.data_ptr())
    sc.sync()
    pushed = canary_take(dst.cpu().numpy(), 4, items, what + ", push")
    check_frame({"rgba": untile(pushed.view(np.uint32), w, h, 0, 1).view(np.uint8)}, fr, w, h, 0, 1, what + ", push")
    dp, db, dr = sc.frame_device_ptrs()
    got = {"primary": untile(device_bytes(dp, items * 8).view(HIT), w, h, 0, 1),
           "bounce": untile(device_bytes(db, items * 8).view(HIT), w, h, 0, 1),
           "rgba": untile(device_bytes(dr, items * 4).view(np.uint32), w, h, 0, 1).view(np.uint8)}
    check_frame(got, fr, w, h, 0, 1, what + ", frame_device_ptrs")


# ---- A. directed tests ----------------------------------------------------------------------------------------------------

# older frames are larger, so that an older frame returned in place of the latest one overruns a buffer sized for it
SWITCH_FRAMES = [(320, 184, 3), (200, 120, 8), (101, 37, 5), (33, 9, 1029)]


@pytest.mark.parametrize("n_in_flight,renders", [(2, 1), (2, 2), (2, 3), (3, 1), (3, 2), (3, 3), (3, 4)])
def test_last_frame_survives_frames_in_flight_switches(refs, n_in_flight, renders):
    """tray_cuda_scene_set_frames_in_flight changes the slot the next render takes, never "the last frame": after
    1 -> 3 -> 2 -> 1 switches without a render in between, every read of the last frame returns the latest render."""
    ref = refs()
    sc = ref.scene()
    try:
        sc.set_frames_in_flight(n_in_flight)
        frames = SWITCH_FRAMES[:renders]
        for i, (w, h, fc) in enumerate(frames):
            sc.render(ref.view(w, h), w, h, fc, BOUNCE | RGBA | KEEP_RAYS | (OVERLAP if i & 1 else 0), timed=False)
        w, h, fc = frames[-1]
        check_last_frame(sc, ref, w, h, fc, f"{renders} renders with {n_in_flight} in flight")
        path = [n_in_flight]
        for n in (1, 3, 2, 1):
            sc.set_frames_in_flight(n)
            path.append(n)
            check_last_frame(sc, ref, w, h, fc, f"{renders} renders, then frames in flight {' -> '.join(map(str, path))}")
        for n, (w, h, fc) in ((1, (101, 37, 6)), (2, (200, 120, 2)), (2, (33, 9, 4))):     # and the next renders land as usual
            sc.set_frames_in_flight(n)
            sc.render(ref.view(w, h), w, h, fc, BOUNCE | RGBA | KEEP_RAYS, timed=False)
            check_last_frame(sc, ref, w, h, fc, f"render of {w}x{h} after the switches")
    finally:
        sc.close()


REFUSALS = {
    "variant_counters": (cuda.VARIANT_TIE_LAST, dict(w=320, h=184, flags=BOUNCE | RGBA | COUNTERS), "without counters"),
    "variant_anyhit_ao": (cuda.VARIANT_BOX_DIVIDE, dict(w=320, h=184, flags=BOUNCE | RGBA | ANYHIT_AO), "without counters"),
    "zero_width": (0, dict(w=0, h=184, flags=BOUNCE | RGBA), "bad frame size"),
    "shard_out_of_range": (0, dict(w=320, h=184, flags=BOUNCE | RGBA | COUNTERS, shard=3, shards=3), "bad frame size"),
}


@pytest.mark.parametrize("counting", [False, True], ids=["counting_off", "counting_on"])
@pytest.mark.parametrize("n_in_flight", [1, 2])
@pytest.mark.parametrize("refusal", list(REFUSALS))
def test_refused_render_changes_nothing(refs, refusal, n_in_flight, counting):
    """A render that tray_cuda_render refuses leaves the last frame (which still downloads with its own hits), the counters,
    the counting state of batch traces and the slot the next render takes exactly as they were."""
    ref = refs()
    variant, kw, match = REFUSALS[refusal]
    sc = ref.scene()
    try:
        sc.set_frames_in_flight(n_in_flight)
        sc.set_counting(counting)
        w, h, fc = 101, 37, 5
        sc.render(ref.view(w, h), w, h, fc, BOUNCE | RGBA | KEEP_RAYS | COUNTERS, timed=False)
        fr = ref.frame(w, h, fc)
        before = sc.counters()
        assert before == expect_counters(fr, w, h, 0, 1)
        stream_before = sc.frame_stream(-1)
        sc.set_variant(variant)
        with pytest.raises(cuda.TrayCudaError, match=match):
            sc.render(ref.view(max(kw["w"], 1), kw["h"]), kw["w"], kw["h"], 7, kw["flags"], kw.get("shard", 0), kw.get("shards", 1))
        sc.set_variant(0)
        what = f"after a refused render ({refusal})"
        check_frame(raw_download(sc, w, h, what), fr, w, h, 0, 1, what + ", download of the last frame")
        assert sc.counters() == before, f"{what}: the counters changed"
        rays = random_rays(3001, 5)
        hits, _, tot = ref.trace(rays)
        got = sc.traverse(rays)
        assert (bits(got) == bits(hits)).all(), f"{what}: batch trace differs from the oracle"
        if counting:
            assert sc.counters() == trace_counters(tot, len(rays)), f"{what}: tray_cuda_set_counting(1) no longer counts batch traces"
        else:
            assert sc.counters() == before, f"{what}: a batch trace counted, though tray_cuda_set_counting was never turned on"
        w2, h2, fc2 = 33, 9, 2
        sc.render(ref.view(w2, h2), w2, h2, fc2, BOUNCE | RGBA | KEEP_RAYS, timed=False)
        if n_in_flight == 2:
            assert sc.frame_stream(-1) != stream_before, f"{what}: the next render took the slot of the last frame (the refusal advanced it)"
        check_last_frame(sc, ref, w2, h2, fc2, f"{what}, the next render")
    finally:
        sc.close()


@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
def test_counters_flag_is_scoped_to_its_render(refs, use_tlas):
    """TRAY_RENDER_COUNTERS counts the render that carries it and nothing else; tray_cuda_set_counting alone governs batch
    traces; neither changes the other.  A variant trace after a counting render runs, and matches the oracle under it."""
    ref = refs(use_tlas)
    sc = ref.scene()
    v = cuda.VARIANT_TIE_LAST | cuda.VARIANT_ZERODIR_BOX_ONLY
    rays = random_rays(4099, 9, axis_fraction=0.1)
    try:
        w, h = 200, 120
        view = ref.view(w, h)
        sc.render(view, w, h, 1, BOUNCE | COUNTERS, timed=False)
        after_render = sc.counters()
        assert after_render == expect_counters(ref.frame(w, h, 1), w, h, 0, 1)
        hits, _, tot = ref.trace(rays)
        assert (bits(sc.traverse(rays)) == bits(hits)).all()
        assert sc.counters() == after_render, "a batch trace after a TRAY_RENDER_COUNTERS render counted: the flag stuck to the scene"
        sc.set_variant(v)
        try:
            got = sc.traverse(rays)
        except cuda.TrayCudaError as e:
            raise AssertionError(f"a variant batch trace after a TRAY_RENDER_COUNTERS render was refused: {e}") from None
        want, _, _ = ref.trace(rays, variant=v)
        assert (bits(got) == bits(want)).all(), f"variant 0x{v:x} batch trace differs from the oracle under it"
        sc.set_variant(0)
        # tray_cuda_set_counting(1): a render without the flag neither counts nor turns batch counting off
        sc.set_counting(True)
        sc.render(view, w, h, 2, BOUNCE, timed=False)
        assert sc.counters() == after_render, "a render without TRAY_RENDER_COUNTERS counted"
        assert (bits(sc.traverse(rays)) == bits(hits)).all()
        assert sc.counters() == trace_counters(tot, len(rays)), \
            "a render without TRAY_RENDER_COUNTERS turned off tray_cuda_set_counting: the batch trace did not count"
        # a counting render leaves batch counting on, and after set_counting(0) a render with the flag still counts
        sc.render(view, w, h, 3, BOUNCE | COUNTERS, timed=False)
        assert sc.counters() == expect_counters(ref.frame(w, h, 3), w, h, 0, 1)
        any_hits, _, any_tot = ref.trace(rays, any_hit=True)
        assert (bits(sc.traverse(rays, any_hit=True)) == bits(any_hits)).all()
        assert sc.counters() == trace_counters(any_tot, len(rays)), "batch counting stopped after a counting render"
        sc.set_counting(False)
        sc.render(view, w, h, 4, BOUNCE | ANYHIT_AO | COUNTERS, timed=False)
        after_ao = sc.counters()
        assert after_ao == expect_counters(ref.frame(w, h, 4, kind="ao"), w, h, 0, 1)
        sc.traverse(rays)
        assert sc.counters() == after_ao, "a batch trace counted after tray_cuda_set_counting(0)"
        # under a variant, batch counting is refused while a render without the flag runs
        sc.set_counting(True)
        sc.set_variant(v)
        with pytest.raises(cuda.TrayCudaError, match="without counters"):
            sc.traverse(rays)
        sc.render(view, w, h, 5, BOUNCE | KEEP_RAYS, timed=False)
        check_frame(raw_download(sc, w, h, "variant render", ("primary", "bounce", "bounce_rays")),
                    ref.frame(w, h, 5, variant=v), w, h, 0, 1, f"variant 0x{v:x} render under tray_cuda_set_counting(1)")
        assert sc.counters() == after_ao
    finally:
        sc.close()


@pytest.mark.parametrize("overlap", [False, True], ids=["two_launch", "overlap"])
@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
@pytest.mark.parametrize("w,h", [(200, 120), (101, 37), (33, 9)])
@pytest.mark.parametrize("shards", [1, 2, 3, 8])
def test_shard_counters_match_the_oracle(refs, shards, w, h, use_tlas, overlap):
    """bench.py sums the counters of render(.., COUNTERS, rank, world) over ranks: each shard's primary and bounce counters are
    the oracle's per-ray counts over the shard's pixels (padding rays of partial tiles excluded), and they add up to the frame's."""
    ref = refs(use_tlas)
    fr = ref.frame(w, h, 0)
    sc = ref.scene()
    total = [dict(NO_COUNTS), dict(NO_COUNTS)]
    try:
        for s in range(shards):
            sc.render(ref.view(w, h), w, h, 0, BOUNCE | COUNTERS | (OVERLAP if overlap else 0), s, shards, timed=False)
            got, want = sc.counters(), expect_counters(fr, w, h, s, shards)
            for kind, g, e in zip(("primary", "bounce"), got, want):
                assert g == e, f"shard {s} of {shards}, {kind} counters: got {g}, the oracle's per-ray counts over the shard give {e}"
            for acc, g in zip(total, got):
                for k in acc:
                    acc[k] += g[k]
        for acc, tot in zip(total, (fr["primary_totals"], fr["bounce_totals"])):
            assert acc == dict(rays=tot["rays"], nodes=tot["nodes"], tris=tot["tris"], instances=tot["insts"], hits=tot["hits"])
    finally:
        sc.close()


def test_caller_stream_orders_frames_traces_and_torch_ops(refs):
    """tray_cuda_scene_set_stream with a torch stream: frames (one and two in flight), batch traces (plain and pipelined),
    readback and download match the oracle; a torch op enqueued on the stream right after a render sees the finished frame
    without a synchronise; frame_stream(-1) is the stream of the last frame; set_stream(0) restores the scene's own stream."""
    import torch
    ref = refs()
    sc = ref.scene()
    st = torch.cuda.Stream()
    w, h = 320, 184
    view = ref.view(w, h)
    try:
        own = sc.frame_stream(0)
        sc.set_stream(st.cuda_stream)
        assert sc.frame_stream(0) == st.cuda_stream and own != st.cuda_stream
        pinned = torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True).numpy()
        for n in (1, 2):
            sc.set_frames_in_flight(n)
            for fc in (0, 3, 4):
                sc.render(view, w, h, fc, BOUNCE | RGBA | KEEP_RAYS, timed=False)
                fr = ref.frame(w, h, fc)
                sc.readback_begin(pinned, fc & 1)
                sc.readback_wait(fc & 1)
                check_frame({"rgba": pinned}, fr, w, h, 0, 1, f"{n} in flight, frame {fc}, readback")
                check_frame(sc.download(primary=True, bounce=True, bounce_rays=True, rgba=True), fr, w, h, 0, 1,
                            f"{n} in flight, frame {fc}, download")
        for n_rays in (1000, (1 << 18) + 1001):                       # the plain path and the host pipeline
            rays = random_rays(n_rays, n_rays)
            assert (bits(sc.traverse(rays)) == bits(ref.trace(rays)[0])).all(), f"{n_rays} rays on the caller's stream"
        # one frame in flight: the frame runs on the caller's stream, so a torch op enqueued there sees it
        sc.set_frames_in_flight(1)
        for fc, shards in ((6, 1), (7, 3)):
            fr = ref.frame(w, h, fc)
            for s in range(shards):
                with torch.cuda.stream(st):
                    frame = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
                    sc.render(view, w, h, fc, BOUNCE | RGBA, s, shards, timed=False)
                    assert sc.frame_stream(-1) == st.cuda_stream
                    _, _, d_rgba = sc.frame_device_ptrs()
                    sc.untile_rgba(d_rgba, w, h, s, shards, frame.data_ptr())
                    snap = frame.clone()
                st.synchronize()
                got = snap.cpu().numpy()
                check_frame({"rgba": got}, fr, w, h, s, shards, f"frame {fc} shard {s} of {shards}, untiled on the caller's stream")
                assert (got == sc.download(rgba=True)["rgba"]).all(), "tray_cuda_untile_rgba differs from download(rgba=True)"
        # two frames in flight: the last frame's stream alternates, and torch work on it sees that frame
        sc.set_frames_in_flight(2)
        seen = []
        for fc in (8, 9, 10):
            sc.render(view, w, h, fc, BOUNCE | RGBA, timed=False)
            fs = torch.cuda.ExternalStream(sc.frame_stream(-1))
            seen.append(fs.cuda_stream)
            with torch.cuda.stream(fs):
                frame = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
                _, _, d_rgba = sc.frame_device_ptrs()
                sc.untile_rgba(d_rgba, w, h, 0, 1, frame.data_ptr())
                snap = frame.clone()
            fs.synchronize()
            check_frame({"rgba": snap.cpu().numpy()}, ref.frame(w, h, fc), w, h, 0, 1, f"frame {fc} on frame_stream(-1)")
        assert seen[0] != seen[1] and seen[0] == seen[2] and st.cuda_stream in seen[:2], seen
        sc.set_stream(0)
        assert sc.frame_stream(0) == own
        sc.set_frames_in_flight(1)
        sc.render(view, w, h, 11, BOUNCE | RGBA, timed=False)
        assert sc.frame_stream(-1) == own
        check_frame(sc.download(primary=True, rgba=True), ref.frame(w, h, 11), w, h, 0, 1, "after set_stream(0)")
    finally:
        sc.close()


# ---- B. seeded call sequences against a model of the header -----------------------------------------------------------------

SEQ_SIZES = [(320, 184), (101, 37), (33, 9), (7, 3)]
SEQ_FRAME_COUNTS = [0, 1, 6, 1029]
SEQ_VARIANTS = [cuda.VARIANT_BOX_DIVIDE, cuda.VARIANT_TIE_LAST, cuda.VARIANT_BOX_TMIN_RAY, cuda.VARIANT_ZERODIR_BOX_ONLY]
SEQ_OPS = ["render"] * 7 + ["render_frame_ms", "frames_in_flight", "frame_target", "variant", "counting", "stream", "counters"] + \
          ["traverse"] * 3 + ["readback_begin"] * 2 + ["readback_wait", "download", "download", "target_contents"]
SEQ_LEN = 40
SEQ_SEEDS = range(4)
FLAG_NAMES = {BOUNCE: "BOUNCE", RGBA: "RGBA", KEEP_RAYS: "KEEP_RAYS", COUNTERS: "COUNTERS", ANYHIT_AO: "ANYHIT_AO", OVERLAP: "OVERLAP"}


def flag_str(flags):
    return "|".join(n for f, n in FLAG_NAMES.items() if flags & f) or "0"


class Model:
    """What include/tray_cuda.h promises about one scene's state, as far as the sequence ops touch it."""

    def __init__(self):
        self.frame = None            # the last successful render: dict(w, h, fc, shard, shards, flags, variant, target, fr)
        self.counting = False
        self.variant = 0
        self.target = None           # index of the frame target, None = the compact buffer
        self.n_in_flight = 1
        self.counters = (dict(NO_COUNTS), dict(NO_COUNTS))
        self.targets = []            # model contents of each frame target, bytes
        self.pending = {}            # readback slot -> (host buffer, expected rgba, description)

    def render_refused(self, flags):
        return self.variant != 0 and bool(flags & COUNTERS or (flags & BOUNCE and flags & ANYHIT_AO))

    def rendered(self, ref, w, h, fc, flags, shard, shards):
        kind = kind_of(flags)
        fr = ref.frame(w, h, fc, self.variant, kind)
        self.frame = dict(w=w, h=h, fc=fc, shard=shard, shards=shards, flags=flags, variant=self.variant, target=self.target, fr=fr)
        if flags & COUNTERS:
            self.counters = expect_counters(fr, w, h, shard, shards)
        if flags & RGBA and self.target is not None:
            own = cuda.shard_mask(w, h, shard, shards)
            t = self.targets[self.target][:w * h * 4].reshape(-1, 4)
            t[own] = fr["rgba"][own]

    def expected_rgba(self):
        f = self.frame
        if f["target"] is not None:
            return self.targets[f["target"]][:f["w"] * f["h"] * 4].reshape(-1, 4).copy()
        own = cuda.shard_mask(f["w"], f["h"], f["shard"], f["shards"])
        out = np.zeros((f["w"] * f["h"], 4), dtype=np.uint8)
        out[own] = f["fr"]["rgba"][own]
        return out

    def downloadable(self, key):
        fl = self.frame["flags"]
        return {"primary": True, "bounce": bool(fl & BOUNCE), "bounce_rays": bool(fl & BOUNCE and fl & KEEP_RAYS),
                "rgba": bool(fl & RGBA) and self.frame["target"] is None}[key]


def assert_rgba_close(got, want, what):
    d = np.abs(np.asarray(got).reshape(-1, 4).astype(int) - want.reshape(-1, 4).astype(int))
    assert d.size == 0 or d.max() <= 1, f"{what}: {int((d > 1).any(axis=1).sum())} pixels differ from the model by more than 1"


@pytest.mark.parametrize("seed", SEQ_SEEDS, ids=[f"seed{s}" for s in SEQ_SEEDS])
@pytest.mark.parametrize("stride", [48, 24], ids=["s48", "s24"])
@pytest.mark.parametrize("use_tlas", [False, True], ids=["flat", "tlas"])
def test_call_sequence_follows_the_header(refs, use_tlas, stride, seed):
    import torch
    ref = refs(use_tlas, stride)
    rng = np.random.default_rng([seed, int(use_tlas), stride])
    m = Model()
    sc = ref.scene()
    st = torch.cuda.Stream()
    target_bufs = [torch.zeros(BIG[0] * BIG[1] * 4, dtype=torch.uint8, device="cuda") for _ in range(2)]
    m.targets = [np.zeros(BIG[0] * BIG[1] * 4, dtype=np.uint8) for _ in target_bufs]
    torch.cuda.synchronize()                       # zeroed before a frame stream stores into them

    def check_pending(slot, what):
        buf, want, desc = m.pending.pop(slot)
        assert_rgba_close(buf, want, f"{what}: readback slot {slot} of {desc}")

    try:
        for i in range(SEQ_LEN):
            op = SEQ_OPS[rng.integers(len(SEQ_OPS))]
            if op in ("download", "readback_begin") and m.frame is None:
                op = "render"
            if op in ("render", "render_frame_ms"):
                w, h = SEQ_SIZES[rng.integers(len(SEQ_SIZES))]
                fc = SEQ_FRAME_COUNTS[rng.integers(len(SEQ_FRAME_COUNTS))]
                flags = 0
                for f, p in ((BOUNCE, 0.7), (RGBA, 0.6), (KEEP_RAYS, 0.4), (COUNTERS, 0.35), (ANYHIT_AO, 0.25), (OVERLAP, 0.4)):
                    flags |= f if rng.random() < p else 0
                shards = [1, 1, 1, 2, 3, 8][rng.integers(6)]
                shard = int(rng.integers(shards))
                what = f"op {i}: {op} {w}x{h} frame {fc} {flag_str(flags)} shard {shard}/{shards}"
                print(what, flush=True)
                call = (lambda: sc.render(ref.view(w, h), w, h, fc, flags, shard, shards, timed=bool(rng.random() < 0.5))) \
                    if op == "render" else (lambda: sc.render_frame_ms(ref.view(w, h), w, h, fc, flags, shard, shards))
                if m.render_refused(flags):
                    with pytest.raises(cuda.TrayCudaError, match="without counters"):
                        call()
                    print("  refused, as the header says", flush=True)
                    continue
                r = call()
                if op == "render_frame_ms":
                    assert r >= 0, what
                m.rendered(ref, w, h, fc, flags, shard, shards)
                if flags & COUNTERS:
                    assert sc.counters() == m.counters, f"{what}: counters differ from the oracle's over the shard"
            elif op == "frames_in_flight":
                n = 1 if m.target is not None else int(rng.integers(1, 4))     # frames in flight into one target race
                print(f"op {i}: set_frames_in_flight({n})", flush=True)
                sc.set_frames_in_flight(n)
                m.n_in_flight = n
            elif op == "frame_target":
                k = None if m.n_in_flight > 1 else [None, 0, 1][rng.integers(3)]
                print(f"op {i}: set_frame_target({k})", flush=True)
                sc.set_frame_target(None if k is None else target_bufs[k].data_ptr())
                m.target = k
            elif op == "variant":
                v = 0 if rng.random() < 0.4 else SEQ_VARIANTS[rng.integers(len(SEQ_VARIANTS))]
                print(f"op {i}: set_variant(0x{v:x})", flush=True)
                sc.set_variant(v)
                m.variant = v
            elif op == "counting":
                on = bool(rng.random() < 0.5)
                print(f"op {i}: set_counting({on})", flush=True)
                sc.set_counting(on)
                m.counting = on
            elif op == "stream":
                mine = bool(rng.random() < 0.5)
                print(f"op {i}: set_stream({'torch stream' if mine else 0})", flush=True)
                sc.set_stream(st.cuda_stream if mine else 0)
            elif op == "counters":
                print(f"op {i}: counters", flush=True)
                assert sc.counters() == m.counters, f"op {i}: counters changed since the last call that counted"
            elif op == "traverse":
                n = int(rng.integers(1, 5001))
                any_hit = bool(rng.random() < 0.3)
                rays = random_rays(n, int(rng.integers(1 << 30)))
                what = f"op {i}: traverse {n} rays{' any_hit' if any_hit else ''}"
                print(what, flush=True)
                if m.variant and (m.counting or any_hit):
                    with pytest.raises(cuda.TrayCudaError, match="without counters"):
                        sc.traverse(rays, any_hit=any_hit)
                    print("  refused, as the header says", flush=True)
                    continue
                want, _, tot = ref.trace(rays, any_hit, m.variant)
                got = sc.traverse(rays, any_hit=any_hit)
                assert (bits(got) == bits(want)).all(), f"{what}: {(got['prim'] != want['prim']).sum()} hits differ from the oracle"
                if m.counting:
                    m.counters = trace_counters(tot, n)
                    assert sc.counters() == m.counters, f"{what}: counters differ from the oracle's totals"
            elif op == "readback_begin":
                slot = int(rng.integers(4))
                f = m.frame
                what = f"op {i}: readback_begin(slot {slot}) of {f['w']}x{f['h']} {flag_str(f['flags'])}"
                print(what, flush=True)
                buf = torch.empty((f["h"], f["w"], 4), dtype=torch.uint8, pin_memory=True).numpy()
                if not f["flags"] & RGBA:
                    with pytest.raises(cuda.TrayCudaError, match="without TRAY_RENDER_RGBA"):
                        sc.readback_begin(buf, slot)
                    print("  refused, as the header says", flush=True)
                    continue
                sc.readback_begin(buf, slot)
                if slot in m.pending:                     # begin waited for the previous copy out of this staging slot
                    check_pending(slot, what)
                m.pending[slot] = (buf, m.expected_rgba(), what)
            elif op == "readback_wait":
                slot = int(rng.integers(4))
                print(f"op {i}: readback_wait(slot {slot})", flush=True)
                sc.readback_wait(slot)
                if slot in m.pending:
                    check_pending(slot, f"op {i}")
            elif op == "download":
                keys = [k for k in DOWNLOAD_ORDER if rng.random() < 0.5] or ["primary"]
                f = m.frame
                what = f"op {i}: download {'+'.join(keys)} of {f['w']}x{f['h']} {flag_str(f['flags'])} shard {f['shard']}/{f['shards']}"
                print(what, flush=True)
                if not all(m.downloadable(k) for k in keys):
                    with pytest.raises(cuda.TrayCudaError, match="rendered without"):
                        sc.download(**{k: True for k in keys})
                    print("  refused, as the header says", flush=True)
                    continue
                got = sc.download(**{k: True for k in keys})
                rgba = got.pop("rgba", None)
                check_frame(got, f["fr"], f["w"], f["h"], f["shard"], f["shards"], what)
                if rgba is not None:
                    assert_rgba_close(rgba, m.expected_rgba(), what)
            elif op == "target_contents":
                print(f"op {i}: frame targets read through torch", flush=True)
                sc.sync()
                for k, buf in enumerate(target_bufs):
                    assert_rgba_close(buf.cpu().numpy(), m.targets[k], f"op {i}: frame target {k}")
        for slot in list(m.pending):
            sc.readback_wait(slot)
            check_pending(slot, "end of sequence")
        sc.sync()
    finally:
        sc.close()
