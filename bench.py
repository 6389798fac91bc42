#!/usr/bin/env python
"""bench.py — the headline measurement of the tray_cuda backend (contract: see the task's bench.py section).

Metric (BASELINE.json): Mrays/s, primary + 1-spp diffuse-bounce rays, on the 2.88 M-triangle hairball-like scene
(config C3), with the achieved fraction of the memory roofline and the host-CPU restatement of rt_cpu beside it.

A "step" is one frame of the reference's render loop body (reference src/rt_cpu/rt_cpu.rs:35-91): generate the
primary rays of this rank's image tiles, closest-hit traversal, one cosine bounce ray per hit pixel, second
traversal, RGBA8 — then the framebuffer gather to rank 0 (the path's one exchange step) and its assembly.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (under torchrun for N > 1)
  python bench.py ... --dump-outputs DIR                        also write the last timed step's frame to DIR/*.npy
  python bench.py --impl reference ...                          the reference's CPU algorithm (oracle port) on host cores

Weak scaling: the frame holds ~N x 1920x1080 pixels (same camera, finer sampling), tiles interleaved over N ranks,
BVH replicated, so every GPU traces the same number of rays as at N = 1.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC, UNIT = "Mrays/s primary+diffuse", "Mrays/s"
TRI_STRIDE = 48
# BASELINE.json configs that are bench lines.  c3 (configs[2], the one the metric's 1-GPU target is quoted on) is the default
# and the only one the driver runs; c1 / c2 (configs[0], configs[1]) are the small 1080p scenes; c4 / c5 (configs[3], configs[4]) are the multi-GPU configs: a FIXED 3840x2160 frame
# tile-sharded over the ranks (strong scaling), c5 through the two-level (--tlas) traversal.
WORKLOADS = {
    "c1": dict(scene="kitchen", seed=1, w=1920, h=1080, tlas=False, scaling="weak",
               label="C1 kitchen-sized 56,939-tri interior (kitchen.ron camera)"),
    "c2": dict(scene="demoscene", seed=2, w=1920, h=1080, tlas=False, scaling="weak",
               label="C2 demoscene stand-in, 2.10M-tri fBm height field"),
    "c3": dict(scene="hairball", seed=3, w=1920, h=1080, tlas=False, scaling="weak",
               label="C3 hairball-like 2.88M-tri soup"),
    "c4": dict(scene="sanmiguel", seed=4, w=3840, h=2160, tlas=False, scaling="strong",
               label="C4 San-Miguel-sized 5.08M-tri scene"),
    "c5": dict(scene="caldera", seed=5, w=3840, h=2160, tlas=True, scaling="strong",
               label="C5 Caldera-sized 19.26M-tri scene, 4096 BLAS + TLAS (--tlas)"),
}
WL = WORKLOADS["c3"]


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner, torchrun notes), so
    stdout is pointed at stderr for the whole run and the result line alone goes to the real stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def frame_size(n_gpus: int):
    if WL["scaling"] == "strong":
        return WL["w"], WL["h"]
    s = n_gpus ** 0.5
    return int(round(WL["w"] * s / 8)) * 8, int(round(WL["h"] * s / 8)) * 8


def workload_name(w, h, n):
    px = f"{n} x {WL['w']}x{WL['h']} px" if WL["scaling"] == "weak" else f"fixed frame, 1/{n} of the tiles per GPU"
    return f"{WL['label']}, {w}x{h} ({px}), primary + 1spp diffuse bounce, ploc-style CWBVH"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_figure(key):
    """a per-launch figure of the committed ncu capture (profiles/roofline_traffic.json), or None"""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(p))[key]
    except Exception:
        return None


DUMP_BYTES = 64_000_000


def dump_frame(path, frame, w, h):
    """--dump-outputs: the RGBA8 frame a step hands its caller (a device tensor or a host array), as float32 [h, w, 4] in
    `path`/frame_rgba.npy.  A frame larger than DUMP_BYTES is cut to a fixed, seeded sample of pixels, [n, 4], with their
    row-major pixel indices in frame_pixel_index.npy."""
    os.makedirs(path, exist_ok=True)
    frame = frame.cpu().numpy() if hasattr(frame, "cpu") else np.ascontiguousarray(frame)
    rgba = frame.view(np.uint8).reshape(h, w, 4).astype(np.float32)
    if rgba.nbytes <= DUMP_BYTES - 4096:
        np.save(os.path.join(path, "frame_rgba.npy"), rgba)
        if os.path.exists(os.path.join(path, "frame_pixel_index.npy")):     # left by an earlier, sampled dump into DIR
            os.remove(os.path.join(path, "frame_pixel_index.npy"))
        return
    idx = np.sort(np.random.default_rng(0).choice(h * w, size=(DUMP_BYTES - 4096) // (16 + 8), replace=False))
    np.save(os.path.join(path, "frame_rgba.npy"), rgba.reshape(-1, 4)[idx])
    np.save(os.path.join(path, "frame_pixel_index.npy"), idx.astype(np.float64))


def build_scene(nthreads=0):
    from tray_racing_b200 import host
    mesh = host.Mesh.generate(WL["scene"], WL["seed"], 1.0)
    packed = host.PackedScene(mesh, use_tlas=WL["tlas"], tri_stride=TRI_STRIDE, nthreads=nthreads)
    return mesh, packed


# ---------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Every host core this process may use — NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to its workers."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_oracle_run(packed, mesh, w, h, seconds_budget: float, frames_min: int):
    """The oracle (C restatement of rt_cpu) timed on this host's cores on a bounded sample of the workload: whole frames of
    the same scene, camera and frame size (primary + bounce), all host threads, as many frames as fit the time budget."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    from tray_racing_b200 import host
    orc = ob.Oracle.from_packed(packed)
    view = host.view_from_camera(mesh.camera, w, h, packed.tlas_start)
    threads = host_threads()
    orc.render(view, w, h, 0, nthreads=threads)                      # warm-up frame (page in the BVH)
    times, rays = [], 0
    t_start = time.perf_counter()
    while len(times) < frames_min or (time.perf_counter() - t_start) < seconds_budget:
        t0 = time.perf_counter()
        r = orc.render(view, w, h, 0, nthreads=threads)
        times.append(time.perf_counter() - t0)
        rays = r["primary_totals"]["rays"] + r["bounce_totals"]["rays"]
        if len(times) >= 64:
            break
    mean = sum(times) / len(times)
    return {"value": rays / mean / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "simd": "AVX2 node test (8 children per vector), scalar triangle test" if ob.simd() else "scalar",
            "sample": f"{len(times)} whole frames of the workload ({w}x{h}, {rays} rays/frame, primary+bounce), mean frame time",
            "ms_per_frame": mean * 1e3, "rays_per_frame": rays}, times


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm for this path.  The Rust reference cannot be built in this
    image (no cargo/rustc; arithmetic in an un-vendored crate), so this is the oracle port, all host threads, on the SAME
    frame as our arm (frame_size(): same scene, camera, width and height)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    mesh, packed = build_scene(nthreads=host_threads())
    w, h = frame_size(args.gpus)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    from tray_racing_b200 import host
    orc = ob.Oracle.from_packed(packed)
    view = host.view_from_camera(mesh.camera, w, h, packed.tlas_start)
    threads = host_threads()
    for _ in range(args.warmup):
        orc.render(view, w, h, 0, nthreads=threads)
    t0 = time.perf_counter()
    rays = 0
    for i in range(args.steps):
        # with --dump-outputs the last step also shades the RGBA8 frame our arm's steps produce
        r = orc.render(view, w, h, 0, nthreads=threads, rgba=bool(args.dump_outputs) and i == args.steps - 1)
        rays += r["primary_totals"]["rays"] + r["bounce_totals"]["rays"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_frame(args.dump_outputs, r["rgba"], w, h)
    val = rays / dt / 1e6
    sample = f"each step = one whole {w}x{h} frame of the workload (same scene, camera and size as our arm), primary+bounce"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": WL["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(w, h, args.gpus), "sample": sample, "n_tris": packed.n_tris, "n_nodes": packed.n_nodes},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------------
class Rig:
    """One rank's scene + the plumbing of a step: render this rank's tile shard, then the path's one exchange step
    (every shard's pixels reach ONE row-major frame on rank 0) — for one or two frames in flight.

    exchange "peer": rank 0 owns row-major frames that every rank maps (CUDA IPC); the traversal kernels store finished
        pixels straight into them over NVLink.  Completion is a set of 32-bit flags moved by the stream front-end
        (tray_cuda_frame_signal / _wait_flag = cuStreamWriteValue32 / cuStreamWaitValue32): rank k writes "frame seq is there"
        into rank 0's memory behind its kernels, rank 0's frame stream waits for all of them, and rank 0 writes "target t is
        consumed" back before a rank may overwrite that target four frames later.  No collective kernel: with two frames in
        flight one would wait for an SM slot until the next frame's persistent grid drains.  (--exchange peer-nccl keeps the
        round-1 barrier, a 4-byte all-reduce, for comparison.)
    exchange "nccl": gather of the compact RGBA8 shards to rank 0 + one untile launch per shard (one frame at a time).
    single GPU: compact buffer + one untile launch into the row-major frame."""

    def __init__(self, torch, dist, cuda, scene, view, w, h, rank, world, local_rank, stream, exchange):
        self.torch, self.dist, self.cuda, self.scene, self.view = torch, dist, cuda, scene, view
        self.w, self.h, self.rank, self.world, self.local_rank, self.main = w, h, rank, world, local_rank, stream
        self.exchange = exchange
        self.in_flight, self.flags = 1, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA
        self.max_items = cuda.local_items(w, h, 0, world)
        self.frames = [torch.zeros(h * w, dtype=torch.int32, device="cuda") for _ in range(2)] if (rank == 0 and (world == 1 or exchange == "nccl")) else None
        self.gathered = [torch.empty(self.max_items, dtype=torch.int32, device="cuda") for _ in range(world)] if (rank == 0 and world > 1 and exchange == "nccl") else None
        self.peer_frames, self.peer_ptrs = [], []          # 4 targets: a frame's target is reused 4 frames later
        self.done = [torch.zeros(1, dtype=torch.int32, device="cuda") for _ in range(3)]
        self.groups = [None, None, None]
        self.ext = {}
        self.k = self.seq = 0
        self.local_flags, self.remote_flags, self.target_seq = None, {}, [0, 0, 0, 0]
        peer = world > 1 and exchange in ("peer", "peer-nccl", "push")
        self.frame_bytes = w * h * 4
        # "push": the 4 rotating targets on rank 0 are STAGING arrays (every shard's compact buffer back to back) followed by the
        # row-major frame they are untiled into; "peer": they are the row-major frames the kernels store into
        self.target_bytes = (world * self.max_items * 4 + self.frame_bytes) if exchange == "push" else self.frame_bytes
        if peer:
            for _ in range(4):
                if rank == 0:
                    f = cuda.frame_alloc(self.target_bytes, local_rank)
                    self.peer_frames.append(f)
                    box = [cuda.ipc_export(f, local_rank)]
                else:
                    box = [None]
                dist.broadcast_object_list(box, src=0)
                self.peer_ptrs.append(self.peer_frames[-1] if rank == 0 else cuda.ipc_open(box[0], local_rank))
        if peer and exchange == "peer-nccl":
            self.groups = [dist.new_group(list(range(world))) for _ in range(3)]
        elif peer:      # "peer" and "push" complete their frames with flags
            # flag words: rank 0's buffer holds "arrived" [r * 4 + slot]; every rank's buffer holds "consumed" [32 + target]
            self.local_flags = cuda.frame_alloc(256, local_rank)
            handles = [None] * world
            dist.all_gather_object(handles, cuda.ipc_export(self.local_flags, local_rank))
            if rank == 0:
                self.remote_flags = {r: cuda.ipc_open(handles[r], local_rank) for r in range(1, world)}
            else:
                self.remote_flags = {0: cuda.ipc_open(handles[0], local_rank)}
            torch.cuda.synchronize()
            dist.barrier()

    def torch_stream(self, ptr):
        if ptr == self.main.cuda_stream:
            return self.main
        if ptr not in self.ext:
            self.ext[ptr] = self.torch.cuda.ExternalStream(ptr)
        return self.ext[ptr]

    def configure(self, overlap, in_flight):
        self.scene.sync()
        self.flags = self.cuda.RENDER_BOUNCE | self.cuda.RENDER_RGBA | (self.cuda.RENDER_OVERLAP if overlap else 0)
        self.in_flight = in_flight if (self.world == 1 or self.exchange in ("peer", "peer-nccl", "push", "none")) else 1
        self.scene.set_frames_in_flight(self.in_flight)
        self.k = 0                                         # (self.seq keeps counting: the flags only ever grow)

    def step(self, copy_out=None):
        """one frame; `copy_out(k)` (rank 0) is called where the COMPLETE frame k may be read on the frame's own stream"""
        sc, k = self.scene, self.k
        self.k += 1
        if self.world > 1 and self.exchange == "push":
            # every rank keeps its compact shard local and moves it with ONE DMA copy into rank 0's staging (no SM, full NVLink
            # packets); flags complete the frame; rank 0 untiles all shards into the row-major frame in one launch
            t = k & 3
            self.seq += 1
            sc.set_frame_target(None)
            sc.render(self.view, self.w, self.h, 0, self.flags, self.rank, self.world, timed=False)
            last = sc.frame_stream(-1)
            slot = next(q for q in range(3) if sc.frame_stream(q) == last)
            if self.rank != 0:
                if self.target_seq[t]:    # staging t must have been untiled on rank 0 before it is overwritten (four frames ago)
                    sc.wait_flag(self.local_flags + 4 * (32 + t), self.target_seq[t])
                sc.push(self.peer_ptrs[t] + self.rank * self.max_items * 4)
                sc.signal(self.remote_flags[0] + 4 * (self.rank * 4 + slot), self.seq)
            else:
                sc.push(self.peer_ptrs[t])
                for r in range(1, self.world):
                    sc.wait_flag(self.local_flags + 4 * (r * 4 + slot), self.seq)
                sc.untile_shards(self.peer_ptrs[t], self.w, self.h, self.world, self.peer_ptrs[t] + self.world * self.max_items * 4)
                if copy_out is not None:
                    copy_out(k)
                for r in range(1, self.world):
                    sc.signal(self.remote_flags[r] + 4 * (32 + t), self.seq)
            self.target_seq[t] = self.seq
        elif self.world > 1 and self.exchange in ("peer", "peer-nccl"):
            t = k & 3
            self.seq += 1
            if self.local_flags is not None and self.rank != 0 and self.target_seq[t]:
                # this target's previous frame must have been consumed on rank 0 before this rank's kernels overwrite it
                sc.wait_flag(self.local_flags + 4 * (32 + t), self.target_seq[t], before_next_frame=True)
            sc.set_frame_target(self.peer_ptrs[t])
            sc.render(self.view, self.w, self.h, 0, self.flags, self.rank, self.world, timed=False)
            last = sc.frame_stream(-1)
            slot = next(q for q in range(3) if sc.frame_stream(q) == last)
            if self.local_flags is None:                  # peer-nccl: the round-1 barrier, on the frame's own stream / communicator
                with self.torch.cuda.stream(self.torch_stream(sc.frame_stream(-1))):
                    self.dist.all_reduce(self.done[slot], group=self.groups[slot])
                if copy_out is not None and self.rank == 0:
                    copy_out(k)
            elif self.rank != 0:
                sc.signal(self.remote_flags[0] + 4 * (self.rank * 4 + slot), self.seq)       # into rank 0's memory, behind my kernels
            else:
                for r in range(1, self.world):
                    sc.wait_flag(self.local_flags + 4 * (r * 4 + slot), self.seq)             # every shard's pixels are there
                if copy_out is not None:
                    copy_out(k)
                for r in range(1, self.world):
                    sc.signal(self.remote_flags[r] + 4 * (32 + t), self.seq)                  # target t may be overwritten again
            self.target_seq[t] = self.seq
        elif self.world > 1 and self.exchange == "none":      # diagnostic: every rank keeps its shard (prices the exchange step)
            sc.set_frame_target(None)
            sc.render(self.view, self.w, self.h, 0, self.flags, self.rank, self.world, timed=False)
        elif self.world > 1:
            sc.set_frame_target(None)
            sc.render(self.view, self.w, self.h, 0, self.flags, self.rank, self.world, timed=False)
            _, _, d_rgba = sc.frame_device_ptrs()
            local = self.torch.as_tensor(self.cuda.DeviceArray(d_rgba, (self.max_items,), "<i4", sc), device="cuda")
            self.dist.gather(local, self.gathered, dst=0)
            if self.rank == 0:
                for s in range(self.world):
                    sc.untile_rgba(self.gathered[s].data_ptr(), self.w, self.h, s, self.world, self.frames[0].data_ptr())
                if copy_out is not None:
                    copy_out(k)
        else:
            sc.set_frame_target(None)
            sc.render(self.view, self.w, self.h, 0, self.flags, 0, 1, timed=False)
            _, _, d_rgba = sc.frame_device_ptrs()
            sc.untile_rgba(d_rgba, self.w, self.h, 0, 1, self.frames[k & 1].data_ptr())      # on the frame's own stream
            if copy_out is not None:
                copy_out(k)
        return k

    def last_frame_tensor(self, k):
        """rank 0: the row-major frame step k produced, as an int32 tensor"""
        if self.world > 1 and self.exchange == "push":
            return self.torch.as_tensor(self.cuda.DeviceArray(self.peer_frames[k & 3] + self.world * self.max_items * 4, (self.h * self.w,), "<i4", self.scene), device="cuda")
        if self.world > 1 and self.exchange in ("peer", "peer-nccl"):
            return self.torch.as_tensor(self.cuda.DeviceArray(self.peer_frames[k & 3], (self.h * self.w,), "<i4", self.scene), device="cuda")
        return self.frames[0 if self.world > 1 else (k & 1)]

    def sync_all(self):
        self.scene.sync()
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed_run(self, steps, flush_buf=None):
        """CUDA-event time of `steps` steps on this rank (ms).  One frame at a time: one event pair per step on the launching
        stream, the L2 flush between steps outside the pairs.  Two frames in flight: one pair around the whole run — the first
        event ahead of every frame (tray_cuda_scene_after), the second behind all of them (tray_cuda_scene_fence)."""
        torch = self.torch
        self.sync_all()
        if self.in_flight == 1:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for i in range(steps):
                if flush_buf is not None:
                    flush_buf.fill_(i & 0xff)                   # L2 flush between timed iterations (not in the timed span)
                ev[i][0].record(self.main)
                self.step()
                ev[i][1].record(self.main)
            self.sync_all()
            return sum(a.elapsed_time(b) for a, b in ev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.main)
        self.scene.after(self.main.cuda_stream)
        for _ in range(steps):
            self.step()
        self.scene.fence(self.main.cuda_stream)
        e1.record(self.main)
        self.sync_all()
        return e0.elapsed_time(e1)

    def close(self):
        self.scene.sync()
        self.torch.cuda.synchronize()
        self.scene.set_frame_target(None)
        self.ext.clear()
        if self.rank != 0:
            for p in self.peer_ptrs:
                self.cuda.ipc_close(p, self.local_rank)
        for p in self.remote_flags.values():
            self.cuda.ipc_close(p, self.local_rank)
        if self.world > 1:
            self.dist.barrier()
        for f in self.peer_frames:
            self.cuda.frame_free(f, self.local_rank)
        if self.local_flags is not None:
            self.cuda.frame_free(self.local_flags, self.local_rank)
        self.peer_frames, self.peer_ptrs, self.remote_flags, self.local_flags = [], [], {}, None


def max_over_ranks(torch, dist, world, x):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


_keep_alive = []


def strong_scaling_record(torch, dist, cuda, host, rank, world, local_rank, stream, steps, which="c4"):
    """BASELINE.json configs[3] (c4) inside every --gpus N line — and configs[4] (c5, `--tlas`) at N = 8: the scene at a FIXED
    3840x2160 frame, tiles dealt over the N ranks (strong scaling).  speedup_vs_n1 = this run's own one-GPU time (rank 0 renders
    the whole frame alone, the other ranks idle) / the N-GPU time — same box, same build, same protocol.  The BVH is built on each
    rank's GPU from the triangle soup (tray_cuda_scene_build[_tlas]: deterministic, so the replicas agree)."""
    global WL
    saved = WL
    WL = WORKLOADS[which]
    try:
        w, h = WL["w"], WL["h"]
        mesh = host.Mesh.generate(WL["scene"], WL["seed"], 1.0)
        scene = cuda.TrayCudaScene.build(mesh.tris(), tri_stride=TRI_STRIDE, device=local_rank,
                                         object_offsets=mesh.object_offsets() if WL["tlas"] else None)
        scene.set_stream(stream.cuda_stream)
        view = host.view_from_camera(mesh.camera, w, h, scene.info()["tlas_start"] if WL["tlas"] else 0)
        flags = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA
        scene.render(view, w, h, 0, flags | cuda.RENDER_COUNTERS, rank, world)
        cp, cb = scene.counters()
        rays = torch.tensor([cp["rays"] + cb["rays"]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(rays)
        rays = float(rays.item())
        out = {"workload": f"{WL['label']} ({mesh.n_tris} tris, BVH built on the device), fixed {w}x{h} frame, tiles dealt over {world} GPU(s), primary + 1spp bounce",
               "rays_per_step": rays}
        forced = os.environ.get("TRAY_BENCH_STRONG_EXCHANGE") or os.environ.get("TRAY_BENCH_EXCHANGE")
        exchanges = ["local"] if world == 1 else ([forced] if forced else ["push", "peer"])
        best_ms, n1_cache = None, {}
        for ex in exchanges:
            rig = Rig(torch, dist, cuda, scene, view, w, h, rank, world, local_rank, stream, ex)
            for in_flight in (3, 2, 1):
                rig.configure(False, in_flight)
                for _ in range(4):
                    rig.step()
                ms = max_over_ranks(torch, dist, world, rig.timed_run(steps)) / steps
                rec = {"ms_per_step": ms, "value": rays / ms / 1e3}
                if world > 1 and in_flight in n1_cache:
                    rec["n1_ms_per_step"], rec["speedup_vs_n1"] = n1_cache[in_flight], n1_cache[in_flight] / ms
                elif world > 1:
                    # the one-GPU time of the same frame in the same run: rank 0 alone, whole frame
                    n1 = 0.0
                    scene.sync()
                    scene.set_frame_target(None)
                    if rank == 0:
                        solo = Rig(torch, dist, cuda, scene, view, w, h, 0, 1, local_rank, stream, "local")
                        solo.configure(False, in_flight)
                        for _ in range(3):
                            solo.step()
                        torch.cuda.synchronize()
                        n1 = solo.timed_run(max(5, steps // 2)) / max(5, steps // 2)
                        scene.sync()
                    n1 = max_over_ranks(torch, dist, world, n1)
                    n1_cache[in_flight] = n1
                    rec["n1_ms_per_step"] = n1
                    rec["speedup_vs_n1"] = n1 / ms
                else:
                    rec["n1_ms_per_step"], rec["speedup_vs_n1"] = ms, 1.0
                out.setdefault("by_exchange", {}).setdefault(ex, {})["one_frame_at_a_time" if in_flight == 1 else f"{in_flight}_frames_in_flight"] = rec
                if in_flight > 1 and (best_ms is None or ms < best_ms):      # the record's own figures: the best mode
                    best_ms = ms
                    out.update(rec)
                    out["frames_in_flight"], out["exchange"] = in_flight, ex
            rig.close()
        out["one_frame_at_a_time"] = out["by_exchange"][out["exchange"]]["one_frame_at_a_time"]
        out["unit"] = UNIT
        out["note"] = ("ms_per_step = CUDA-event time of the steps / steps, max over ranks, exchange included (kernels store pixels into "
                       "rank 0's frame over NVLink, or push their compact shard with one DMA copy; completion flags); no L2 flush "
                       "(working set 0.3 / 1.1 GB > 126 MB L2)")
        torch.cuda.synchronize()
        _keep_alive.append(scene)        # closed by the caller after the process group is gone
        return out
    finally:
        WL = saved


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tray_racing_b200 import cuda, host

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs `python -m torch.distributed.run --nproc-per-node {args.gpus} bench.py ...`")
        raise SystemExit(f"WORLD_SIZE {world} != --gpus {args.gpus}")
    if not torch.cuda.is_available() or cuda.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device: tray_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ncpu = host_threads()
    mesh, packed = build_scene(nthreads=max(1, ncpu // world))
    w, h = frame_size(world)
    view = host.view_from_camera(mesh.camera, w, h, packed.tlas_start)
    scene = cuda.TrayCudaScene.from_packed(packed, device=local_rank)
    # one explicit (non-default) torch stream carries slot-0 frames, the collectives, the untile and the timing events
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    scene.set_stream(stream.cuda_stream)
    steps, warmup = args.steps, max(args.warmup, 3)

    # ---- which of the byte-identical ways to run the step: exchange (push: DMA copy of the compact shard + untile on rank 0 /
    # peer: the kernels store pixels into rank 0's frame) x two launches / one-launch frame kernel x one / two / three frames in
    # flight.  An untimed calibration decides, the way tray_cuda_start picks its frame path (--exchange, TRAY_BENCH_OVERLAP and
    # TRAY_BENCH_IN_FLIGHT force a choice).
    if world == 1:
        candidates = ["local"]
    elif args.exchange == "auto":
        candidates = [os.environ["TRAY_BENCH_EXCHANGE"]] if os.environ.get("TRAY_BENCH_EXCHANGE") else ["push", "peer"]
    else:
        candidates = [args.exchange]
    rigs = {}
    for ex in candidates:
        try:
            rigs[ex] = Rig(torch, dist, cuda, scene, view, w, h, rank, world, local_rank, stream, ex)
        except cuda.TrayCudaError as e:
            if args.exchange != "auto":
                raise
            print(f"[bench] rank {rank}: exchange {ex} unavailable ({e})", file=sys.stderr)
    ok = torch.tensor([float(len(rigs))], device="cuda")
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if float(ok.item()) < len(candidates):              # some rank could not map peer memory: everybody falls back to the NCCL gather
        for r_ in rigs.values():
            r_.close()
        rigs = {"nccl": Rig(torch, dist, cuda, scene, view, w, h, rank, world, local_rank, stream, "nccl")}
    f_overlap, f_inflight = os.environ.get("TRAY_BENCH_OVERLAP"), os.environ.get("TRAY_BENCH_IN_FLIGHT")
    calib = {}
    for ex, r_ in rigs.items():
        for ov in ((False, True) if f_overlap is None else (f_overlap != "0",)):
            for nf in ((1, 2, 3) if f_inflight is None else (int(f_inflight),)):
                r_.configure(ov, nf)
                for _ in range(3):
                    r_.step()
                calib[(ex, ov, r_.in_flight)] = max_over_ranks(torch, dist, world, r_.timed_run(10)) / 10
        scene.set_frame_target(None)
    (exchange, overlap, in_flight), _ = min(calib.items(), key=lambda kv: kv[1])
    rig = rigs.pop(exchange)
    for r_ in rigs.values():
        r_.close()
    flags2 = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA            # the two-launch path: per-kernel figures, counters

    # one counting frame (outside the timed region): rays and algorithmic bytes per step
    rig.configure(False, 1)
    scene.render(view, w, h, 0, flags2 | cuda.RENDER_COUNTERS, rank, world)
    cp, cb = scene.counters()
    scene.render(view, w, h, 0, flags2, rank, world)          # switch back to the non-counting kernels
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    # ---- bit-equality of the exchange paths, once, outside the timed region: peer frame == NCCL gather + untile ----
    exchange_verified = None
    if world > 1 and exchange in ("peer", "peer-nccl", "push"):
        chk = Rig(torch, dist, cuda, scene, view, w, h, rank, world, local_rank, stream, "nccl")
        chk.configure(overlap, 1); chk.step(); chk.sync_all()
        rig.configure(overlap, in_flight)
        ks = [rig.step() for _ in range(3)]             # three frames, so that both frame slots and three targets are checked
        rig.sync_all()
        if rank == 0:
            exchange_verified = all(bool(torch.equal(rig.last_frame_tensor(k), chk.last_frame_tensor(0))) for k in ks)
        scene.set_frame_target(None)

    # ---- headline: `steps` timed steps in the calibrated mode ----
    rig.configure(overlap, in_flight)
    for _ in range(warmup):
        flush_buf.fill_(1)
        rig.step()
    rig.sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_wall0 = time.time()
    try:
        total_ms = rig.timed_run(steps, flush_buf)
    finally:                                           # no nvidia-smi left running when the timed run fails
        t_wall1 = time.time()
        clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_frame(args.dump_outputs, rig.last_frame_tensor(rig.k - 1), w, h)
    total_ms = max_over_ranks(torch, dist, world, total_ms)
    rays_step = torch.tensor([cp["rays"] + cb["rays"], cp["rays"], cb["rays"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(rays_step, op=dist.ReduceOp.SUM)
    rays_all, rays_p, rays_b = (float(x) for x in rays_step.tolist())
    value = rays_all * steps / (total_ms * 1e-3) / 1e6

    # ---- beside it: one frame at a time with the L2 flushed between steps (round 1's protocol), and without the flush ----
    side = {}
    for name, nf, fl in (("one_frame_at_a_time_l2_flushed", 1, flush_buf), ("one_frame_at_a_time_warm_l2", 1, None)):
        rig.configure(overlap, nf)
        for _ in range(3):
            rig.step()
        n = max(5, min(steps, 50))
        ms = max_over_ranks(torch, dist, world, rig.timed_run(n, fl)) / n
        side[name] = {"ms_per_step": ms, "value": rays_all / ms / 1e3}

    scene.set_frame_target(None)                       # the per-rank measurements below use the compact local buffers
    rig.configure(False, 1)
    # ---- the traversal kernels alone (this rank): live CUDA-event duration of primary and bounce launches, L2 flushed ----
    kp, kb = [], []
    for _ in range(max(5, min(steps, 20))):
        flush_buf.fill_(3)
        a, b = scene.render(view, w, h, 0, flags2, rank, world, timed=True)
        kp.append(a); kb.append(b)
    kp_ms, kb_ms = sum(kp) / len(kp), sum(kb) / len(kb)
    kf_ms = None
    if overlap:                                        # the frame kernel (+ primary ray generation), CUDA events, L2 flushed
        kf = []
        for _ in range(max(5, min(steps, 20))):
            flush_buf.fill_(3)
            kf.append(scene.render(view, w, h, 0, flags2 | cuda.RENDER_OVERLAP, rank, world, timed=True)[0])
        kf_ms = sum(kf) / len(kf)
    bytes_p = 80 * cp["nodes"] + TRI_STRIDE * cp["tris"] + 4 * cp["instances"] + 8 * cp["rays"]
    bytes_b = 80 * cb["nodes"] + TRI_STRIDE * cb["tris"] + 4 * cb["instances"] + 8 * cb["rays"] + 8 * cp["rays"]
    hbm_peak, hbm_src = measured_peaks()
    l2_peak = cuda.bandwidth_probe(48 << 20, 50, local_rank)          # streaming read of an L2-resident 48 MiB buffer
    hbm_read = cuda.bandwidth_probe(2048 << 20, 8, local_rank)        # same kernel, buffer >> L2
    l1_gather = cuda.l1_gather_probe(32 << 10, 200, local_rank)       # every lane its own 16-byte record of an L1-resident table

    # ---- end to end through the public API with HOST buffers ----
    # Every step: tray_cuda_render on every rank (view + frame parameters go in by value, 160 B per rank), the exchange step,
    # and the readback of that frame's RGBA8 into pinned host memory on rank 0 through a small ring of buffers: the D2H of frame k
    # overlaps the kernels of the next frames; frame k is in host memory before frame k + 3 is issued, the last frames are
    # waited for inside the timed region.  N = 1: tray_cuda_frame_readback_begin / _wait.  N > 1
    # (peer exchange): rank 0 snapshots the complete frame out of its target on the frame's own stream, behind the flag waits that
    # complete it, hands the target back (consumed flags) and copies the snapshot to the host on a copy stream.
    rig.configure(overlap, in_flight)
    e2e_steps = max(3, min(steps, 50))
    owner = rank == 0
    RING = 3                                         # host / staging buffers: frame i is in host memory before frame i + RING is issued
    host_frames = [torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True) for _ in range(RING)] if owner else None
    stage = [torch.empty(h * w, dtype=torch.int32, device="cuda") for _ in range(RING)] if (owner and world > 1) else None
    copy_stream = torch.cuda.Stream() if (owner and world > 1) else None
    copy_ev = [None] * RING
    ring_of = {}

    def copy_out(k):
        """rank 0, N > 1: called by Rig.step where frame k is complete on the frame's own stream — snapshot it there (device to
        device, so the target can be handed back at once), then D2H on a copy stream of its own"""
        b = ring_of[k]
        st = rig.torch_stream(scene.frame_stream(-1))
        with torch.cuda.stream(st):
            stage[b].copy_(rig.last_frame_tensor(k))
            snap = torch.cuda.Event(); snap.record(st)
        copy_stream.wait_event(snap)
        with torch.cuda.stream(copy_stream):
            host_frames[b].view(-1).view(torch.int32).copy_(stage[b], non_blocking=True)
            copy_ev[b] = torch.cuda.Event(); copy_ev[b].record(copy_stream)

    def e2e_step(i):
        b = i % RING
        if world == 1:
            scene.render(view, w, h, 0, rig.flags, 0, 1, timed=False)
            scene.readback_begin(host_frames[b].numpy(), b)       # untile on the frame's stream, D2H on the copy stream
            if i > 1:
                scene.readback_wait((i - 2) % RING)               # frame i - 2 is in host memory before frame i + 1 is issued
            return
        if owner and copy_ev[b] is not None:
            copy_ev[b].synchronize()                    # frame i - RING has landed: host buffer b and staging b are free again
        ring_of[rig.k] = b
        rig.step(copy_out if owner else None)

    def e2e_drain():
        if world == 1:
            for b in range(RING):
                scene.readback_wait(b)
        elif owner:
            for e in copy_ev:
                if e is not None:
                    e.synchronize()

    rig.k = 0
    for i in range(RING):
        e2e_step(i)                                   # untimed: every staging buffer allocated, copy paths warm
    e2e_drain()
    rig.sync_all()
    rig.k = 0
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    e2e_drain()
    scene.sync()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(torch, dist, world, time.perf_counter() - t0)
    e2e_val = rays_all * e2e_steps / e2e_s / 1e6
    # the same, fully synchronous (render, then download, then the next frame): what a caller without the readback pair gets
    scene.set_frame_target(None)
    rig.configure(overlap, 1)
    into = {"rgba": host_frames[0].numpy() if owner else np.zeros((h, w, 4), dtype=np.uint8)}
    scene.render(view, w, h, 0, rig.flags, rank, world, timed=False); scene.download(rgba=True, into=into)     # allocates its staging
    rig.sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        scene.render(view, w, h, 0, rig.flags, rank, world, timed=False)
        scene.download(rgba=True, into=into)
    torch.cuda.synchronize()
    e2e_sync_val = rays_all * e2e_steps / max_over_ranks(torch, dist, world, time.perf_counter() - t0) / 1e6

    # ---- strong scaling on BASELINE.json configs[3] (every N), outside every timed region above ----
    strong = strong_c5 = None
    if args.workload == "c3" and os.environ.get("TRAY_BENCH_STRONG", "1") != "0":
        strong = strong_scaling_record(torch, dist, cuda, host, rank, world, local_rank, stream, max(10, min(steps, 40)))
        if world == 8 or os.environ.get("TRAY_BENCH_STRONG_C5") == "1":
            strong_c5 = strong_scaling_record(torch, dist, cuda, host, rank, world, local_rank, stream, max(10, min(steps, 30)), which="c5")

    # ---- beside the headline (N = 1 only, outside every timed region above): the rows SURVEY.md §8 marks "next" ----
    extras = None
    if rank == 0 and world == 1 and args.workload == "c3":
        extras = {}
        rig.configure(False, 1)
        # f4: AO rays as an any-hit query (rt_cpu.rs:78-79) — same rays, each stopped at its first hit
        ka = [scene.render(view, w, h, 0, flags2 | cuda.RENDER_ANYHIT_AO, rank, world, timed=True) for _ in range(6)][1:]
        kb_any = min(b for _, b in ka)
        extras["anyhit_ao"] = {"bounce_kernel_ms": kb_any, "bounce_kernel_mrays_s": cb["rays"] / kb_any / 1e3,
                               "closest_hit_bounce_kernel_ms": kb_ms, "note": "TRAY_RENDER_ANYHIT_AO: visibility only, not the reference image"}
        # f3: the same triangles built into a CWBVH on the device (PLOC) instead of by the host producer
        tris = mesh.tris()
        cuda.TrayCudaScene.build(tris, tri_stride=TRI_STRIDE, device=local_rank).close()      # warm-up: modules, pinned upload slots, allocator
        g, wall = None, None
        for _ in range(3):                                                                    # best of 3 (host wall clock around the call)
            if g is not None:
                g.close()
            t0 = time.perf_counter()
            g2 = cuda.TrayCudaScene.build(tris, tri_stride=TRI_STRIDE, device=local_rank)
            w2 = (time.perf_counter() - t0) * 1e3
            if wall is None or w2 < wall:
                wall, stats_best = w2, dict(g2.build_stats)
            g = g2
        kg = [g.render(view, w, h, 0, flags2) for _ in range(6)][1:]
        extras["device_builder"] = {"wall_ms": wall, **stats_best, "protocol": "one untimed warm-up build, then the best of 3",
                                    "host_producer_ms": packed.build_seconds * 1e3,
                                    "primary_kernel_ms_on_device_built_bvh": min(a for a, _ in kg),
                                    "bounce_kernel_ms_on_device_built_bvh": min(b for _, b in kg),
                                    "note": "PLOC radius 14 on the GPU vs binned SAH on the host cores; same collapse + encoder"}
        g.close()
        # b: the one-process entry point on this box's GPU(s): tray_group (peer access + events, no torch / NCCL) gives the same frame
        grp = cuda.TrayCudaGroup.from_packed(packed, devices=[local_rank])
        grp.set_frames_in_flight(2)
        for _ in range(4):
            grp.render(view, w, h, 0, flags2)
        grp.sync()
        t0 = time.perf_counter()
        for _ in range(40):
            grp.render(view, w, h, 0, flags2)
        grp.sync()
        gms = (time.perf_counter() - t0) * 1e3 / 40
        same = bool((grp.frame().reshape(-1).view(np.int32) == rig.frames[0].cpu().numpy()).all()) if rig.frames is not None else None
        extras["single_process_group"] = {"devices": 1, "ms_per_frame": gms, "mrays_s": rays_all / gms / 1e3, "frames_in_flight": 2,
                                          "frame_equals_bench_frame": same, "note": "tray_cuda_group_render, two-launch path, host wall clock over 40 frames"}
        grp.close()

    if rank == 0:
        cpu_base, _ = cpu_oracle_run(packed, mesh, w, h, seconds_budget=10.0, frames_min=3) if world == 1 else (None, None)
        clk_hz = (clocks or {}).get("sm_mhz") or 1965.0
        sm_count = scene.info()["sm_count"]
        issue_peak = sm_count * 4 * clk_hz * 1e6                    # warp instructions per second the chip can issue
        winst_p = ncu_figure("primary_kernel_warp_inst_per_launch") if (args.workload == "c3" and world == 1) else None
        tinst_p = ncu_figure("primary_kernel_thread_inst_per_launch") if (args.workload == "c3" and world == 1) else None
        roof = {
            # what the north_star names: the node + triangle bytes the PRIMARY rays fetch x rays/s against the measured L2 bandwidth
            "bound": "l2", "kernel": "trace_kernel (primary rays; two-launch path, CUDA events, L2 flushed before each launch)",
            "achieved": bytes_p / kp_ms / 1e6, "peak": l2_peak, "unit": "GB/s", "frac": bytes_p / kp_ms / 1e6 / l2_peak,
            "peak_source": "measured in this run: streaming 16-byte reads of an L2-resident 48 MiB buffer by a chip-filling grid "
                           "(tray_cuda_bandwidth_probe); MEASURED_PEAKS.json holds no L2 figure",
            "traffic": ncu_figure("primary_kernel_dram_bytes_per_launch") if args.workload == "c3" else None,
            "algorithmic_bytes_per_launch": bytes_p, "bytes_per_ray": bytes_p / max(1, cp["rays"]), "ms_per_launch": kp_ms,
            "nodes_per_ray": cp["nodes"] / max(1, cp["rays"]), "tris_per_ray": cp["tris"] / max(1, cp["rays"]),
            "what_binds": "SM issue slots (ALU pipe) first, the L1's gather rate second; not DRAM (~4 % of the algorithmic bytes) and not L2 (~12 % of its throughput; ncu, profiles/)",
            "issue": {"peak_warp_inst_per_s": issue_peak, "sm_mhz": clk_hz,
                      "warp_inst_per_launch": winst_p, "thread_inst_per_launch": tinst_p,
                      "warp_inst_per_ray": (winst_p / cp["rays"]) if winst_p else None,
                      "lanes_per_inst": (tinst_p / winst_p) if (winst_p and tinst_p) else None,
                      "frac_of_issue_peak": (winst_p / (kp_ms * 1e-3) / issue_peak) if winst_p else None,
                      "note": "instruction counts per launch from the committed ncu capture of this kernel (profiles/roofline_traffic.json), duration live"},
            "l1_gather": {"peak": l1_gather, "achieved": bytes_p / kp_ms / 1e6, "frac": bytes_p / kp_ms / 1e6 / l1_gather, "unit": "GB/s",
                          "bytes_per_clk_per_sm": l1_gather * 1e9 / (sm_count * clk_hz * 1e6),
                          "peak_source": "measured in this run (tray_cuda_l1_gather_probe): every lane of every warp reads its own 16-byte record "
                                         "from a different 128-byte line of an L1-resident 32 KiB table — how a traversal warp reads nodes and triangles",
                          "note": "the memory pipe this kernel loads most: every node visit is 5 and every triangle test 3 such accesses per lane "
                                  "(ncu l1tex__throughput 42 % on this launch; 75 % with 128-byte nodes, profiles/experiments/r2_tnode_*)"},
            "hbm": {"peak": hbm_peak, "peak_source": hbm_src, "frac": bytes_p / kp_ms / 1e6 / hbm_peak,
                    "hbm_read_gbs_measured_here": hbm_read, "note": "side figure: the kernel is not HBM-bound (see traffic)"},
            "bounce_kernel": {"achieved": bytes_b / kb_ms / 1e6 if cb["rays"] else None, "frac": (bytes_b / kb_ms / 1e6 / l2_peak) if cb["rays"] else None,
                              "ms_per_launch": kb_ms, "algorithmic_bytes_per_launch": bytes_b},
        }
        if kf_ms:
            roof["frame_kernel"] = {"achieved": (bytes_p + bytes_b) / kf_ms / 1e6, "frac": (bytes_p + bytes_b) / kf_ms / 1e6 / l2_peak,
                                    "ms_per_launch": kf_ms, "algorithmic_bytes_per_launch": bytes_p + bytes_b,
                                    "note": "trace_kernel<FRAME>: both ray kinds in one launch; span includes raygen_primary"}
        per_frame = (2 if overlap else 4) + (0 if exchange in ("peer", "peer-nccl") else 1)        # "push": + one untile launch on rank 0
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": WL["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(w, h, world), "n_tris": packed.n_tris, "n_nodes": packed.n_nodes,
                       "working_set_mb": round(packed.working_set_bytes() / 1e6, 1), "tri_stride": TRI_STRIDE,
                       "rays_per_step": {"primary": rays_p, "bounce": rays_b},
                       "frame_path": ("one launch per frame (TRAY_RENDER_OVERLAP: raygen_primary + trace_kernel<FRAME>)" if overlap
                                      else "two launches per frame (raygen_primary, trace, raygen_bounce, trace)"),
                       "frames_in_flight": in_flight,
                       "calibration_ms_per_step": {f"{ex}_{'one' if ov else 'two'}_launch_x{nf}_in_flight": v for (ex, ov, nf), v in calib.items()},
                       "l2": ("flushed between timed steps (256 MiB device write)" if in_flight == 1 else
                              f"not flushed: two frames in flight, consecutive frames of a {round(packed.working_set_bytes() / 1e6)} MB working set "
                              "(> 126 MB L2 for c3/c4/c5); the one-frame-at-a-time figures beside it are with and without the flush"),
                       "parallelism": f"tile-sharded x{world}, BVH replicated",
                       "exchange": ("push: every rank's compact RGBA8 shard goes to rank 0's IPC-mapped staging with one DMA copy over NVLink, completion by 32-bit "
                                    "flags the stream front-end writes / awaits (cuStreamWriteValue32 / cuStreamWaitValue32), one untile launch on rank 0; "
                                    "no collective kernel" if exchange == "push" else
                                    "peer: kernels store pixels into rank 0's IPC-mapped row-major frame over NVLink; completion by 32-bit flags the stream "
                                    "front-end writes / awaits (cuStreamWriteValue32 / cuStreamWaitValue32), no collective kernel" if exchange == "peer" else
                                    "peer-nccl: same stores, a 4-byte all-reduce on the frame's own stream as barrier" if exchange == "peer-nccl" else
                                    "NCCL gather of RGBA8 shards to rank 0 + untile per shard") if world > 1
                       else "untile only (single GPU)",
                       "exchange_verified_bit_equal_to_nccl_path": exchange_verified},
            **side,
            "mrays_s": {"primary_kernel": cp["rays"] / kp_ms / 1e3, "bounce_kernel": (cb["rays"] / kb_ms / 1e3) if cb["rays"] else None,
                        "note": "rank-0 shard, the two-launch path's kernels alone, CUDA events, L2 flushed"},
            "roofline": roof,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": 160 * world, "d2h_bytes_per_step": w * h * 4,
                    "l2": "not flushed (back-to-back frames; the flushed and unflushed one-frame-at-a-time device figures are beside `value`)",
                    "synchronous_note": "per rank: render, then tray_cuda_frame_download of a full-size frame (other shards zero), no exchange, no overlap",
                    "synchronous_value": e2e_sync_val,
                    "note": "per step and rank: tray_cuda_render + exchange + the complete RGBA8 frame to pinned host memory on rank 0, double-buffered "
                            "(the D2H of frame k overlaps the kernels of frame k+1; every frame is waited for inside the timed region), wall clock"},
            "gpu_launches": steps * world * per_frame,
            "clocks": clocks,
        }
        if strong is not None:
            line["strong"] = strong
        if strong_c5 is not None:
            line["strong_c5"] = strong_c5
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        if extras:
            line["next_rows"] = extras
        emit(line)
    rig.close()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()                   # before the scenes go: NCCL may hold events of the scenes' streams
    scene.close()
    for sc in _keep_alive:
        sc.close()
    return 0


def run_single_process(args):
    """--single-process: the same frames from ONE process driving all N GPUs through the C ABI's tray_group (peer access + events;
    no torchrun, no NCCL, no torch on the data path) — the shape of the reference's slot, one call from one host thread
    (rt_gpu_software.rs:24-32).  The frame is checked byte for byte against the single-GPU frame of the same process."""
    import torch
    from tray_racing_b200 import cuda, host
    n = args.gpus
    if cuda.device_count() < n:
        raise SystemExit(f"--single-process --gpus {n}: only {cuda.device_count()} CUDA device(s) visible")
    mesh, packed = build_scene(nthreads=host_threads())
    w, h = frame_size(n)
    view = host.view_from_camera(mesh.camera, w, h, packed.tlas_start)
    flags = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA
    one = cuda.TrayCudaScene.from_packed(packed, device=0)
    one.render(view, w, h, 0, flags | cuda.RENDER_COUNTERS)
    cp, cb = one.counters()
    rays = cp["rays"] + cb["rays"]
    one.render(view, w, h, 0, flags)
    want = one.download(rgba=True)["rgba"].copy()
    one.close()
    g = cuda.TrayCudaGroup.from_packed(packed, devices=list(range(n)))
    steps, warmup = args.steps, max(args.warmup, 3)
    res = {}
    for nf in (1, 2, 3):
        g.set_frames_in_flight(nf)
        for _ in range(warmup):
            g.render(view, w, h, 0, flags)
        same = bool((g.frame() == want).all())
        g.sync()
        t0 = time.perf_counter()
        for _ in range(steps):
            g.render(view, w, h, 0, flags)
        g.sync()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        res[nf] = {"ms_per_step": ms, "value": rays / ms / 1e3, "frame_equals_single_gpu_frame": same}
    if args.dump_outputs:                              # the frame of the last timed step (three frames in flight)
        dump_frame(args.dump_outputs, g.frame(), w, h)
    nf = min(res, key=lambda q: res[q]["ms_per_step"])
    g.set_frames_in_flight(nf)
    per_frame_ms = [g.render(view, w, h, 0, flags, timed=True) for _ in range(12)][2:]
    host_frames = [torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)]
    e2e_steps = max(3, min(steps, 50))

    def e2e(i):
        g.render(view, w, h, 0, flags)
        g.readback_begin(host_frames[i & 1], i & 1)
        if i > 0:
            g.readback_wait((i - 1) & 1)
    e2e(0); e2e(1); g.readback_wait(0); g.readback_wait(1); g.sync()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e(i)
    g.readback_wait((e2e_steps - 1) & 1)
    g.sync()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_same = bool((host_frames[(e2e_steps - 1) & 1] == want).all())
    g.close()
    line = {"metric": METRIC, "value": res[nf]["value"], "unit": UNIT, "n_gpus": n, "steps": steps, "warmup": warmup,
            "ms_per_step": res[nf]["ms_per_step"], "higher_is_better": True, "scaling": WL["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl_note": "--single-process: one process, tray_cuda_group_* (C ABI), no torchrun / NCCL",
            "config": {"workload": workload_name(w, h, n), "n_tris": packed.n_tris, "n_nodes": packed.n_nodes, "frames_in_flight": nf,
                       "frame_path": "two launches per frame", "parallelism": f"one process, {n} device(s), tiles dealt round-robin, BVH replicated",
                       "exchange": ("one peer DMA copy of every device's compact shard into devices[0]'s staging + one untile launch there"
                                    if os.environ.get("TRAY_CUDA_GROUP_EXCHANGE", "1") != "0" else
                                    "kernels store pixels into devices[0]'s frame over peer access") + "; completion by events",
                       "timing": "host clock around the asynchronous frames, tray_cuda_group_sync on both sides (CUDA events do not span devices); "
                                 "per_frame_ms_cuda_events = tray_cuda_group_render_timed, one frame at a time"},
            "by_frames_in_flight": res, "per_frame_ms_cuda_events": {"min": min(per_frame_ms), "mean": sum(per_frame_ms) / len(per_frame_ms)},
            "e2e": {"value": rays / e2e_ms / 1e3, "unit": UNIT, "h2d_bytes_per_step": 160 * n, "d2h_bytes_per_step": w * h * 4,
                    "frame_in_host_memory_equals_single_gpu_frame": e2e_same,
                    "note": "tray_cuda_group_render + tray_cuda_group_readback_begin / _wait into pinned host memory, double-buffered, wall clock"},
            "gpu_launches": steps * n * 4}
    emit(line)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS),
                    help="c3 (default, the metric's config; weak scaling) | c1 | c2 (1080p) | c4 | c5 (fixed 3840x2160 frame sharded over the GPUs)")
    ap.add_argument("--single-process", action="store_true",
                    help="one process drives all --gpus N devices through tray_cuda_group_* (no torchrun)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "push", "peer", "peer-nccl", "nccl"],
                    help="how shards reach rank 0's frame: peer-mapped frame written by the kernels, or NCCL gather + untile")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame of the last one to DIR/frame_rgba.npy (float32; a seeded "
                         "sample of pixels when the frame exceeds 64 MB), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global WL
    WL = WORKLOADS[args.workload]
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if args.single_process:
        return run_single_process(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
