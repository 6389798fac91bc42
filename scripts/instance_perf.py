"""Instanced scenes on one GPU (tray_cuda_scene_set_instances).

    python scripts/instance_perf.py [out.jsonl]

One JSON line per measurement; the first names the GPU and its power limit.
  "c5_identity"   C5 built on the device, and the same tree with 4096 identity instances (instance k = object k): the frame
                  (render_frame_ms, two-launch path, median of 10 after 3 warm-up frames) of each, alternating five times in
                  the same run.  The difference is the cost of the transform kernels.
  "c5_rigid"      every C5 object translated by up to 5 % of the scene's extent (host.rigid's shifts): set_instances with the
                  shifts as transforms against refit_rebuild_tlas_device on the moved triangles (CUDA-event ms, median of 20
                  after 3 warm-up calls), the frame after each, and nodes / instances / triangles per primary and bounce ray
                  of one counted frame of each.
  "c1_grid"       C1 as ONE BLAS placed on a g x g x g grid (g = 16: 4096 instances, g = 8: 512): device_bytes, set_instances
                  ms, and the batch rate (Mrays/s, tray_cuda_trace_device, 2^22 random rays through the grid, median of 5 after
                  2 warm-up launches); for g = 8 also a flat device build of the 512 copies' triangles, which g = 16 (233 M
                  triangles) is not given."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench import WORKLOADS  # noqa: E402
from tray_racing_b200 import cuda, host  # noqa: E402


def frame_ms(sc, view, w, h):
    for _ in range(3):
        sc.render_frame_ms(view, w, h, 0)
    return float(np.median([sc.render_frame_ms(view, w, h, 0) for _ in range(10)]))


def per_ray(sc, view, w, h):
    sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_COUNTERS, timed=False)
    sc.sync()
    return {which: {k: c[k] / max(c["rays"], 1) for k in ("nodes", "instances", "tris")} for which, c in zip(("primary", "bounce"), sc.counters())}


def median_ms(call, warm=3, reps=20):
    for _ in range(warm):
        call()
    return float(np.median([call() for _ in range(reps)]))


def translations(shift):
    xf = np.zeros((shift.shape[0], 3, 4), np.float32)
    xf[:, :, :3] = np.eye(3, dtype=np.float32)
    xf[:, :, 3] = shift
    return xf


def grid_rays(lo, hi, n, seed):
    """n rays from random points of the box [lo, hi] in random directions"""
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, dtype=host.RAY_DTYPE)
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays["o"] = rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)
    rays["d"] = d.astype(np.float32)
    rays["tmax"] = np.float32(3.402823466e+38)
    return rays


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None
    if cuda.device_count() < 1:
        raise SystemExit("instance_perf needs a CUDA device")

    def emit(d):
        print(json.dumps(d), flush=True)
        if out:
            out.write(json.dumps(d) + "\n"); out.flush()

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    emit({"gpu": gpu})

    # ---- C5: identity instances, then rigid motion ----
    wl = WORKLOADS["c5"]
    m = host.Mesh.generate(wl["scene"], wl["seed"], 1.0)
    tris = np.ascontiguousarray(m.tris(), np.float32).reshape(-1, 3, 3)
    offs = m.object_offsets()
    w, h = wl["w"], wl["h"]
    view = host.view_from_camera(m.camera, w, h)
    plain = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    inst = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    n_obj = offs.size - 1
    roots = np.arange(n_obj, dtype=np.uint32)                      # object k's BLAS root is node k
    inst.set_instances(roots, translations(np.zeros((n_obj, 3), np.float32)))
    runs = [(frame_ms(plain, view, w, h), frame_ms(inst, view, w, h)) for _ in range(5)]
    emit(dict(measure="c5_identity", n_tris=int(tris.shape[0]), n_instances=n_obj, frame=f"{w}x{h}",
              frame_ms_plain=[r[0] for r in runs], frame_ms_instanced=[r[1] for r in runs],
              per_ray_plain=per_ray(plain, view, w, h), per_ray_instanced=per_ray(inst, view, w, h)))

    moved = host.rigid(tris, offs, 2)
    ext = float((tris.reshape(-1, 3).max(axis=0) - tris.reshape(-1, 3).min(axis=0)).max())
    shift = np.random.default_rng(2).uniform(-0.05 * ext, 0.05 * ext, (n_obj, 3)).astype(np.float32)   # host.rigid's shifts
    assert np.array_equal(moved[offs[1]:offs[2]], (tris[offs[1]:offs[2]] + shift[1]).astype(np.float32))
    d = torch.from_numpy(np.ascontiguousarray(moved).reshape(-1, 9)).cuda()
    ms_rebuild = median_ms(lambda: plain.refit_rebuild_tlas_device(d.data_ptr(), d.shape[0], timed=True))
    xf = translations(shift)
    t = {}

    def set_once():
        inst.set_instances(roots, xf, timings=t)
        return t["ms_set_instances"]
    ms_set = median_ms(set_once)
    runs = [(frame_ms(plain, view, w, h), frame_ms(inst, view, w, h)) for _ in range(3)]
    emit(dict(measure="c5_rigid", ms_refit_rebuild_tlas_device=ms_rebuild, ms_set_instances=ms_set,
              frame_ms_refit_rebuild_tlas=[r[0] for r in runs], frame_ms_set_instances=[r[1] for r in runs],
              per_ray_refit_rebuild_tlas=per_ray(plain, view, w, h), per_ray_set_instances=per_ray(inst, view, w, h),
              device_bytes_plain=plain.info()["device_bytes"], device_bytes_instanced=inst.info()["device_bytes"]))
    plain.close(); inst.close()
    del d
    torch.cuda.empty_cache()

    # ---- C1 as one BLAS on a grid ----
    wl = WORKLOADS["c1"]
    m = host.Mesh.generate(wl["scene"], wl["seed"], 1.0)
    tris = np.ascontiguousarray(m.tris(), np.float32).reshape(-1, 3, 3)
    lo, hi = tris.reshape(-1, 3).min(axis=0), tris.reshape(-1, 3).max(axis=0)
    step = (hi - lo) * np.float32(1.1)
    one = np.array([0, tris.shape[0]], np.uint64)
    n_rays = 1 << 22
    for g in (8, 16):
        cells = np.stack(np.meshgrid(*[np.arange(g)] * 3, indexing="ij"), axis=-1).reshape(-1, 3).astype(np.float32)
        xf = translations(cells * step)
        sc = cuda.TrayCudaScene.build(tris, object_offsets=one)
        t = {}
        for _ in range(3):
            sc.set_instances(np.zeros(cells.shape[0], np.uint32), xf, timings=t)
        rays = grid_rays(lo, lo + step * g, n_rays, seed=g)
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_hits = torch.zeros(n_rays * 8, dtype=torch.uint8, device="cuda")

        def rate(s):
            ms = median_ms(lambda: s.traverse_device(d_rays.data_ptr(), n_rays, d_hits.data_ptr(), timed=True), warm=2, reps=5)
            return n_rays / ms / 1e3
        line = dict(measure="c1_grid", grid=g, n_instances=int(cells.shape[0]), n_tris_blas=int(tris.shape[0]),
                    device_bytes_instanced=sc.info()["device_bytes"], ms_set_instances=t["ms_set_instances"], mrays_s_instanced=rate(sc))
        hit = d_hits.cpu().numpy().view(host.HIT_DTYPE)["prim"] != 0xFFFFFFFF
        line["hit_fraction"] = float(hit.mean())
        sc.close()
        if g == 8:
            flat = (tris[None] + (cells * step)[:, None, None, :]).reshape(-1, 3, 3)
            f = cuda.TrayCudaScene.build(flat)
            line.update(n_tris_flat=int(flat.shape[0]), device_bytes_flat=f.info()["device_bytes"], mrays_s_flat=rate(f),
                        ms_build_flat=f.build_stats["ms_total"])
            f.close()
            del flat
        emit(line)
        del d_rays, d_hits
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
