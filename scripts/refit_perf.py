"""Refit cost on one GPU, per BASELINE config: tray_cuda_scene_refit_device against a device build of the same triangles, and
the frame time (two-launch path) before and after a motion, next to a scene rebuilt on the moved triangles.

    python scripts/refit_perf.py [c1,c2,...] [out.jsonl]

For each config and each tree producer (the host's binned SAH, the device's PLOC) one JSON line:
  ms_refit_median   CUDA-event time of refit_device over the scene's own triangles (median of 20 after 3 warm-up calls)
  ms_build          tray_cuda_scene_build(_tlas)'s own ms_total for the same triangles (median of 3)
  frame_ms          render_frame_ms at the config's size, median of 10 after 3 warm-up frames: before any motion, after each
                    motion refit, and on a scene built on the device from the moved triangles
Motions: "jitter", every vertex moved by up to 1 % of the mean triangle size; "rigid" (two-level configs), every object
translated by up to 5 % of the scene's extent.  Two-level configs also get, per motion k:
  ms_refit_rebuild_tlas[k]   CUDA-event time of tray_cuda_scene_refit_rebuild_tlas_device on the moved triangles (every BLAS
                             refit, the TLAS rebuilt), median of 20 after 3 warm-up calls; measured after the refit-only frames
  frame_ms.after_k_refit_rebuild_tlas   the frame on that tree
  per_ray[k]                 nodes, instances and triangles per primary and per bounce ray, from one TRAY_RENDER_COUNTERS frame
                             of each tree: "refit", "refit_rebuild_tlas", "rebuild" (counts: they do not depend on the card)
The first line names the GPU and its power limit."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import WORKLOADS  # noqa: E402
from tray_racing_b200 import cuda, host  # noqa: E402


def frame_ms(sc, view, w, h):
    for _ in range(3):
        sc.render_frame_ms(view, w, h, 0)
    return float(np.median([sc.render_frame_ms(view, w, h, 0) for _ in range(10)]))


def per_ray(sc, view, w, h):
    """nodes, instances and triangles per primary and per bounce ray of one counted frame"""
    sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_COUNTERS, timed=False)
    sc.sync()
    return {which: {k: c[k] / max(c["rays"], 1) for k in ("nodes", "instances", "tris")} for which, c in zip(("primary", "bounce"), sc.counters())}


def rebuild_tlas_ms(sc, d):
    for _ in range(3):
        sc.refit_rebuild_tlas_device(d.data_ptr(), d.shape[0])
    return [sc.refit_rebuild_tlas_device(d.data_ptr(), d.shape[0], timed=True) for _ in range(20)]


def refit_ms(sc, d):
    for _ in range(3):
        sc.refit_device(d.data_ptr(), d.shape[0])
    return [sc.refit_device(d.data_ptr(), d.shape[0], timed=True) for _ in range(20)]


def main():
    names = sys.argv[1].split(",") if len(sys.argv) > 1 else ["c1", "c2", "c3", "c4", "c5"]
    out = open(sys.argv[2], "w") if len(sys.argv) > 2 else None
    if cuda.device_count() < 1:
        raise SystemExit("refit_perf needs a CUDA device")

    def emit(d):
        print(json.dumps(d), flush=True)
        if out:
            out.write(json.dumps(d) + "\n"); out.flush()

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    emit({"gpu": gpu})
    for name in names:
        wl = WORKLOADS[name]
        m = host.Mesh.generate(wl["scene"], wl["seed"], 1.0)
        tris = np.ascontiguousarray(m.tris(), np.float32).reshape(-1, 3, 3)
        offs = m.object_offsets() if wl["tlas"] else None
        w, h = wl["w"], wl["h"]
        view = host.view_from_camera(m.camera, w, h)
        motions = {"jitter": host.jitter(tris, 1)}
        if offs is not None:
            motions["rigid"] = host.rigid(tris, offs, 2)
        builds = []
        for _ in range(3):
            b = cuda.TrayCudaScene.build(tris, object_offsets=offs)
            builds.append(b.build_stats["ms_total"])
            b.close()
        rebuilt, rebuilt_counts = {}, {}
        for k, moved in motions.items():
            sc = cuda.TrayCudaScene.build(moved, object_offsets=offs)
            rebuilt[k] = frame_ms(sc, view, w, h)
            if offs is not None:
                rebuilt_counts[k] = per_ray(sc, view, w, h)
            sc.close()
        for producer in ("host", "device"):
            if producer == "host":
                p = host.PackedScene(m, use_tlas=wl["tlas"])
                sc = cuda.TrayCudaScene.from_packed(p)
                order = p.prim_to_mesh_tri
            else:
                sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
                order = None
            slots = (lambda t: t[order]) if order is not None else (lambda t: t)
            line = dict(config=name, producer=producer, n_tris=int(tris.shape[0]), n_nodes=sc.info()["n_nodes"], frame=f"{w}x{h}",
                        frame_ms={"before": frame_ms(sc, view, w, h)})
            d = torch.from_numpy(np.ascontiguousarray(slots(tris)).reshape(-1, 9)).cuda()
            ms = refit_ms(sc, d)
            line.update(ms_refit_median=float(np.median(ms)), ms_refit_min=float(np.min(ms)), ms_build=float(np.median(builds)))
            for k, moved in motions.items():
                dm = torch.from_numpy(np.ascontiguousarray(slots(moved)).reshape(-1, 9)).cuda()
                sc.refit_device(dm.data_ptr(), tris.shape[0])
                line["frame_ms"][f"after_{k}_refit"] = frame_ms(sc, view, w, h)
                line["frame_ms"][f"after_{k}_rebuild"] = rebuilt[k]
                if offs is not None:
                    line.setdefault("per_ray", {})[k] = {"refit": per_ray(sc, view, w, h), "rebuild": rebuilt_counts[k]}
                sc.refit_device(d.data_ptr(), tris.shape[0])
            if offs is not None:
                # last: a TLAS rebuild replaces the producer's TLAS for good
                line["ms_refit_rebuild_tlas"] = {}
                for k, moved in motions.items():
                    dm = torch.from_numpy(np.ascontiguousarray(slots(moved)).reshape(-1, 9)).cuda()
                    line["ms_refit_rebuild_tlas"][k] = float(np.median(rebuild_tlas_ms(sc, dm)))
                    line["frame_ms"][f"after_{k}_refit_rebuild_tlas"] = frame_ms(sc, view, w, h)
                    line["per_ray"][k]["refit_rebuild_tlas"] = per_ray(sc, view, w, h)
                    del dm
            emit(line)
            sc.close()
            del d
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
