"""Cost of the hit-attribute pass on one GPU (tray_cuda_hit_attributes_device, tray_cuda_frame_download_attributes).

    python scripts/hit_attr_perf.py [out.jsonl]

One JSON line per measurement; the first names the GPU and its power limit.
  "batch"   2^22 bounce rays of one frame of the scene (KEEP_RAYS, the rays of hit pixels, repeated up to 2^22), traced with
            trace_device (trace_instance_device on an instanced scene), then hit_attributes_device over those rays and hits:
            CUDA-event ms of each, median of 20 after 3 warm-up launches.  L2 is not flushed between launches; the working set of
            the attribute pass (rays 128 MiB, hits 32 MiB, out 80 MiB) is larger than the 126 MB L2 anyway.
  "frame"   render_frame_ms of the frame (default flags: bounce + RGBA; two-launch or overlap as the scene renders by default),
            and the wall clock of download_attributes(primary, bounce) after it (attribute kernel, untile, copy of 2 x 20 B per
            pixel to the host), median of 10 after 3 warm-ups.
Scenes: C1 and C3 built flat on the device, C5 built two-level (--tlas), and C5 with one identity instance per object."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import WORKLOADS  # noqa: E402
from tray_racing_b200 import cuda, host  # noqa: E402

N_RAYS = 1 << 22


def median_ms(call, warm=3, reps=20):
    for _ in range(warm):
        call()
    return float(np.median([call() for _ in range(reps)]))


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None
    if cuda.device_count() < 1:
        raise SystemExit("hit_attr_perf needs a CUDA device")

    def emit(d):
        print(json.dumps(d), flush=True)
        if out:
            out.write(json.dumps(d) + "\n"); out.flush()

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    emit({"gpu": gpu})

    for name, which, instanced in (("c1", "c1", False), ("c3", "c3", False), ("c5_tlas", "c5", False), ("c5_identity_instances", "c5", True)):
        wl = WORKLOADS[which]
        m = host.Mesh.generate(wl["scene"], wl["seed"], 1.0)
        tris = np.ascontiguousarray(m.tris(), np.float32).reshape(-1, 3, 3)
        offs = m.object_offsets() if wl["tlas"] else None
        sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
        if instanced:
            n_obj = offs.size - 1
            sc.set_instances(np.arange(n_obj, dtype=np.uint32), np.tile(np.eye(3, 4, dtype=np.float32), (n_obj, 1, 1)))
        del tris
        w, h = wl["w"], wl["h"]
        view = host.view_from_camera(m.camera, w, h)

        # ---- batch: bounce rays of a frame ----
        sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_KEEP_RAYS, timed=False)
        sc.sync()
        f = sc.download(primary=True, bounce_rays=True)
        rays = f["bounce_rays"][f["primary"]["t"] < np.float32(3.402823466e+38)]
        rays = np.resize(rays, N_RAYS)
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_hits = torch.zeros(N_RAYS * 8, dtype=torch.uint8, device="cuda")
        d_ids = torch.zeros(N_RAYS, dtype=torch.int32, device="cuda") if instanced else None
        d_attrs = torch.zeros(N_RAYS * 20, dtype=torch.uint8, device="cuda")
        if instanced:
            trace = lambda: sc.traverse_instance_device(d_rays.data_ptr(), N_RAYS, d_hits.data_ptr(), d_ids.data_ptr(), timed=True)
        else:
            trace = lambda: sc.traverse_device(d_rays.data_ptr(), N_RAYS, d_hits.data_ptr(), timed=True)
        ms_trace = median_ms(trace)
        ms_attr = median_ms(lambda: sc.hit_attributes_device(d_rays.data_ptr(), d_hits.data_ptr(), None if d_ids is None else d_ids.data_ptr(),
                                                             N_RAYS, d_attrs.data_ptr(), timed=True))
        hit = float((d_hits.cpu().numpy().view(host.HIT_DTYPE)["prim"] != 0xFFFFFFFF).mean())
        emit(dict(measure="batch", scene=name, n_rays=N_RAYS, hit_fraction=hit, ms_trace=ms_trace, ms_hit_attributes=ms_attr,
                  attr_over_trace=ms_attr / ms_trace, l2_flushed=False))
        del d_rays, d_hits, d_ids, d_attrs
        torch.cuda.empty_cache()

        # ---- frame ----
        for fw, fh in ((1920, 1080), (3840, 2160)):
            v = host.view_from_camera(m.camera, fw, fh)
            ms_frame = median_ms(lambda: sc.render_frame_ms(v, fw, fh, 0), reps=10)

            def download():
                t0 = time.perf_counter()
                sc.download_attributes(primary=True, bounce=True)
                return (time.perf_counter() - t0) * 1e3
            ms_dl = median_ms(download, reps=10)
            emit(dict(measure="frame", scene=name, frame=f"{fw}x{fh}", ms_render_frame=ms_frame, ms_download_attributes_wall=ms_dl))
        sc.close()


if __name__ == "__main__":
    main()
