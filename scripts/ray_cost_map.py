#!/usr/bin/env python
"""Where in the image does a BVH cost what it costs?  Per-pixel ray cost maps of the BASELINE configs, for the host builder's
tree (binned SAH, libtray_host) and the device builder's (tray_cuda_scene_build), from the counting kernels' per-ray records
(tray_cuda_scene_set_ray_cost + tray_cuda_frame_download_cost).  GPU only.

For each config and builder one frame is rendered with TRAY_RENDER_BOUNCE | TRAY_RENDER_COUNTERS and ray costs on; written to
--out DIR:
  <config>_<builder>.npz                   the per-pixel records (primary, bounce; row-major h x w, fields nodes tris instances
                                           stack) and the primary hit mask (bounce records exist where it is set)
  <config>_<builder>_<pass>_<field>.ppm    heat maps of `nodes` and `tris` for the primary and the bounce pass
  <config>_device_minus_host_<pass>_nodes.ppm   the per-pixel difference of `nodes` (device tree minus host tree)
  ray_cost_summary.json                    per config, builder and pass: mean, p50, p90, p99 and max of every field and a
                                           histogram of `stack`; per config the host/device difference of `nodes`
With --time N it also times the counted frame of each config with ray costs off and on, N times each, alternated.

Heat-map ramp: black -> blue -> cyan -> green -> yellow -> red -> white, linear in the value, clipped at the frame's 99th
percentile (so that a few extreme pixels do not flatten the rest).  It is this project's own ramp, not the reference's
PROFILE_RT `temperature()` colouring, which is not available here.  The difference map is blue (device tree cheaper) through
black to red (device tree dearer), clipped at the 99th percentile of |difference|.

  python scripts/ray_cost_map.py --out DIR [--configs c1,c3,c4] [--builders host,device] [--time N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tray_racing_b200 import cuda, host  # noqa: E402

CONFIGS = {
    "c1": ("kitchen", 1, 1920, 1080, False), "c2": ("demoscene", 2, 1920, 1080, False), "c3": ("hairball", 3, 1920, 1080, False),
    "c4": ("sanmiguel", 4, 3840, 2160, False), "c5": ("caldera", 5, 3840, 2160, True),
}
FIELDS = ("nodes", "tris", "instances", "stack")
FLAGS = cuda.RENDER_BOUNCE | cuda.RENDER_COUNTERS
INVALID = 0xFFFFFFFF
RAMP = np.array([[0, 0, 0], [0, 0, 255], [0, 255, 255], [0, 255, 0], [255, 255, 0], [255, 0, 0], [255, 255, 255]], np.float64)


def ramp(v, top):
    """values -> RGB8 on RAMP, linear in v / top, clipped to [0, 1]"""
    x = np.clip(v.astype(np.float64) / max(float(top), 1e-9), 0.0, 1.0) * (len(RAMP) - 1)
    i = np.minimum(x.astype(np.int64), len(RAMP) - 2)
    f = (x - i)[..., None]
    return (RAMP[i] * (1 - f) + RAMP[i + 1] * f).round().astype(np.uint8)


def diverging(d, top):
    x = np.clip(d.astype(np.float64) / max(float(top), 1e-9), -1.0, 1.0)
    rgb = np.zeros(d.shape + (3,), np.float64)
    rgb[..., 0] = np.maximum(x, 0) * 255
    rgb[..., 2] = np.maximum(-x, 0) * 255
    return rgb.round().astype(np.uint8)


def write_ppm(path, rgb):
    h, w, _ = rgb.shape
    with open(path, "wb") as f:
        f.write(b"P6\n%d %d\n255\n" % (w, h))
        f.write(np.ascontiguousarray(rgb).tobytes())


def stats(c):
    """mean, p50, p90, p99, max of every field over the records `c`, and the histogram of `stack` (index = entries)"""
    out = {"rays": int(c.size)}
    for f in FIELDS:
        v = c[f].astype(np.float64)
        out[f] = {"mean": float(v.mean()) if v.size else 0.0,
                  **{f"p{q}": float(np.percentile(v, q)) if v.size else 0.0 for q in (50, 90, 99)},
                  "max": int(c[f].max()) if v.size else 0, "sum": int(c[f].sum(dtype=np.uint64))}
    out["stack_histogram"] = np.bincount(c["stack"], minlength=int(c["stack"].max()) + 1 if c.size else 1).tolist()
    return out


def scene_for(builder, mesh, tlas):
    if builder == "host":
        p = host.PackedScene(mesh, use_tlas=tlas)
        return cuda.TrayCudaScene.from_packed(p), p.tlas_start
    if tlas:
        raise SystemExit("the device builder's two-level scenes take object offsets; run the flat configs (c1 .. c4)")
    return cuda.TrayCudaScene.build(mesh.tris()), 0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--configs", default="c1,c3,c4")
    ap.add_argument("--builders", default="host,device")
    ap.add_argument("--out", required=True)
    ap.add_argument("--time", type=int, default=0, help="also time the counted frame with ray costs off / on, N times each")
    a = ap.parse_args()
    if cuda.device_count() < 1:
        raise SystemExit("ray_cost_map.py needs a CUDA device (the counting kernels run there; there is no CPU path)")
    os.makedirs(a.out, exist_ok=True)
    builders = a.builders.split(",")
    summary = {"device": None, "configs": {}}
    try:                                                # a number is only worth something with the card and its power limit
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        summary["device"] = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        pass
    for cfg in a.configs.split(","):
        name, seed, w, h, tlas = CONFIGS[cfg]
        mesh = host.Mesh.generate(name, seed, 1.0)
        res = {"scene": name, "frame": [w, h], "tlas": tlas, "builders": {}}
        nodes = {}
        for b in builders:
            sc, tlas_start = scene_for(b, mesh, tlas)
            try:
                view = host.view_from_camera(mesh.camera, w, h, tlas_start)
                sc.set_ray_cost(True)
                sc.render(view, w, h, 0, FLAGS)
                c = sc.download_cost(primary=True, bounce=True)
                hit = sc.download(primary=True)["primary"]["prim"] != INVALID
                cp, cb = sc.counters()
                for k, cnt in (("primary", cp), ("bounce", cb)):          # the records are the counters, ray by ray
                    assert all(int(c[k][f].sum(dtype=np.uint64)) == cnt[f] for f in ("nodes", "tris", "instances")), (cfg, b, k)
                timing = None
                if a.time:
                    ms = {"off": [], "on": []}
                    for _ in range(2):                                   # warm-up, both settings
                        for on in (False, True):
                            sc.set_ray_cost(on)
                            sc.render_frame_ms(view, w, h, 0, FLAGS)
                    for _ in range(a.time):
                        for on in (False, True):
                            sc.set_ray_cost(on)
                            ms["on" if on else "off"].append(sc.render_frame_ms(view, w, h, 0, FLAGS))
                    timing = {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "n": len(v)} for k, v in ms.items()}
                    print(f"{cfg} {b}: counted frame {timing['off']['median_ms']:.3f} ms with ray costs off, "
                          f"{timing['on']['median_ms']:.3f} ms on (median of {a.time})", flush=True)
            finally:
                sc.close()
            np.savez_compressed(os.path.join(a.out, f"{cfg}_{b}.npz"), primary=c["primary"].reshape(h, w),
                                bounce=c["bounce"].reshape(h, w), primary_hit=hit.reshape(h, w))
            for k in ("primary", "bounce"):
                for f in ("nodes", "tris"):
                    v = c[k][f].reshape(h, w)
                    sel = c[k][f][hit] if k == "bounce" else c[k][f]
                    top = np.percentile(sel, 99) if sel.size else 1
                    write_ppm(os.path.join(a.out, f"{cfg}_{b}_{k}_{f}.ppm"), ramp(v, top))
            res["builders"][b] = {"primary": stats(c["primary"]), "bounce": stats(c["bounce"][hit]),
                                  "counters": {"primary": cp, "bounce": cb}}
            if timing:
                res["builders"][b]["counted_frame_ms"] = timing
            nodes[b] = {"primary": c["primary"]["nodes"].astype(np.int64), "bounce": c["bounce"]["nodes"].astype(np.int64)}
            print(cfg, b, json.dumps({k: {f: res["builders"][b][k][f]["mean"] for f in FIELDS} for k in ("primary", "bounce")}), flush=True)
        if "host" in nodes and "device" in nodes:
            res["device_minus_host_nodes"] = {}
            for k in ("primary", "bounce"):
                d = nodes["device"][k] - nodes["host"][k]
                n1 = max(1, d.size // 100)
                worst = np.sort(d)[::-1][:n1]                             # the 1 % of pixels the device tree made dearest
                worst_abs = np.sort(np.abs(d))[::-1][:n1]
                total, total_abs = int(d.sum()), int(np.abs(d).sum())
                res["device_minus_host_nodes"][k] = {
                    "total": total, "mean_per_pixel": float(d.mean()), "host_total": int(nodes["host"][k].sum()),
                    "pixels_dearer": int((d > 0).sum()), "pixels_cheaper": int((d < 0).sum()),
                    "worst_1pct_share_of_total": float(worst.sum() / total) if total else None,
                    "worst_1pct_share_of_abs_total": float(worst_abs.sum() / total_abs) if total_abs else None}
                top = np.percentile(np.abs(d), 99)
                write_ppm(os.path.join(a.out, f"{cfg}_device_minus_host_{k}_nodes.ppm"), diverging(d.reshape(h, w), top))
            print(cfg, "device - host nodes:", json.dumps(res["device_minus_host_nodes"]), flush=True)
        summary["configs"][cfg] = res
    with open(os.path.join(a.out, "ray_cost_summary.json"), "w") as f:
        json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
