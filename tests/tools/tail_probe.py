"""Dev: what does one DEPENDENT traversal step cost when a warp holds a single long ray (the drain phase of a launch)?

Test infrastructure (it uses the CPU oracle for the step counts): takes the longest primary rays of a scene, and times launches of
  (a) the L longest rays packed 32 to a warp,
  (b) the same rays one per warp: every aligned group of 32 rays is 1 long ray + 31 rays that miss the root (tmax = 0),
for each setting of the knobs given on the command line, e.g.
  python tests/tools/tail_probe.py hairball '{"TRAY_CUDA_REFILL_MIN": [4, 6], "TRAY_CUDA_TRI_WEIGHT": [3, 4]}'"""
import itertools, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_binding as ob
from tray_racing_b200 import cuda, host

scene = sys.argv[1] if len(sys.argv) > 1 else "hairball"
knobs = eval(sys.argv[2]) if len(sys.argv) > 2 else {"TRAY_CUDA_REFILL_MIN": [4, 6]}
m = host.Mesh.generate(scene, 3, 1.0)
p = host.PackedScene(m)
w, h = 1920, 1080
view = host.view_from_camera(m.camera, w, h)
orc = ob.Oracle.from_packed(p)
rays = ob.primary_rays(view, w, h)
_, cnt, tot = orc.trace(rays, counts=True)
steps = cnt["nodes"].astype(np.int64) + cnt["tris"]
order = np.argsort(-steps, kind="stable")
print(f"{scene}: steps/ray mean {steps.mean():.1f} max {steps.max()} p99.9 {np.percentile(steps, 99.9):.0f}", flush=True)
names = list(knobs)
for combo in itertools.product(*[knobs[n] for n in names]):
    for n, v in zip(names, combo):
        os.environ[n] = str(v)
    sc = cuda.TrayCudaScene.from_packed(p)
    line = []
    for L in (32, 1024, 4736):
        sel = rays[order[:L]]
        smax, smean = int(steps[order[0]]), float(steps[order[:L]].mean())
        spread = np.zeros(L * 32, dtype=ob.RAY_DTYPE)
        spread["o"] = rays["o"][0]; spread["d"] = rays["d"][0]; spread["tmax"] = 0.0      # misses the root: one node step
        spread[::32] = sel
        for label, batch in (("packed", sel), ("1/warp", spread)):
            best = 1e9
            for _ in range(5):
                t = {}
                sc.traverse(batch, t)
                best = min(best, t["ms_kernel"])
            line.append(f"L={L} {label} {best * 1e3:.0f}us ({best * 1e3 / smax:.2f} us/step of the longest, mean {smean:.0f})")
    sc.close()
    print(dict(zip(names, combo)), " | ".join(line), flush=True)
