"""Dev: sweep the scheduler knobs (env-read at scene creation) on one scene; prints ms primary/bounce."""
import itertools, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tray_racing_b200 import cuda, host
scene = sys.argv[1] if len(sys.argv) > 1 else "hairball"
m = host.Mesh.generate(scene, 3, 1.0)
p = host.PackedScene(m)
w, h = 1920, 1080
view = host.view_from_camera(m.camera, w, h)
knobs = {"TRAY_CUDA_TRI_WEIGHT": [1, 2, 3, 4, 8, 64], "TRAY_CUDA_REFILL_MIN": [1, 4, 8, 16, 24]}
if len(sys.argv) > 2:
    knobs = eval(sys.argv[2])
names = list(knobs)
for combo in itertools.product(*[knobs[n] for n in names]):
    for n, v in zip(names, combo):
        os.environ[n] = str(v)
    sc = cuda.TrayCudaScene.from_packed(p)
    best = None
    for f in range(6):
        ms = sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | (cuda.RENDER_OVERLAP if os.environ.get("SWEEP_OVERLAP") == "1" else 0))
        if f >= 1:
            best = ms if best is None else (min(best[0], ms[0]), min(best[1], ms[1]))
    sc.close()
    print(scene, dict(zip(names, combo)), "primary %.3f bounce %.3f  sum %.3f" % (best + (best[0] + best[1],)), flush=True)
