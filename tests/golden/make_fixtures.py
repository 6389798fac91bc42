"""Regenerates tests/golden/*.npz from the reference's in-tree assets; the tests only read the committed .npz files.

  python tests/golden/make_fixtures.py <checkout of the reference>

  cornell_box.npz  triangles (n,9) f32 + per-object offsets of assets/obj/cornell_box.obj parsed with
                   `load_meshs` semantics (reference src/main.rs:530-559), camera of
                   assets/scenes/cornell_box.ron:3-8
  box.npz          same for assets/obj/box.obj / assets/scenes/box.ron:3-8
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tray_racing_b200 import host  # noqa: E402

if len(sys.argv) != 2:
    sys.exit("usage: python tests/golden/make_fixtures.py <checkout of the reference>")
REF = os.path.join(sys.argv[1], "assets")
for name, eye, look, fov in (("cornell_box", (0.0, 1.0, 2.1), (0.0, 1.0, 0.0), 90.0),
                             ("box", (3.0, 1.5, 1.4), (-3.9438584, 1.5, -1.7303504), 90.0)):
    m = host.Mesh.load_obj(f"{REF}/obj/{name}.obj")
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), tris=m.tris(), offsets=m.object_offsets(),
                        eye=np.float32(eye), look_at=np.float32(look), fov=np.float32(fov))
    print(name, m.n_tris, "triangles", m.n_objects, "objects")
