"""Device builder against the serial reference builder (oracle/build_ref.c) on the full-size bench.py scenes C1-C5.

tests/test_build_reference.py makes the same comparison on small scenes; at 2-19 M triangles the single-threaded reference
takes minutes, so this runs by hand.  For every config it prints one line: whether nodes, prim_indices, triangle records,
blas_offsets, tlas_start and the statistics match, the device build time and the reference build time.  The references run
in worker processes while the device builds in this one.

    python tests/tools/build_parity.py [--configs c1,c2,c3,c4,c5] [--workers 5]
"""
import argparse
import concurrent.futures as cf
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCENES = {"c1": ("kitchen", 1, False), "c2": ("demoscene", 2, False), "c3": ("hairball", 3, False),
          "c4": ("sanmiguel", 4, False), "c5": ("caldera", 5, True)}
STATS = ("n_nodes", "ploc_iterations", "levels", "reinsert_passes", "reinsert_moves")


def scene(cfg):
    from tray_racing_b200 import host
    name, seed, tlas = SCENES[cfg]
    m = host.Mesh.generate(name, seed, 1.0)
    return m.tris(), (m.object_offsets() if tlas else None)


def reference(cfg):
    import oracle_binding as ob
    tris, offs = scene(cfg)
    t0 = time.perf_counter()
    r = ob.build_reference(tris, object_offsets=offs)
    r["seconds"] = time.perf_counter() - t0
    r.pop("tri_bytes")                          # rebuilt in the parent from prim_indices: keeps the pickle small
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--configs", default="c1,c2,c3,c4,c5")
    ap.add_argument("--workers", type=int, default=5)
    args = ap.parse_args()
    cfgs = [c.strip() for c in args.configs.split(",") if c.strip()]
    from tray_racing_b200 import cuda, host
    for k in ("TRAY_CUDA_BUILD_REINSERT", "TRAY_CUDA_BUILD_REINSERT_VISITS", "TRAY_CUDA_BUILD_REINSERT_ROUNDS", "TRAY_BUILD_PLOC_TAIL"):
        os.environ.pop(k, None)                 # the defaults, which the reference's defaults restate
    ok_all = True
    with cf.ProcessPoolExecutor(max_workers=args.workers) as pool:
        futs = {c: pool.submit(reference, c) for c in cfgs}
        for c in cfgs:
            tris, offs = scene(c)
            t0 = time.perf_counter()
            sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
            dev_s = time.perf_counter() - t0
            nodes, tri_bytes, pi = sc.download_bvh()
            blas, info, st = sc.download_instances(), sc.info(), sc.build_stats
            sc.close()
            r = futs[c].result()
            checks = {
                "nodes": np.array_equal(nodes, r["nodes"]),
                "prim_indices": np.array_equal(pi, r["prim_indices"]),
                "tri_bytes": np.array_equal(tri_bytes, host.tri_records(tris.reshape(-1, 3, 3)[r["prim_indices"]], 48)),
                "blas_offsets": np.array_equal(blas, r["blas_offsets"]),
                "tlas_start": info["tlas_start"] == r["info"]["tlas_start"],
                "stats": all(st[k] == r["build_stats"][k] for k in STATS),
                "sah": all(abs(st[k] - r["build_stats"][k]) <= 1e-5 * abs(r["build_stats"][k]) for k in ("sah_before", "sah_after")),
            }
            ok = all(checks.values())
            ok_all &= ok
            bad = [k for k, v in checks.items() if not v]
            print(f"{c} {SCENES[c][0]:9s} {tris.shape[0]:>9,d} tris {'two-level' if offs is not None else 'flat     '}  "
                  f"{'MATCH' if ok else 'DIFFER: ' + ', '.join(bad)}  nodes {int(st['n_nodes']):,}  moves {st['reinsert_moves']:,}  "
                  f"device build {dev_s:.2f} s ({st['ms_total']:.0f} ms in the builder)  reference {r['seconds']:.1f} s", flush=True)
            if not ok:
                print("   device   ", {k: st[k] for k in STATS + ("sah_before", "sah_after")})
                print("   reference", {k: r["build_stats"][k] for k in STATS + ("sah_before", "sah_after")})
    return 0 if ok_all else 1


if __name__ == "__main__":
    sys.exit(main())
