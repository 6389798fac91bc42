"""CPU tests of the host-side mirror: OBJ loading (reference src/main.rs:493-561), the CWBVH producer and its
format (reference embree/src/bvh_embree_to_cwbvh.rs:85-186), the cwbvh_gpu_runner marshalling
(reference src/rt_gpu/mod.rs:16-112) and the camera uniform (reference src/main.rs:589-617)."""
import os

import numpy as np
import pytest

import oracle_binding as ob
from conftest import ROOT
from tray_racing_b200 import host


def prim_boxes(tris):
    t = np.asarray(tris, dtype=np.float32).reshape(-1, 3, 3)
    return t.min(1), t.max(1)


def test_obj_loader_semantics(tmp_path):
    """triangles, quads -> (a,b,c),(a,c,d), one object per `o`, 1-based and negative indices, v/vt/vn forms."""
    p = tmp_path / "m.obj"
    p.write_text("""# test
o first
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
vn 0 0 1
f 1/1/1 2/1/1 3/1/1
f 1 2 3 4
o second
v 0 0 1
v 1 0 1
v 0 1 1
f -3//1 -2//1 -1//1
""")
    m = host.Mesh.load_obj(str(p))
    assert m.n_objects == 2 and m.n_tris == 4
    assert list(m.object_offsets()) == [0, 3, 4]
    t = m.tris().reshape(-1, 3, 3)
    assert (t[0] == [[0, 0, 0], [1, 0, 0], [1, 1, 0]]).all()
    assert (t[1] == [[0, 0, 0], [1, 0, 0], [1, 1, 0]]).all() and (t[2] == [[0, 0, 0], [1, 1, 0], [0, 1, 0]]).all()
    assert (t[3] == [[0, 0, 1], [1, 0, 1], [0, 1, 1]]).all()
    with pytest.raises(RuntimeError):
        host.Mesh.load_obj(str(tmp_path / "missing.obj"))


def test_golden_fixtures_match_reference_asset_counts(cornell, box):
    # SURVEY.md §4: cornell_box.obj = 3,968 triangles in 5 objects, box.obj = 14 triangles in 2 objects
    assert (cornell.n_tris, cornell.n_objects) == (3968, 5)
    assert (box.n_tris, box.n_objects) == (14, 2)


def test_obj_loader_reads_back_the_golden_meshes(cornell, box, tmp_path):
    """The golden meshes written as OBJ files the way exporters write them (shared vertices per object, vt / vn records,
    v/vt/vn and negative v//vn face references, full float32 precision): the loader gives the same triangles and objects."""
    for name, mesh in (("cornell_box", cornell), ("box", box)):
        tris, offs = mesh.tris().reshape(-1, 3, 3), mesh.object_offsets()
        lines, base = ["# written by test_obj_loader_reads_back_the_golden_meshes", "vt 0 0", "vn 0 0 1"], 0
        for k in range(len(offs) - 1):
            verts, face = np.unique(tris[int(offs[k]):int(offs[k + 1])].reshape(-1, 3), axis=0, return_inverse=True)
            lines.append(f"o object{k}")
            lines += [f"v {x:.9g} {y:.9g} {z:.9g}" for x, y, z in verts.tolist()]
            base += len(verts)
            if k % 2:   # relative to the last vertex read
                lines += ["f " + " ".join(f"{int(i) - len(verts)}//1" for i in f) for f in face.reshape(-1, 3)]
            else:
                lines += ["f " + " ".join(f"{base - len(verts) + 1 + int(i)}/1/1" for i in f) for f in face.reshape(-1, 3)]
        p = tmp_path / f"{name}.obj"
        p.write_text("\n".join(lines) + "\n")
        m = host.Mesh.load_obj(str(p))
        assert (m.tris() == mesh.tris()).all() and (m.object_offsets() == offs).all()


@pytest.mark.parametrize("name,size", [("kitchen", 0.2), ("hairball", 0.01), ("demoscene", 0.01), ("sanmiguel", 0.004),
                                       ("caldera", 0.002), ("soup", 0.01)])
def test_builder_emits_valid_cwbvh(name, size):
    m = host.Mesh.generate(name, 11, size)
    tris = m.tris()
    nodes, pidx, depth = host.build_cwbvh(tris)
    assert nodes.shape[1] == 80 and nodes.dtype == np.uint8
    assert sorted(pidx.tolist()) == list(range(m.n_tris))                  # a permutation: every triangle once
    mn, mx = prim_boxes(tris)
    rc, rep = host.validate_cwbvh(nodes, pidx, mn, mx, stack_limit=32)     # obvhs stack depth, cwbvh.rs:87-89
    assert rc == 0, rep
    assert rep["nodes_reached"] == nodes.shape[0] and rep["prims_reached"] == m.n_tris
    assert rep["max_depth"] == depth and rep["max_stack"] < 32
    # inner children are contiguous and in slot order: child index = child_base + popcount(imask below slot)
    imask = nodes[:, 15]
    cb = nodes[:, 16:20].copy().view(np.uint32).ravel()
    n_inner = np.array([bin(int(x)).count("1") for x in imask])
    has = n_inner > 0
    assert ((cb[has] + n_inner[has]) <= nodes.shape[0]).all()
    # exponent bytes encode a power-of-two scale with 255 * scale >= node extent (bvh_embree_to_cwbvh.rs:97-110)
    assert (nodes[:, 12:15] > 0).all() and (nodes[:, 12:15] < 255).all()


def test_builder_deterministic_and_seeded():
    a = host.Mesh.generate("hairball", 3, 0.01)
    b = host.Mesh.generate("hairball", 3, 0.01)
    c = host.Mesh.generate("hairball", 4, 0.01)
    assert (a.tris() == b.tris()).all() and not (a.tris() == c.tris()).all()
    n1, p1, _ = host.build_cwbvh(a.tris(), nthreads=1)
    n2, p2, _ = host.build_cwbvh(a.tris(), nthreads=8)
    assert (n1 == n2).all() and (p1 == p2).all()                            # thread count does not change the BVH


def test_builder_edge_cases():
    one = np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], dtype=np.float32)
    nodes, pidx, depth = host.build_cwbvh(one)
    assert nodes.shape == (1, 80) and list(pidx) == [0] and depth == 1
    assert nodes[0, 15] == 0 and nodes[0, 24] == 0x20                       # imask 0, one leaf child with one triangle
    # coincident triangles (identical centroids) and a degenerate zero-area one
    many = np.repeat(one, 7, axis=0)
    many = np.concatenate([many, np.zeros((1, 9), np.float32)])
    nodes, pidx, _ = host.build_cwbvh(many)
    rc, rep = host.validate_cwbvh(nodes, pidx, *prim_boxes(many))
    assert rc == 0 and rep["prims_reached"] == 8
    # empty
    nodes, pidx, depth = host.build_cwbvh(np.zeros((0, 9), np.float32))
    assert nodes.shape == (0, 80) and len(pidx) == 0
    # max_prims_per_leaf outside the CWBVH limit of 3 is rejected (main.rs:104-108 "For CWBVH the limit is 3")
    with pytest.raises(RuntimeError):
        host.build_cwbvh(one, max_prims_per_leaf=4)


def test_validate_detects_corruption(cornell):
    nodes, pidx, _ = host.build_cwbvh(cornell.tris())
    mn, mx = prim_boxes(cornell.tris())
    bad = nodes.copy(); bad[0, 40:48] = 0; bad[0, 56:64] = 0                # collapse the root's child boxes
    rc, rep = host.validate_cwbvh(bad, pidx, mn, mx)
    assert rc != 0 and rep["box_violations"] > 0
    bad = pidx.copy(); bad[0] = bad[1]
    rc, rep = host.validate_cwbvh(nodes, bad, mn, mx)
    assert rc != 0 and rep["prim_seen_twice"] > 0 and rep["prims_missing"] > 0


def test_pack_flat_matches_cwbvh_gpu_runner_layout(cornell):
    """flat: objects flattened into one BLAS (main.rs:300-308); bvh_bytes = nodes, instance_bytes = [0;16],
    tlas_start = 0 (mod.rs:101-111); triangles permuted by primitive_indices (mod.rs:34-38)."""
    p = host.PackedScene(cornell)
    assert p.bvh_bytes.size == p.n_nodes * 5 * 4 * 4                         # mod.rs:105
    assert p.tri_bytes.size == cornell.n_tris * 48
    assert p.instance_bytes.size == 16 and not p.instance_bytes.any() and p.tlas_start == 0
    tris = cornell.tris().reshape(-1, 3, 3)
    rec = p.tri_bytes.view(np.float32).reshape(-1, 12)
    src = tris[p.prim_to_mesh_tri]
    assert (rec[:, 0:3] == src[:, 0]).all()
    assert (rec[:, 4:7] == src[:, 0] - src[:, 1]).all() and (rec[:, 8:11] == src[:, 2] - src[:, 0]).all()
    assert (host.tri_records(src.reshape(-1, 9)) == p.tri_bytes).all()


def test_pack_tlas_layout(cornell):
    """--tlas: BLAS0|BLAS1|..|TLAS, tlas_start = sum of BLAS node counts (mod.rs:62-69,88-91,99), blas_offsets in
    TLAS-leaf order (mod.rs:72-78), primitive_base_idx globalised per BLAS (mod.rs:45-47)."""
    p = host.PackedScene(cornell, use_tlas=True)
    offs = cornell.object_offsets()
    blas_nodes, tri_base = [], []
    for k in range(cornell.n_objects):
        n, pi, _ = host.build_cwbvh(cornell.tris()[int(offs[k]):int(offs[k + 1])])
        blas_nodes.append(n); tri_base.append(len(pi))
    starts = np.concatenate([[0], np.cumsum([len(n) for n in blas_nodes])])
    assert p.tlas_start == starts[-1]
    assert sorted(p.blas_offsets.tolist()) == starts[:-1].tolist()
    tri_starts = np.concatenate([[0], np.cumsum(tri_base)])
    assert (p.blas_tri_offsets == tri_starts).all()
    nodes = p.bvh_bytes.reshape(-1, 80)
    for k, n in enumerate(blas_nodes):
        got = nodes[starts[k]:starts[k + 1]].copy()
        pb = got[:, 20:24].copy().view(np.uint32).ravel() - np.uint32(tri_starts[k])
        got[:, 20:24] = pb.view(np.uint8).reshape(-1, 4)
        assert (got == n).all()
    # the TLAS is a CWBVH over the 5 BLAS boxes whose leaf "triangles" are instance slots
    tl = nodes[p.tlas_start:]
    assert len(tl) >= 1 and p.n_instances == 5
    g, l = p.geometry_of(np.array([0, tri_starts[1], tri_starts[-1] - 1]))
    assert g.tolist() == [0, 1, 4] and l.tolist() == [0, 0, tri_base[4] - 1]
    p64 = host.PackedScene(cornell, use_tlas=True, tri_stride=64)
    assert p64.tri_bytes.size == cornell.n_tris * 64 and (p64.bvh_bytes == p.bvh_bytes).all()


def test_view_uniform_is_inverse_of_glam_matrices(cornell):
    """view_inv / proj_inv against numpy float64 inverses of look_at_rh / perspective_infinite_reverse_rh."""
    w, h = 1920, 1080
    cam = cornell.camera
    v = host.view_from_camera(cam, w, h, 7)
    f = 1.0 / np.tan(0.5 * np.radians(cam.fov))
    P = np.array([[f / (w / h), 0, 0, 0], [0, f, 0, 0], [0, 0, 0, 0.01], [0, 0, -1, 0]])
    eye, at = np.array(cam.eye), np.array(cam.look_at)
    fw = (at - eye) / np.linalg.norm(at - eye)
    s = np.cross(fw, [0, 1, 0]); s /= np.linalg.norm(s)
    u = np.cross(s, fw)
    V = np.eye(4); V[0, :3], V[1, :3], V[2, :3] = s, u, -fw
    V[:3, 3] = [-s @ eye, -u @ eye, fw @ eye]
    got_p = np.array(v.proj_inv).reshape(4, 4).T
    got_v = np.array(v.view_inv).reshape(4, 4).T
    assert np.allclose(got_p, np.linalg.inv(P), rtol=1e-6, atol=1e-7)
    assert np.allclose(got_v, np.linalg.inv(V), rtol=1e-6, atol=1e-6)
    assert tuple(v.eye) == tuple(np.float32(cam.eye)) and v.tlas_start == 7
    import ctypes
    assert ctypes.sizeof(v) == 160


def test_runner_options_mirror_reference_defaults():
    from tray_racing_b200.runner import Options
    o = Options()
    # reference src/main.rs:78-83,104-108,139-142: render_time 1.0, max_prims_per_leaf 3, 1920x1080
    assert (o.width, o.height, o.render_time, o.max_prims_per_leaf, o.build) == (1920, 1080, 1.0, 3, "ploc_cwbvh")


def test_bench_workloads_and_frame_sizes():
    """bench.py: c3 grows the frame with the GPU count (weak scaling, ~N x 1080p pixels, multiples of 8); c4 / c5 keep the
    3840x2160 frame of BASELINE.json's multi-GPU configs (strong scaling), c5 through the two-level traversal."""
    import importlib
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    assert set(bench.WORKLOADS) == {"c1", "c2", "c3", "c4", "c5"}
    old = bench.WL
    try:
        bench.WL = bench.WORKLOADS["c3"]
        assert bench.frame_size(1) == (1920, 1080)
        for n in (2, 4, 8):
            w, h = bench.frame_size(n)
            assert w % 8 == 0 and h % 8 == 0 and abs(w * h / (n * 1920 * 1080) - 1) < 0.01
        for key in ("c4", "c5"):
            bench.WL = bench.WORKLOADS[key]
            assert all(bench.frame_size(n) == (3840, 2160) for n in (1, 2, 4, 8)) and bench.WL["scaling"] == "strong"
        assert bench.WORKLOADS["c5"]["tlas"] and not bench.WORKLOADS["c4"]["tlas"]
        assert "fixed frame" in bench.workload_name(3840, 2160, 8)
    finally:
        bench.WL = old


def test_host_copy_pool(tmp_path):
    """The persistent copy threads behind tray_cuda_trace's pipeline and the pinned uploads (csrc/host_copy.h): random
    sizes, three caller threads at once, byte-exact — compiled for the host alone, no CUDA call is made."""
    import subprocess
    from conftest import ROOT
    exe = tmp_path / "copy_pool_test"
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-pthread", "-I" + cuda_inc, "-I" + os.path.join(ROOT, "tray_racing_b200", "csrc"),
                           os.path.join(ROOT, "tests", "tools", "copy_pool_test.cpp"), "-o", str(exe),
                           "-L" + os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64"), "-lcudart"])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64") + ":" + os.environ.get("LD_LIBRARY_PATH", ""),
               TRAY_CUDA_COPY_THREADS="6")
    out = subprocess.run([str(exe)], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr
