"""Hit attributes (tray_cuda_hit_attributes, tray_cuda_frame_download_attributes): u, v and Ng of every hit, as the triangle test
computed them.

tests/hit_attr_ref.c restates the triangle test's arithmetic for one (ray, prim[, W]) and also returns its own t.  The CPU tests
hold that reference to the oracle (its t is the oracle's t, bit for bit, on every oracle hit) and to geometry (u, v, 1 - u - v in
[0, 1], the barycentric point on the ray); the `gpu` tests hold the device to the reference byte for byte, for batches and
frames, on flat, two-level and instanced scenes."""
import ctypes as C
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_binding as ob
from conftest import ROOT, random_rays
from test_build_reference import many_small_objects, rays_at
from test_instances import cornell_instances, xforms
from tray_racing_b200 import cuda, host

gpu = pytest.mark.gpu
INVALID = 0xFFFFFFFF
F32_MAX = np.float32(3.402823466e+38)
KERNEL_STACK = 48


# ---- the serial reference --------------------------------------------------------------------------------------------------

_alib = None


def _attr_lib():
    """tests/hit_attr_ref.c compiled with oracle/Makefile's flags, linked against the oracle library"""
    global _alib
    if _alib is None:
        ob.lib()
        d = tempfile.mkdtemp(prefix="tray_hit_attr_ref_")
        try:
            so = os.path.join(d, "libhit_attr_ref.so")
            odir = os.path.join(ROOT, "oracle")
            subprocess.check_call(["/usr/bin/gcc", "-O3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", so,
                                   os.path.join(ROOT, "tests", "hit_attr_ref.c"), "-L" + odir, "-ltray_oracle", "-Wl,-rpath," + odir, "-lm"])
            L = C.CDLL(so)
        finally:
            shutil.rmtree(d, ignore_errors=True)
        vp = C.c_void_p
        L.attr_ref.restype = None
        L.attr_ref.argtypes = [vp, C.c_uint64, C.c_uint32, vp, C.c_uint32, vp, vp, vp, C.c_uint64, C.c_int, vp, vp]
        _alib = L
    return _alib


def reference(rec, stride, rays, hits, w2o=None, inst=None, zerodir_box_only=False):
    """(attrs ATTR_DTYPE, t float32) of every hit; w2o: world_to_object by instance (n, 3, 4), inst: the instance of each hit"""
    rec = np.ascontiguousarray(rec, np.uint8)
    rays = np.ascontiguousarray(rays, ob.RAY_DTYPE)
    hits = np.ascontiguousarray(hits, ob.HIT_DTYPE)
    n = rays.size
    attrs, t = np.empty(n, cuda.ATTR_DTYPE), np.empty(n, np.float32)
    w = None if w2o is None else np.ascontiguousarray(w2o, np.float32).reshape(-1, 12)
    ids = None if inst is None else np.ascontiguousarray(inst, np.uint32)
    _attr_lib().attr_ref(rec.ctypes.data, rec.size // stride, stride, None if w is None else w.ctypes.data, 0 if w is None else w.shape[0],
                         rays.ctypes.data, hits.ctypes.data, None if ids is None else ids.ctypes.data, n, int(zerodir_box_only),
                         attrs.ctypes.data, t.ctypes.data)
    return attrs, t


def words(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32).reshape(len(a), a.dtype.itemsize // 4)


def same_bytes(a, b):
    return np.array_equal(words(a), words(b))


def is_miss(a):
    return (words(a) == 0xFFFFFFFF).all(axis=1)


def golden_scene(name, stride):
    g = np.load(os.path.join(ROOT, "tests", "golden", f"{name}.npz"))
    cam = host.Camera(tuple(float(x) for x in g["eye"]), tuple(float(x) for x in g["look_at"]), float(g["fov"]))
    mesh = host.Mesh.from_tris(g["tris"], g["offsets"], cam)
    return host.PackedScene(mesh, tri_stride=stride), g["tris"].reshape(-1, 3, 3), cam


def mixed_rays(tris, n, seed):
    """rays at triangles, random rays around the scene, and axis-aligned rays (zero direction components)"""
    ext = float(np.abs(tris).max())
    a = rays_at(tris, n, seed)
    b = random_rays(n, seed=seed + 1, lo=-ext, hi=ext, axis_fraction=0.2)
    c = a[: n // 4].copy()
    rng = np.random.default_rng(seed + 2)
    ax = rng.integers(0, 3, c.size)
    c["d"] = 0
    c["d"][np.arange(c.size), ax] = rng.choice([-1.0, 1.0], c.size).astype(np.float32)
    tgt = tris.reshape(-1, 3, 3)[rng.integers(0, tris.reshape(-1, 3, 3).shape[0], c.size)].astype(np.float64).mean(axis=1)
    c["o"] = (tgt - c["d"].astype(np.float64) * 3 * ext).astype(np.float32)
    return np.concatenate([a, b, c])


def vertices(rec, stride, prim):
    """(v0, v1, v2) in double from the BVH-ordered records (stride 24: the f16 edges as the test unpacks them)"""
    r = np.asarray(rec, np.uint8).reshape(-1, stride)[prim]
    v0 = r[:, 0:12].copy().view(np.float32).astype(np.float64)
    if stride == 24:
        e = r[:, 12:24].copy().view(np.uint32)
        e2 = (e & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)
        e1 = -(e >> 16).astype(np.uint16).view(np.float16).astype(np.float64)
    else:
        e1 = r[:, 16:28].copy().view(np.float32).astype(np.float64)
        e2 = r[:, 32:44].copy().view(np.float32).astype(np.float64)
    return v0, v0 - e1, v0 + e2


# ---- CPU -------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("stride", [24, 48, 64])
@pytest.mark.parametrize("name", ["cornell_box", "box"])
def test_reference_follows_the_oracle_test(name, stride):
    """the reference's t is the oracle's t on every oracle hit, bit for bit; u, v, 1 - u - v in [0, 1]; the barycentric point is
    on the ray"""
    packed, tris, cam = golden_scene(name, stride)
    orc = ob.Oracle.from_packed(packed)
    rec = packed.tri_bytes
    rays = np.concatenate([mixed_rays(tris, 6000, seed=stride), ob.primary_rays(host.view_from_camera(cam, 96, 64), 96, 64)])
    for any_hit in (False, True):
        hits = orc.trace(rays, any_hit=any_hit, stack_limit=KERNEL_STACK)
        hit = hits["prim"] != INVALID
        assert hit.sum() > 3000
        attrs, t = reference(rec, stride, rays, hits)
        assert np.array_equal(t[hit].view(np.uint32), hits["t"][hit].view(np.uint32))
        assert is_miss(attrs[~hit]).all() and (t[~hit].view(np.uint32) == 0xFFFFFFFF).all()
        u, v = attrs["u"][hit].astype(np.float64), attrs["v"][hit].astype(np.float64)
        for x in (u, v, 1.0 - u - v):
            assert (x >= -1e-6).all() and (x <= 1 + 1e-6).all()
        assert (attrs["u"][hit] >= 0).all() and (attrs["v"][hit] >= 0).all()
        # w v0 + u v1 + v v2 against o + t d in double, away from grazing incidence: the f32 errors of u, v and t scale with the
        # triangle's and the ray's coordinates over |cos|; the bound is 2^-16 of those.
        h = np.flatnonzero(hit)
        v0, v1, v2 = vertices(rec, stride, hits["prim"][h])
        o, d = rays["o"][h].astype(np.float64), rays["d"][h].astype(np.float64)
        p = (1 - u - v)[:, None] * v0 + u[:, None] * v1 + v[:, None] * v2
        q = o + t[h].astype(np.float64)[:, None] * d
        n = np.cross(v1 - v0, v2 - v0)
        cos = np.abs((n * d).sum(1)) / (np.linalg.norm(n, axis=1) * np.linalg.norm(d, axis=1))
        steep = cos > 0.1
        assert steep.sum() > 1000
        scale = np.abs(np.concatenate([v0, v1, v2, o, q], axis=1)).max(axis=1)
        err = np.linalg.norm(p - q, axis=1)
        assert (err[steep] <= np.ldexp(scale[steep], -16) / cos[steep]).all(), float((err[steep] / scale[steep] * cos[steep]).max())
        if stride == 64:                                               # the record's normal, as stored
            stored = np.asarray(rec, np.uint8).reshape(-1, 64)[hits["prim"][hit], 48:60].copy().view(np.float32)
            assert np.array_equal(attrs["ng"][hit].view(np.uint32), stored.view(np.uint32))


@pytest.mark.parametrize("stride", [24, 48, 64])
def test_identity_instances_reference_is_the_plain_one(stride):
    tris, offs = many_small_objects(200, seed=stride)
    r = ob.build_reference(tris, tri_stride=stride, object_offsets=offs)
    orc = ob.Oracle(r["nodes"], r["tri_bytes"], stride, r["blas_offsets"], r["info"]["tlas_start"], True)
    rays = np.concatenate([rays_at(tris, 4000, seed=1), random_rays(4000, seed=2, axis_fraction=0.2)])
    hits = orc.trace(rays, stack_limit=KERNEL_STACK)
    assert (hits["prim"] != INVALID).sum() > 2000
    inst = np.random.default_rng(3).integers(0, 7, rays.size).astype(np.uint32)
    plain, t = reference(r["tri_bytes"], stride, rays, hits)
    ident, ti = reference(r["tri_bytes"], stride, rays, hits, np.tile(np.eye(3, 4, dtype=np.float32), (7, 1, 1)), inst)
    assert same_bytes(plain, ident) and np.array_equal(t.view(np.uint32), ti.view(np.uint32))
    # an instance past the transforms is a miss
    inst[:10] = 7
    out, _ = reference(r["tri_bytes"], stride, rays, hits, np.tile(np.eye(3, 4, dtype=np.float32), (7, 1, 1)), inst)
    assert is_miss(out[:10]).all()


def test_wrappers_reject_bad_input_before_the_library():
    sc = cuda.TrayCudaScene.__new__(cuda.TrayCudaScene)
    sc._h = C.c_void_p()
    rays, hits = np.zeros(4, ob.RAY_DTYPE), np.zeros(4, ob.HIT_DTYPE)
    bad = [(np.zeros(4, np.float32), hits, None),                           # not rays
           (rays, np.zeros(4, np.uint64), None),                             # not hits
           (rays, hits[:3], None),                                           # lengths differ
           (rays.reshape(2, 2), hits.reshape(2, 2), None),                   # 2-D
           (rays, hits, np.zeros(3, np.uint32)),                             # ids of another length
           (rays, hits, np.zeros(4, np.float32)),                            # float ids
           (rays, hits, np.array([-1, 0, 0, 0])),                            # negative id
           (rays, hits, np.zeros(4, np.uint32))]                             # ids on a scene that is not instanced
    for r, h, i in bad:
        with pytest.raises(ValueError):
            sc.hit_attributes(r, h, i)


def test_attribute_calls_without_a_scene():
    L = cuda.lib()
    ms = C.c_float()
    assert L.tray_cuda_hit_attributes(None, None, None, None, 0, None, C.byref(ms)) == -1
    assert L.tray_cuda_hit_attributes_device(None, None, None, None, 0, None, None, None) == -1
    assert L.tray_cuda_frame_download_attributes(None, None, None) == -1


def test_attr_layout_agrees_between_header_numpy_and_rust():
    header = open(os.path.join(ROOT, "include", "tray_cuda.h")).read()
    body = re.search(r"typedef struct tray_hit_attr \{(.*?)\} tray_hit_attr;", header, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    assert re.findall(r"float\s+([a-z_\[\]0-9, ]+);", body) == ["u, v", "ng[3]"]
    assert cuda.ATTR_DTYPE.itemsize == 20
    assert [(n, cuda.ATTR_DTYPE.fields[n][1]) for n in ("u", "v", "ng")] == [("u", 0), ("v", 4), ("ng", 8)]
    assert cuda.ATTR_DTYPE.fields["ng"][0].shape == (3,)
    rust = open(os.path.join(ROOT, "tray_cuda", "src", "lib.rs")).read()
    m = re.search(r"#\[repr\(C\)\]\s*#\[derive\([^)]*\)\]\s*pub struct TrayHitAttr \{ pub u: f32, pub v: f32, pub ng: \[f32; 3\] \}", rust)
    assert m, "TrayHitAttr in tray_cuda/src/lib.rs differs from tray_hit_attr"
    src = open(os.path.join(ROOT, "tray_racing_b200", "csrc", "tray_cuda.cu")).read()
    assert "static_assert(sizeof(tray_hit_attr) == 20" in src


# ---- GPU: batches ----------------------------------------------------------------------------------------------------------


def device_attrs(sc, rays, hits, ids=None, stream=0):
    """hit_attributes_device on copies of the arrays in device memory"""
    import torch
    n = rays.size
    d_rays = torch.from_numpy(np.ascontiguousarray(rays).view(np.uint8).copy()).cuda()
    d_hits = torch.from_numpy(np.ascontiguousarray(hits).view(np.uint8).copy()).cuda()
    d_ids = None if ids is None else torch.from_numpy(np.ascontiguousarray(ids, np.uint32).view(np.int32).copy()).cuda()
    d_out = torch.zeros(n * 20, dtype=torch.uint8, device="cuda")
    sc.hit_attributes_device(d_rays.data_ptr(), d_hits.data_ptr(), None if d_ids is None else d_ids.data_ptr(), n, d_out.data_ptr(),
                             stream=stream, timed=True)
    return d_out.cpu().numpy().view(cuda.ATTR_DTYPE)


def check_batch(sc, rays, any_hit, ids_of=None, zerodir=False):
    """host and device forms == the reference, byte for byte; returns (hits, attrs)"""
    rec = sc.download_bvh(prim_indices=False)[1]
    stride = sc.info()["tri_stride"]
    w2o = ids = None
    if ids_of is None:
        hits = sc.traverse(rays, any_hit=any_hit)
    else:
        hits, ids = sc.traverse_instance(rays, any_hit=any_hit)
        w2o = sc.download_instance_xforms()[1]
    want, _ = reference(rec, stride, rays, hits, w2o, ids, zerodir)
    got = sc.hit_attributes(rays, hits, ids)
    assert same_bytes(got, want), int((words(got) != words(want)).any(axis=1).sum())
    assert same_bytes(device_attrs(sc, rays, hits, ids), want)
    assert same_bytes(sc.hit_attributes(rays, hits, ids), got)           # deterministic
    return hits, got


@gpu
@pytest.mark.parametrize("builder", ["host", "device"])
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_flat_scenes(stride, builder):
    packed, tris, _ = golden_scene("cornell_box", stride)
    sc = cuda.TrayCudaScene.from_packed(packed) if builder == "host" else cuda.TrayCudaScene.build(tris, tri_stride=stride)
    try:
        small = mixed_rays(tris, 3000, seed=stride)
        for any_hit in (False, True):
            hits, _ = check_batch(sc, small, any_hit)
            assert (hits["prim"] != INVALID).sum() > 3000
        big = mixed_rays(tris, 1 << 17, seed=7)                        # >= 2^18 rays: the pipelined trace
        assert big.size >= 1 << 18
        check_batch(sc, big, False)
    finally:
        sc.close()


@gpu
def test_zero_direction_variant():
    packed, tris, _ = golden_scene("cornell_box", 48)
    sc = cuda.TrayCudaScene.from_packed(packed)
    try:
        rays = mixed_rays(tris, 4000, seed=5)
        zero = (rays["d"] == 0).any(axis=1)
        assert zero.sum() > 1000
        hits, default = check_batch(sc, rays, False)
        sc.set_variant(cuda.VARIANT_ZERODIR_BOX_ONLY)
        _, raw = check_batch(sc, rays, False, zerodir=True)
        # the same hits, attributed with the caller's direction instead of the patched one
        again = sc.hit_attributes(rays, hits)
        want, _ = reference(sc.download_bvh(prim_indices=False)[1], 48, rays, hits, zerodir_box_only=True)
        assert same_bytes(again, want)
        hit = hits["prim"] != INVALID
        assert not same_bytes(again[zero & hit], default[zero & hit])
        assert same_bytes(again[~zero], default[~zero])
        sc.set_variant(0)
        assert same_bytes(sc.hit_attributes(rays, hits), default)
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_two_level_scenes(stride):
    tris, offs = many_small_objects(300, seed=stride + 40)
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=offs)
    try:
        rays = np.concatenate([rays_at(tris, 5000, seed=1), random_rays(3000, seed=2, axis_fraction=0.2)])
        for any_hit in (False, True):
            hits, _ = check_batch(sc, rays, any_hit)
            assert (hits["prim"] != INVALID).sum() > 2000
    finally:
        sc.close()


def placed(kind, stride, n_obj=30, n_inst=400, seed=7):
    tris, offs = many_small_objects(n_obj, seed=seed + 1)
    sc = cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=offs)
    rng = np.random.default_rng(seed)
    roots = rng.integers(0, n_obj, size=n_inst).astype(np.uint32)
    xf = xforms(kind, n_inst, seed)
    sc.set_instances(roots, xf)
    return sc, tris, offs, roots, xf


def rays_at_instances(tris, offs, roots, xf, n, seed):
    m = xf.astype(np.float64)
    rng = np.random.default_rng(seed)
    k = rng.integers(0, roots.size, n)
    obj = tris.reshape(-1, 3, 3).astype(np.float64)
    c = np.einsum("nij,nj->ni", m[k, :, :3], obj[offs[roots[k]].astype(np.int64)].mean(axis=1)) + m[k, :, 3]
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.zeros(n, ob.RAY_DTYPE)
    rays["o"] = (c - d * 3.0).astype(np.float32); rays["d"] = d.astype(np.float32); rays["tmax"] = F32_MAX
    rays["d"][: n // 10, 1:] = 0; rays["d"][: n // 10, 0] = 1                 # zero components
    return rays


@gpu
@pytest.mark.parametrize("stride", [24, 48, 64])
@pytest.mark.parametrize("kind", ["identity", "translation", "rotation", "uniform", "nonuniform", "mirror", "shear", "large", "mixed"])
def test_instanced_scenes(kind, stride):
    sc, tris, offs, roots, xf = placed(kind, stride)
    try:
        rays = rays_at_instances(tris, offs, roots, xf, 6000, seed=3)
        for any_hit in (False, True):
            hits, _ = check_batch(sc, rays, any_hit, ids_of=True)
            if kind != "large":
                assert (hits["prim"] != INVALID).sum() > 2000
        with pytest.raises(ValueError):                                 # an instanced scene needs the instance ids
            sc.hit_attributes(rays, hits)
        L = cuda.lib()
        out = np.zeros(rays.size, cuda.ATTR_DTYPE)
        assert L.tray_cuda_hit_attributes(sc._h, rays.ctypes.data, hits.ctypes.data, None, rays.size, out.ctypes.data, None) == -1
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("kind", ["mixed", "mirror", "shear"])
def test_instanced_normal_is_the_world_normal(kind):
    """the world-space Ng of an instanced hit points along the normal of the world-space triangle (in double), with the sign of
    det(object_to_world): Wᵀ n = det(M)⁻¹ cof(M) n"""
    sc, tris, offs, roots, xf = placed(kind, 48, n_obj=20, n_inst=60, seed=21)
    try:
        rays = rays_at_instances(tris, offs, roots, xf, 4000, seed=22)
        hits, ids = sc.traverse_instance(rays)
        hit = hits["prim"] != INVALID
        assert hit.sum() > 1000
        a = sc.hit_attributes(rays, hits, ids)[hit]
        rec = sc.download_bvh(prim_indices=False)[1]
        v = vertices(rec, 48, hits["prim"][hit])
        m = xf.astype(np.float64)[ids[hit]]
        w = [np.einsum("nij,nj->ni", m[:, :, :3], x) + m[:, :, 3] for x in v]
        nw = np.cross(w[0] - w[1], w[2] - w[0]) * np.sign(np.linalg.det(m[:, :, :3]))[:, None]
        ng = a["ng"].astype(np.float64)
        cos = (ng * nw).sum(1) / (np.linalg.norm(ng, axis=1) * np.linalg.norm(nw, axis=1))
        assert (cos > 1 - 1e-5).all(), float(cos.min())
    finally:
        sc.close()


@gpu
def test_miss_records_and_out_of_range_hits():
    sc, tris, offs, roots, xf = placed("mixed", 48, n_inst=50)
    flat = cuda.TrayCudaScene.build(tris)
    try:
        rays = rays_at_instances(tris, offs, roots, xf, 1000, seed=9)
        hits, ids = sc.traverse_instance(rays)
        n_tris = sc.info()["n_tris"]
        h, i = hits.copy(), ids.copy()
        h["prim"][:100] = INVALID
        h["prim"][100:200] = n_tris
        h["prim"][200:300] = 0xFFFFFFF0
        i[300:400] = INVALID
        i[400:500] = 50
        got = sc.hit_attributes(rays, h, i)
        assert is_miss(got[:500]).all()
        assert same_bytes(got[500:], sc.hit_attributes(rays[500:], hits[500:], ids[500:]))
        assert same_bytes(device_attrs(sc, rays, h, i), got)
        fh = flat.traverse(rays)
        fh["prim"][:100] = flat.info()["n_tris"] + np.arange(100, dtype=np.uint32)
        fa = flat.hit_attributes(rays, fh)
        assert is_miss(fa[:100]).all() and is_miss(fa[fh["prim"] == INVALID]).all()
        assert (~is_miss(fa[100:][fh["prim"][100:] != INVALID])).all()
        assert same_hits_after(sc, rays, hits, ids)                       # the device is fine afterwards
        assert flat.hit_attributes(rays[:0], fh[:0]).size == 0
    finally:
        sc.close()
        flat.close()


def same_hits_after(sc, rays, hits, ids):
    h2, i2 = sc.traverse_instance(rays)
    return np.array_equal(words(h2), words(hits)) and np.array_equal(i2, ids)


@gpu
def test_device_form_on_a_caller_stream_follows_the_scene_stream():
    """hits of a trace_device on the scene stream are complete when the attribute pass runs on another stream"""
    import torch
    packed, tris, _ = golden_scene("cornell_box", 48)
    sc = cuda.TrayCudaScene.from_packed(packed)
    try:
        rays = mixed_rays(tris, 1 << 16, seed=31)
        d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
        d_hits = torch.full((rays.size * 8,), 0xFF, dtype=torch.uint8, device="cuda")
        d_out = torch.zeros(rays.size * 20, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        sc.traverse_device(d_rays.data_ptr(), rays.size, d_hits.data_ptr())
        sc.hit_attributes_device(d_rays.data_ptr(), d_hits.data_ptr(), None, rays.size, d_out.data_ptr(), stream=side.cuda_stream)
        side.synchronize()
        hits = d_hits.cpu().numpy().view(ob.HIT_DTYPE)
        want, _ = reference(sc.download_bvh(prim_indices=False)[1], 48, rays, hits)
        assert same_bytes(d_out.cpu().numpy().view(cuda.ATTR_DTYPE), want)
    finally:
        sc.close()


# ---- GPU: frames -----------------------------------------------------------------------------------------------------------


def frame_expectation(sc, view, w, h, shard, shards, instanced):
    """(primary, bounce) attributes of the last frame from hit_attributes over its own rays, hits and instances"""
    got = sc.download(primary=True, bounce=True, bounce_rays=True)
    ids = sc.download_instance(primary=True, bounce=True) if instanced else {"primary": None, "bounce": None}
    own = cuda.shard_mask(w, h, shard, shards)
    prays = ob.primary_rays(view, w, h)
    shoot = own & (got["primary"]["t"] < F32_MAX)
    out = {}
    for name, rays, mask in (("primary", prays, own), ("bounce", got["bounce_rays"], shoot)):
        want = np.frombuffer(b"\xff" * (20 * w * h), dtype=cuda.ATTR_DTYPE).copy()
        i = None if ids[name] is None else ids[name][mask]
        want[mask] = sc.hit_attributes(rays[mask], got[name][mask], i)
        out[name] = want
    return out, got, own


def frame_state(sc, instanced):
    got = sc.download(primary=True, bounce=True, rgba=True)
    ids = sc.download_instance(primary=True, bounce=True) if instanced else {}
    return [got["primary"], got["bounce"], got["rgba"]] + list(ids.values())


def check_frames(sc, view, w, h, instanced, in_flight):
    sc.set_frames_in_flight(in_flight)
    flags = cuda.RENDER_BOUNCE | cuda.RENDER_RGBA | cuda.RENDER_KEEP_RAYS
    runs = [(flags, 0, 1), (flags | cuda.RENDER_OVERLAP, 0, 1), (flags | cuda.RENDER_ANYHIT_AO, 0, 1), (flags, 1, 2), (flags, 2, 3)]
    for f, shard, shards in runs:
        sc.render(view, w, h, 0, f, shard=shard, shards=shards)
        sc.sync()
        before = frame_state(sc, instanced)
        got = sc.download_attributes(primary=True, bounce=True)
        want, hits, own = frame_expectation(sc, view, w, h, shard, shards, instanced)
        for name in ("primary", "bounce"):
            assert same_bytes(got[name], want[name]), (name, f, shard, int((words(got[name]) != words(want[name])).any(axis=1).sum()))
        hit = own & (hits["primary"]["prim"] != INVALID)                   # (other shards' pixels download as zeros)
        assert (~is_miss(got["primary"][hit])).all() and hit.sum() > 1000
        assert is_miss(got["primary"][~own]).all() and is_miss(got["bounce"][~own]).all()
        after = frame_state(sc, instanced)
        assert all(np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)) for a, b in zip(before, after))


@gpu
@pytest.mark.parametrize("in_flight", [1, 2, 3])
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_frames_of_flat_and_two_level_scenes(cornell, stride, in_flight):
    w, h = 200, 120
    view = host.view_from_camera(cornell.camera, w, h)
    tris = cornell.tris().reshape(-1, 3, 3)
    for sc in (cuda.TrayCudaScene.from_packed(host.PackedScene(cornell, tri_stride=stride)),
               cuda.TrayCudaScene.build(tris, tri_stride=stride, object_offsets=cornell.object_offsets())):
        try:
            check_frames(sc, view, w, h, False, in_flight)
        finally:
            sc.close()


@gpu
@pytest.mark.parametrize("in_flight", [1, 2, 3])
@pytest.mark.parametrize("stride", [24, 48, 64])
def test_frames_of_instanced_scenes(cornell, stride, in_flight):
    sc, *_ = cornell_instances(cornell, stride)
    try:
        w, h = 200, 120
        check_frames(sc, host.view_from_camera(cornell.camera, w, h), w, h, True, in_flight)
    finally:
        sc.close()


@gpu
def test_frame_of_2_26_items(cornell):
    """8192 x 8192 pixels: 2^26 items, whose attribute staging (64 B per item) is 4 GiB, past 32-bit sizes; a sample of its
    pixels has the attributes of hit_attributes over the frame's own rays and hits"""
    w = h = 8192
    assert cuda.local_items(w, h) == 1 << 26
    view = host.view_from_camera(cornell.camera, w, h)
    sc = cuda.TrayCudaScene.from_packed(host.PackedScene(cornell))
    try:
        sc.render(view, w, h, 0, cuda.RENDER_BOUNCE | cuda.RENDER_KEEP_RAYS)
        sc.sync()
        got = sc.download_attributes(primary=True, bounce=True)
        frame = sc.download(primary=True, bounce=True, bounce_rays=True)
        pick = np.sort(np.random.default_rng(5).choice(w * h, 1 << 20, replace=False))
        shoot = frame["primary"]["t"][pick] < F32_MAX
        assert shoot.sum() > 100000
        want_b = np.frombuffer(b"\xff" * (20 * pick.size), dtype=cuda.ATTR_DTYPE).copy()
        want_b[shoot] = sc.hit_attributes(frame["bounce_rays"][pick][shoot], frame["bounce"][pick][shoot])
        assert same_bytes(got["bounce"][pick], want_b)
        prays = ob.primary_rays(view, w, h)[pick]
        assert same_bytes(got["primary"][pick], sc.hit_attributes(prays, frame["primary"][pick]))
    finally:
        sc.close()


def refused_without_writing(sc, n):
    L = cuda.lib()
    p = np.full(n * 5, 0x12345678, np.uint32)
    b = p.copy()
    rc = L.tray_cuda_frame_download_attributes(sc._h, p.ctypes.data, b.ctypes.data)
    return rc == -1 and (p == 0x12345678).all() and (b == 0x12345678).all()


@gpu
def test_frame_refusals(cornell):
    w, h = 64, 48
    view = host.view_from_camera(cornell.camera, w, h)
    tris = cornell.tris().reshape(-1, 3, 3)
    offs = cornell.object_offsets()
    sc = cuda.TrayCudaScene.build(tris, object_offsets=offs)
    flat = cuda.TrayCudaScene.build(tris)
    try:
        assert refused_without_writing(sc, w * h)                            # no frame yet
        sc.render(view, w, h, 0, cuda.RENDER_RGBA)
        sc.sync()
        sc.download_attributes(primary=True)
        with pytest.raises(cuda.TrayCudaError):
            sc.download_attributes(primary=True, bounce=True)                # no bounce in that frame
        flags = cuda.RENDER_BOUNCE
        # each change of the geometry refuses the frame before it; the next frame is fine
        for change in (lambda: sc.refit(host.jitter(tris, 1, frac=0.01)),
                       lambda: sc.refit_rebuild_tlas(host.jitter(tris, 2, frac=0.01)),
                       lambda: sc.set_instances(sc.download_instances(), np.tile(np.eye(3, 4, dtype=np.float32), (offs.size - 1, 1, 1))),
                       lambda: sc.refit_rebuild_tlas(host.jitter(tris, 3, frac=0.01))):
            sc.render(view, w, h, 0, flags)
            sc.sync()
            sc.download_attributes(primary=True, bounce=True)
            change()
            assert refused_without_writing(sc, w * h)
            with pytest.raises(cuda.TrayCudaError):
                sc.download_attributes(primary=True)
        sc.render(view, w, h, 0, flags)
        sc.sync()
        sc.download_attributes(primary=True, bounce=True)
        # a refused change leaves the frame valid
        with pytest.raises(cuda.TrayCudaError):
            sc.refit(tris)                                                     # refused on an instanced scene
        sc.download_attributes(primary=True, bounce=True)
        # set_variant on a flat scene
        flat.render(view, w, h, 0, flags)
        flat.sync()
        flat.download_attributes(primary=True, bounce=True)
        flat.set_variant(cuda.VARIANT_ZERODIR_BOX_ONLY)
        assert refused_without_writing(flat, w * h)
        flat.render(view, w, h, 0, flags)
        flat.sync()
        a = flat.download_attributes(primary=True, bounce=True)
        assert (~is_miss(a["primary"])).sum() > 1000
    finally:
        sc.close()
        flat.close()
