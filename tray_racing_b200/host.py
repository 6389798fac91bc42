"""ctypes binding of libtray_host.so (include/tray_host.h): meshes, the CWBVH producer, the
`cwbvh_gpu_runner` marshalling (reference src/rt_gpu/mod.rs:16-112) and the camera uniform
(reference src/main.rs:589-617).  CPU only — nothing here is on the timed path."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libtray_host.so")

NODE_BYTES = 80
RAY_DTYPE = np.dtype([("o", "<f4", 3), ("tmin", "<f4"), ("d", "<f4", 3), ("tmax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("prim", "<u4")])
INVALID_PRIM = 0xFFFFFFFF
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 8


class TrayView(C.Structure):
    """`ViewUniform` (reference src/main.rs:589-597), 160 bytes."""
    _fields_ = [("view_inv", C.c_float * 16), ("proj_inv", C.c_float * 16), ("eye", C.c_float * 3),
                ("exposure", C.c_float), ("tlas_start", C.c_uint32), ("pad", C.c_uint32 * 3)]


assert C.sizeof(TrayView) == 160


class ValidateReport(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "nodes_reached", "nodes_unreached", "prims_reached", "prims_missing", "prim_seen_twice",
        "node_visited_twice", "bad_child_index", "bad_prim_index", "bad_meta", "bad_quant",
        "box_violations", "children_total", "leaf_children")] + [
        ("max_depth", C.c_uint32), ("max_stack", C.c_uint32), ("stack_too_deep", C.c_uint32), ("pad", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "pad"}


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(_LIB_PATH)
        vp, u64, u32, i32, f32p = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(C.c_float)
        sig = {
            "tray_host_build_cwbvh_from_tris": (i32, [vp, u64, u32, i32, C.POINTER(vp)]),
            "tray_host_build_cwbvh_from_aabbs": (i32, [vp, vp, u64, u32, i32, C.POINTER(vp)]),
            "tray_host_cwbvh_node_count": (u64, [vp]), "tray_host_cwbvh_prim_count": (u64, [vp]),
            "tray_host_cwbvh_max_depth": (u32, [vp]), "tray_host_cwbvh_nodes": (vp, [vp]),
            "tray_host_cwbvh_prim_indices": (vp, [vp]), "tray_host_cwbvh_aabb": (None, [vp, f32p, f32p]),
            "tray_host_cwbvh_free": (None, [vp]),
            "tray_host_cwbvh_validate": (i32, [vp, u64, vp, u64, vp, vp, u32, C.POINTER(ValidateReport)]),
            "tray_host_mesh_load_obj": (i32, [C.c_char_p, C.POINTER(vp)]),
            "tray_host_mesh_from_tris": (i32, [vp, u64, vp, u32, C.POINTER(vp)]),
            "tray_host_mesh_generate": (i32, [C.c_char_p, u64, C.c_double, C.POINTER(vp)]),
            "tray_host_mesh_tri_count": (u64, [vp]), "tray_host_mesh_object_count": (u32, [vp]),
            "tray_host_mesh_tris": (vp, [vp]), "tray_host_mesh_object_offsets": (vp, [vp]),
            "tray_host_mesh_camera": (None, [vp, f32p, f32p, f32p]), "tray_host_mesh_free": (None, [vp]),
            "tray_host_pack": (i32, [vp, i32, u32, u32, i32, C.POINTER(vp)]),
            "tray_host_packed_bvh_bytes": (vp, [vp, C.POINTER(u64)]),
            "tray_host_packed_tri_bytes": (vp, [vp, C.POINTER(u64)]),
            "tray_host_packed_instance_bytes": (vp, [vp, C.POINTER(u64)]),
            "tray_host_packed_prim_to_mesh_tri": (vp, [vp, C.POINTER(u64)]),
            "tray_host_packed_blas_tri_offsets": (vp, [vp, C.POINTER(u32)]),
            "tray_host_packed_tlas_start": (u32, [vp]), "tray_host_packed_max_depth": (u32, [vp]),
            "tray_host_packed_build_seconds": (C.c_double, [vp, C.POINTER(C.c_double)]),
            "tray_host_packed_free": (None, [vp]),
            "tray_host_view_from_camera": (None, [f32p, f32p, C.c_float, C.c_float, C.c_float, C.c_float, u32, C.POINTER(TrayView)]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _np_from(ptr, nbytes, dtype):
    if nbytes == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_uint8 * nbytes).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype).copy()


@dataclass
class Camera:
    """reference `Camera` (src/main.rs:619-625)"""
    eye: tuple
    look_at: tuple
    fov: float
    exposure: float = 0.0


class Mesh:
    """`Vec<Vec<Triangle>>` as produced by `load_meshs` (reference src/main.rs:493-561)."""

    def __init__(self, handle, camera: Camera | None = None):
        self._h = C.c_void_p(handle)
        self.camera = camera

    @classmethod
    def load_obj(cls, path: str, camera: Camera | None = None) -> "Mesh":
        h = C.c_void_p()
        if lib().tray_host_mesh_load_obj(path.encode(), C.byref(h)) != 0:
            raise RuntimeError(f"Error while loading obj file {path!r}")
        return cls(h.value, camera)

    @classmethod
    def generate(cls, name: str, seed: int = 1, size: float = 1.0) -> "Mesh":
        h = C.c_void_p()
        if lib().tray_host_mesh_generate(name.encode(), seed, float(size), C.byref(h)) != 0:
            raise ValueError(f"unknown synthetic scene {name!r} or bad size {size}")
        m = cls(h.value)
        eye, look, fov = (C.c_float * 3)(), (C.c_float * 3)(), C.c_float()
        lib().tray_host_mesh_camera(m._h, eye, look, C.byref(fov))
        m.camera = Camera(tuple(eye), tuple(look), fov.value)
        return m

    @classmethod
    def from_tris(cls, tris: np.ndarray, object_offsets=None, camera: Camera | None = None) -> "Mesh":
        t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
        h = C.c_void_p()
        if object_offsets is None:
            rc = lib().tray_host_mesh_from_tris(t.ctypes.data, t.shape[0], None, 0, C.byref(h))
        else:
            off = np.ascontiguousarray(object_offsets, dtype=np.uint64)
            rc = lib().tray_host_mesh_from_tris(t.ctypes.data, t.shape[0], off.ctypes.data, len(off) - 1, C.byref(h))
        if rc != 0:
            raise ValueError("bad triangle / object_offsets arrays")
        return cls(h.value, camera)

    @property
    def n_tris(self) -> int:
        return lib().tray_host_mesh_tri_count(self._h)

    @property
    def n_objects(self) -> int:
        return lib().tray_host_mesh_object_count(self._h)

    def tris(self) -> np.ndarray:
        n = self.n_tris
        return _np_from(lib().tray_host_mesh_tris(self._h), n * 36, np.float32).reshape(n, 9)

    def object_offsets(self) -> np.ndarray:
        return _np_from(lib().tray_host_mesh_object_offsets(self._h), (self.n_objects + 1) * 8, np.uint64)

    def __del__(self):
        if getattr(self, "_h", None) is not None and self._h.value and _lib is not None:
            _lib.tray_host_mesh_free(self._h)
            self._h = None


class PackedScene:
    """The three byte buffers + tlas_start that `cwbvh_gpu_runner` hands to `start`
    (reference src/rt_gpu/mod.rs:92-100,108-110)."""

    def __init__(self, mesh: Mesh, use_tlas: bool = False, tri_stride: int = 48, max_prims_per_leaf: int = 3, nthreads: int = 0):
        h = C.c_void_p()
        rc = lib().tray_host_pack(mesh._h, int(use_tlas), tri_stride, max_prims_per_leaf, nthreads, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"tray_host_pack failed ({rc})")
        L = lib()
        n = C.c_uint64()
        p = L.tray_host_packed_bvh_bytes(h, C.byref(n))
        self.bvh_bytes = _np_from(p, n.value, np.uint8)
        p = L.tray_host_packed_tri_bytes(h, C.byref(n))
        self.tri_bytes = _np_from(p, n.value, np.uint8)
        p = L.tray_host_packed_instance_bytes(h, C.byref(n))
        self.instance_bytes = _np_from(p, n.value, np.uint8)
        p = L.tray_host_packed_prim_to_mesh_tri(h, C.byref(n))
        self.prim_to_mesh_tri = _np_from(p, n.value * 4, np.uint32)
        nb = C.c_uint32()
        p = L.tray_host_packed_blas_tri_offsets(h, C.byref(nb))
        self.blas_tri_offsets = _np_from(p, (nb.value + 1) * 8, np.uint64)
        self.tlas_start = L.tray_host_packed_tlas_start(h)
        self.max_depth = L.tray_host_packed_max_depth(h)
        ts = C.c_double()
        self.build_seconds = L.tray_host_packed_build_seconds(h, C.byref(ts))
        self.tlas_build_seconds = ts.value
        L.tray_host_packed_free(h)
        self.use_tlas = bool(use_tlas)
        self.tri_stride = tri_stride
        self.camera = mesh.camera

    @property
    def n_nodes(self) -> int:
        return self.bvh_bytes.size // NODE_BYTES

    @property
    def n_tris(self) -> int:
        return self.tri_bytes.size // self.tri_stride

    @property
    def blas_offsets(self) -> np.ndarray:
        return self.instance_bytes.view(np.uint32)

    @property
    def n_instances(self) -> int:
        return self.blas_offsets.size if self.use_tlas else 0

    def working_set_bytes(self) -> int:
        return int(self.bvh_bytes.size + self.tri_bytes.size)

    def geometry_of(self, prim: np.ndarray):
        """global BVH-ordered prim -> (geometry_id, primitive_id) as the CPU path reports them
        (reference src/cwbvh.rs:150-160)."""
        prim = np.asarray(prim, dtype=np.uint64)
        geom = np.searchsorted(self.blas_tri_offsets, prim, side="right") - 1
        return geom.astype(np.uint32), (prim - self.blas_tri_offsets[geom]).astype(np.uint32)


def build_cwbvh(tris: np.ndarray, max_prims_per_leaf: int = 3, nthreads: int = 0):
    """`cwbvh_from_tris` (reference src/cwbvh.rs:24-105) -> (nodes[n,80] u8, primitive_indices u32, max_depth)."""
    t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
    h = C.c_void_p()
    if lib().tray_host_build_cwbvh_from_tris(t.ctypes.data, t.shape[0], max_prims_per_leaf, nthreads, C.byref(h)) != 0:
        raise RuntimeError("CWBVH build failed")
    L = lib()
    nn, npr = L.tray_host_cwbvh_node_count(h), L.tray_host_cwbvh_prim_count(h)
    nodes = _np_from(L.tray_host_cwbvh_nodes(h), nn * NODE_BYTES, np.uint8).reshape(nn, NODE_BYTES)
    pidx = _np_from(L.tray_host_cwbvh_prim_indices(h), npr * 4, np.uint32)
    depth = L.tray_host_cwbvh_max_depth(h)
    L.tray_host_cwbvh_free(h)
    return nodes, pidx, depth


def validate_cwbvh(nodes: np.ndarray, prim_indices, prim_min: np.ndarray, prim_max: np.ndarray, stack_limit: int = 32):
    nodes = np.ascontiguousarray(nodes, dtype=np.uint8).reshape(-1, NODE_BYTES)
    pmin = np.ascontiguousarray(prim_min, dtype=np.float32)
    pmax = np.ascontiguousarray(prim_max, dtype=np.float32)
    pi = None if prim_indices is None else np.ascontiguousarray(prim_indices, dtype=np.uint32)
    rep = ValidateReport()
    rc = lib().tray_host_cwbvh_validate(nodes.ctypes.data, nodes.shape[0], None if pi is None else pi.ctypes.data,
                                        pmin.shape[0], pmin.ctypes.data, pmax.ctypes.data, stack_limit, C.byref(rep))
    return rc, rep.as_dict()


def view_from_camera(cam: Camera, width: int, height: int, tlas_start: int = 0) -> TrayView:
    """`ViewUniform::from_camera` (reference src/main.rs:599-616)."""
    v = TrayView()
    eye = (C.c_float * 3)(*cam.eye)
    look = (C.c_float * 3)(*cam.look_at)
    lib().tray_host_view_from_camera(eye, look, cam.fov, float(width), float(height), cam.exposure, tlas_start, C.byref(v))
    return v


def tri_records(tris: np.ndarray, stride: int = 48) -> np.ndarray:
    """`RtTriangle::from(&Triangle)`: {v0, e1 = v0 - v1, e2 = v2 - v0 [, ng]} as padded f32 records; stride 24 is the wgpu
    path's `RtCompressedTriangle` {v0: f32 x 3, e[k] = half(v2 - v0)[k] | half(v1 - v0)[k] << 16}
    (reference src/rt_gpu/mod.rs:39-43)."""
    t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 3, 3)
    if stride == 24:
        rec = np.zeros((t.shape[0], 6), dtype=np.uint32)
        rec[:, 0:3] = t[:, 0].view(np.uint32)
        with np.errstate(over="ignore"):
            lo = (t[:, 2] - t[:, 0]).astype(np.float16).view(np.uint16).astype(np.uint32)
            hi = (t[:, 1] - t[:, 0]).astype(np.float16).view(np.uint16).astype(np.uint32)
        rec[:, 3:6] = lo | (hi << 16)
        return rec.view(np.uint8).reshape(-1)
    rec = np.zeros((t.shape[0], stride // 4), dtype=np.float32)
    rec[:, 0:3] = t[:, 0]
    rec[:, 4:7] = t[:, 0] - t[:, 1]
    rec[:, 8:11] = t[:, 2] - t[:, 0]
    if stride == 64:
        e1, e2 = rec[:, 4:7], rec[:, 8:11]
        rec[:, 12] = e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1]
        rec[:, 13] = e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2]
        rec[:, 14] = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
    return rec.view(np.uint8).reshape(-1)


def jitter(tris: np.ndarray, seed: int, frac: float = 0.01) -> np.ndarray:
    """(n, 3, 3) float32: every vertex moved by up to `frac` of the mean triangle size (a small deformation, as a skinned or
    simulated mesh moves between two frames)"""
    t = np.asarray(tris, np.float32).reshape(-1, 3, 3)
    size = float(np.mean(np.linalg.norm(t.max(axis=1) - t.min(axis=1), axis=1)))
    rng = np.random.default_rng(seed)
    return (t + rng.uniform(-frac * size, frac * size, t.shape).astype(np.float32)).astype(np.float32)


def rigid(tris: np.ndarray, object_offsets, seed: int, frac: float = 0.05) -> np.ndarray:
    """(n, 3, 3) float32: object k (triangles object_offsets[k] .. [k + 1]) translated as a whole by up to `frac` of the scene's
    extent"""
    t = np.asarray(tris, np.float32).reshape(-1, 3, 3)
    offs = np.asarray(object_offsets, np.int64)
    ext = float((t.reshape(-1, 3).max(axis=0) - t.reshape(-1, 3).min(axis=0)).max())
    rng = np.random.default_rng(seed)
    shift = rng.uniform(-frac * ext, frac * ext, (offs.size - 1, 3)).astype(np.float32)
    return (t + np.repeat(shift, np.diff(offs), axis=0)[:, None, :]).astype(np.float32)
