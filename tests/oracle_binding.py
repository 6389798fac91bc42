"""ctypes binding of oracle/libtray_oracle.so.  TEST INFRASTRUCTURE: importable only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs — never from the package."""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import subprocess

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_ORACLE_DIR = os.path.join(_ROOT, "oracle")
_LIB_PATH = os.path.join(_ORACLE_DIR, "libtray_oracle.so")

RAY_DTYPE = np.dtype([("o", "<f4", 3), ("tmin", "<f4"), ("d", "<f4", 3), ("tmax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("prim", "<u4")])
COUNT_DTYPE = np.dtype([("nodes", "<u4"), ("tris", "<u4"), ("insts", "<u4")])
INVALID_PRIM = 0xFFFFFFFF
VARIANT_BOX_DIVIDE = 1
VARIANT_TIE_LAST = 2
VARIANT_BOX_TMIN_RAY = 4
VARIANT_ZERODIR_BOX_ONLY = 8
RENDER_BOUNCE = 1
RENDER_RGBA = 2
STACK_DEFAULT = 32          # obvhs' traversal stack (cwbvh.rs:88)
STACK_MAX = 64              # ORC_STACK_MAX


class OrcView(C.Structure):
    _fields_ = [("view_inv", C.c_float * 16), ("proj_inv", C.c_float * 16), ("eye", C.c_float * 3),
                ("exposure", C.c_float), ("tlas_start", C.c_uint32), ("pad", C.c_uint32 * 3)]


class OrcScene(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("n_nodes", C.c_uint64), ("tris", C.c_void_p), ("n_tris", C.c_uint64),
                ("tri_stride", C.c_uint32), ("blas_offsets", C.c_void_p), ("n_instances", C.c_uint32),
                ("tlas_start", C.c_uint32), ("use_tlas", C.c_int)]


class OrcTotals(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "nodes", "tris", "insts", "hits")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class OrcBuildParams(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("max_leaf", "radius", "passes", "visits", "rounds")]


class OrcBuildStats(C.Structure):
    _fields_ = [("n_nodes", C.c_uint64), ("ploc_iterations", C.c_uint32), ("levels", C.c_uint32),
                ("reinsert_passes", C.c_uint32), ("reinsert_moves", C.c_uint32), ("sah_before", C.c_double), ("sah_after", C.c_double)]


class OrcBuildResult(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("n_nodes", C.c_uint64), ("prim_indices", C.c_void_p), ("n_prims", C.c_uint64),
                ("blas_offsets", C.c_void_p), ("n_instances", C.c_uint32), ("tlas_start", C.c_uint32), ("force_exact", C.c_int),
                ("stats", OrcBuildStats), ("bvh2", C.c_void_p), ("n_bvh2", C.c_uint32), ("n_bvh2_leaves", C.c_uint32)]


# orc_bvh2_node: leaf left = -1, right = primitive; parent = -1 at a root
BVH2_DTYPE = np.dtype([("lo", "<f4", 3), ("hi", "<f4", 3), ("left", "<i4"), ("right", "<i4"), ("count", "<u4"), ("parent", "<i4")])
assert BVH2_DTYPE.itemsize == 40


_lib = None


def build():
    subprocess.check_call(["make", "-s", "-C", _ORACLE_DIR])


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
        L.orc_set_variant.argtypes = [u32]
        L.orc_set_stack_limit.restype = i32
        L.orc_set_stack_limit.argtypes = [u32]
        L.orc_stack_limit.restype = u32
        L.orc_stack_need.restype = i32
        L.orc_stack_need.argtypes = [C.POINTER(OrcScene), vp, u64, vp, i32, i32]
        L.orc_max_threads.restype = i32
        L.orc_set_simd.argtypes = [i32]
        L.orc_simd.restype = i32
        L.orc_trace.restype = i32
        L.orc_trace.argtypes = [C.POINTER(OrcScene), vp, u64, vp, vp, C.POINTER(OrcTotals), i32]
        L.orc_trace_any.restype = i32
        L.orc_trace_any.argtypes = [C.POINTER(OrcScene), vp, u64, vp, vp, C.POINTER(OrcTotals), i32]
        L.orc_brute_force.restype = i32
        L.orc_brute_force.argtypes = [C.POINTER(OrcScene), vp, u64, vp, vp, i32]
        L.orc_intersect_tri.restype = C.c_float
        L.orc_intersect_tri.argtypes = [C.POINTER(OrcScene), u32, vp]
        L.orc_half_to_float.restype = C.c_float
        L.orc_half_to_float.argtypes = [C.c_uint16]
        L.orc_primary_rays.argtypes = [C.POINTER(OrcView), u32, u32, vp, i32]
        L.orc_render.restype = i32
        L.orc_render.argtypes = [C.POINTER(OrcScene), C.POINTER(OrcView), u32, u32, u32, u32, vp, vp, vp, vp,
                                 C.POINTER(OrcTotals), C.POINTER(OrcTotals), i32]
        L.orc_uhash.restype = u32
        L.orc_uhash.argtypes = [u32, u32]
        L.orc_hash_noise.restype = C.c_float
        L.orc_hash_noise.argtypes = [u32, u32, u32]
        L.orc_sincos_tau.argtypes = [C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.orc_node_intersect.restype = u32
        L.orc_node_intersect.argtypes = [vp, vp, C.c_float]
        L.orc_build_ref.restype = i32
        L.orc_build_ref.argtypes = [vp, u64, vp, u32, C.POINTER(OrcBuildParams), C.POINTER(OrcBuildResult)]
        L.orc_build_free.argtypes = [C.POINTER(OrcBuildResult)]
        _lib = L
    return _lib


@contextlib.contextmanager
def _stack_limit(entries):
    """the oracle's stack capacity for the calls inside the block (1 .. STACK_MAX), the default again after it"""
    if lib().orc_set_stack_limit(int(entries)) != 0:
        raise ValueError(f"stack_limit must be 1 .. {STACK_MAX} (got {entries})")
    try:
        yield
    finally:
        lib().orc_set_stack_limit(STACK_DEFAULT)


def _view(view) -> OrcView:
    v = OrcView()
    C.memmove(C.byref(v), C.byref(view), C.sizeof(OrcView))
    return v


class Oracle:
    """CPU restatement of CwBvhScene / CwBvhTlasScene (reference src/cwbvh.rs:139-193) over raw byte buffers."""

    def __init__(self, bvh_bytes, tri_bytes, tri_stride=48, blas_offsets=None, tlas_start=0, use_tlas=False):
        self.nodes = np.ascontiguousarray(bvh_bytes, dtype=np.uint8).reshape(-1)
        self.tris = np.ascontiguousarray(tri_bytes, dtype=np.uint8).reshape(-1)
        self.blas = None if blas_offsets is None else np.ascontiguousarray(blas_offsets, dtype=np.uint32)
        s = OrcScene()
        s.nodes, s.n_nodes = self.nodes.ctypes.data, self.nodes.size // 80
        s.tris, s.n_tris, s.tri_stride = self.tris.ctypes.data, self.tris.size // tri_stride, tri_stride
        s.blas_offsets = None if self.blas is None else self.blas.ctypes.data
        s.n_instances = 0 if self.blas is None else self.blas.size
        s.tlas_start, s.use_tlas = tlas_start, int(use_tlas)
        self.scene = s

    @classmethod
    def from_packed(cls, p) -> "Oracle":
        return cls(p.bvh_bytes, p.tri_bytes, p.tri_stride, p.blas_offsets if p.use_tlas else None, p.tlas_start, p.use_tlas)

    def trace(self, rays, counts=False, nthreads=0, any_hit=False, stack_limit=STACK_DEFAULT):
        """closest hit per ray; any_hit=True stops each ray at the first accepted triangle (orc_trace_any).
        Raises when a ray needs more than `stack_limit` stack entries (obvhs' 32 by default; the kernels hold 48)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        cnt = np.empty(rays.shape[0], dtype=COUNT_DTYPE) if counts else None
        tot = OrcTotals()
        fn = lib().orc_trace_any if any_hit else lib().orc_trace
        with _stack_limit(stack_limit):
            rc = fn(C.byref(self.scene), rays.ctypes.data, rays.shape[0], hits.ctypes.data,
                    None if cnt is None else cnt.ctypes.data, C.byref(tot), nthreads)
        if rc != 0:
            raise RuntimeError(f"oracle traversal stack overflow ({rc})")
        return (hits, cnt, tot.as_dict()) if counts else hits

    def stack_need(self, rays, any_hit=False, nthreads=0) -> np.ndarray:
        """per ray, the most stack entries its traversal holds at once (node groups, and the two pushes of a TLAS instance
        entry), whatever the stack capacity; raises when a ray needs more than STACK_MAX"""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        need = np.empty(rays.shape[0], dtype=np.uint32)
        rc = lib().orc_stack_need(C.byref(self.scene), rays.ctypes.data, rays.shape[0], need.ctypes.data, int(any_hit), nthreads)
        if rc != 0:
            raise RuntimeError(f"a ray needs more than {STACK_MAX} stack entries ({rc})")
        return need

    def brute_force(self, rays, nthreads=0):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        ties = np.empty(rays.shape[0], dtype=np.uint32)
        lib().orc_brute_force(C.byref(self.scene), rays.ctypes.data, rays.shape[0], hits.ctypes.data, ties.ctypes.data, nthreads)
        return hits, ties

    def intersect_tri(self, prim, ray) -> float:
        r = np.ascontiguousarray(ray, dtype=RAY_DTYPE).reshape(1)
        return lib().orc_intersect_tri(C.byref(self.scene), int(prim), r.ctypes.data)

    def render(self, view, w, h, frame_count=0, flags=RENDER_BOUNCE, nthreads=0, rgba=False, stack_limit=STACK_DEFAULT):
        n = w * h
        primary = np.empty(n, dtype=HIT_DTYPE)
        bounce = np.empty(n, dtype=HIT_DTYPE)
        brays = np.empty(n, dtype=RAY_DTYPE)
        img = np.zeros((n, 4), dtype=np.uint8) if rgba else None
        pt, bt = OrcTotals(), OrcTotals()
        v = _view(view)
        with _stack_limit(stack_limit):
            rc = lib().orc_render(C.byref(self.scene), C.byref(v), w, h, frame_count, flags | (RENDER_RGBA if rgba else 0),
                                  primary.ctypes.data, bounce.ctypes.data, brays.ctypes.data,
                                  None if img is None else img.ctypes.data, C.byref(pt), C.byref(bt), nthreads)
        if rc != 0:
            raise RuntimeError(f"oracle traversal stack overflow ({rc})")
        return dict(primary=primary, bounce=bounce, bounce_rays=brays, rgba=img, primary_totals=pt.as_dict(), bounce_totals=bt.as_dict())


def _copy(ptr, count, dtype):
    if not count or not ptr:
        return np.zeros(0, dtype=dtype)
    n = count * np.dtype(dtype).itemsize
    return np.frombuffer((C.c_uint8 * n).from_address(ptr), dtype=dtype).copy()


def build_reference(tris, tri_stride=48, max_leaf=3, radius=14, object_offsets=None, passes=4, visits=192, rounds=3, bvh2=False):
    """The serial reference of the device builder (oracle/build_ref.c), shaped like what a device-built TrayCudaScene reports:
    nodes / tri_bytes / prim_indices as download_bvh(), blas_offsets as download_instances(), `info` with the fields of
    info() it determines, `build_stats` with the fields of build_stats it determines, force_exact, and with bvh2=True the
    final BVH2 of the flat / forest run (BVH2_DTYPE, leaves first).  radius 0 means 14, as in the C ABI."""
    from tray_racing_b200 import host
    t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
    prm = OrcBuildParams(max_leaf, radius, passes, visits, rounds)
    res = OrcBuildResult()
    if object_offsets is None:
        rc = lib().orc_build_ref(t.ctypes.data, t.shape[0], None, 0, C.byref(prm), C.byref(res))
    else:
        off = np.ascontiguousarray(object_offsets, dtype=np.uint64)
        rc = lib().orc_build_ref(t.ctypes.data, t.shape[0], off.ctypes.data, off.size - 1, C.byref(prm), C.byref(res))
    if rc != 0:
        raise RuntimeError(f"reference build failed ({rc})")
    try:
        nodes = _copy(res.nodes, res.n_nodes * 80, np.uint8)
        pi = _copy(res.prim_indices, res.n_prims, np.uint32)
        blas = _copy(res.blas_offsets, res.n_instances, np.uint32)
        tree = _copy(res.bvh2, res.n_bvh2, BVH2_DTYPE) if bvh2 else None
        st = res.stats
        out = dict(
            nodes=nodes, tri_bytes=host.tri_records(t.reshape(-1, 3, 3)[pi], tri_stride), prim_indices=pi, blas_offsets=blas,
            info=dict(n_nodes=res.n_nodes, n_tris=t.shape[0], tri_stride=tri_stride, n_instances=res.n_instances,
                      tlas_start=res.tlas_start, is_tlas=int(object_offsets is not None)),
            build_stats=dict(n_tris=t.shape[0], n_nodes=st.n_nodes, ploc_iterations=st.ploc_iterations, levels=st.levels,
                             reinsert_passes=st.reinsert_passes, reinsert_moves=st.reinsert_moves,
                             sah_before=st.sah_before, sah_after=st.sah_after),
            force_exact=bool(res.force_exact), bvh2=tree, bvh2_leaves=res.n_bvh2_leaves)
    finally:
        lib().orc_build_free(C.byref(res))
    return out


def primary_rays(view, w, h, nthreads=0):
    rays = np.empty(w * h, dtype=RAY_DTYPE)
    v = _view(view)
    lib().orc_primary_rays(C.byref(v), w, h, rays.ctypes.data, nthreads)
    return rays


def node_intersect(node80, ray, tmax) -> int:
    n = np.ascontiguousarray(node80, dtype=np.uint8).reshape(80)
    r = np.ascontiguousarray(ray, dtype=RAY_DTYPE).reshape(1)
    return lib().orc_node_intersect(n.ctypes.data, r.ctypes.data, float(tmax))


def set_simd(on: bool):
    """node test on AVX2 vectors (default when the CPU has them) or scalar; results are bit-identical"""
    lib().orc_set_simd(int(on))


def simd() -> bool:
    return bool(lib().orc_simd())


def set_variant(flags: int):
    lib().orc_set_variant(flags)


def sincos_tau(u: float):
    s, c = C.c_float(), C.c_float()
    lib().orc_sincos_tau(u, C.byref(s), C.byref(c))
    return s.value, c.value
