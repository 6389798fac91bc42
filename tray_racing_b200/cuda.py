"""ctypes binding of libtray_cuda.so (include/tray_cuda.h) — the product path.

There is no CPU fallback: if the shared library is missing, or there is no CUDA device, every entry
point raises.  Nothing here imports or calls the oracle."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .host import HIT_DTYPE, RAY_DTYPE, TrayView

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TRAY_CUDA_LIB") or os.path.join(_HERE, "libtray_cuda.so")   # override: A/B builds only

RENDER_BOUNCE, RENDER_RGBA, RENDER_COUNTERS, RENDER_KEEP_RAYS, RENDER_ANYHIT_AO, RENDER_OVERLAP = 1, 2, 4, 8, 16, 32

EXPORTS = (
    "tray_cuda_device_count", "tray_cuda_abi_version", "tray_cuda_scene_create", "tray_cuda_scene_destroy",
    "tray_cuda_scene_info", "tray_cuda_trace", "tray_cuda_trace_device", "tray_cuda_render",
    "tray_cuda_shard_pixels", "tray_cuda_frame_download", "tray_cuda_frame_device_ptrs", "tray_cuda_sync",
    "tray_cuda_counters", "tray_cuda_set_counting", "tray_cuda_start", "tray_cuda_last_error",
    "tray_cuda_untile_rgba", "tray_cuda_scene_set_stream", "tray_cuda_bandwidth_probe", "tray_cuda_l1_gather_probe",
    "tray_cuda_frame_alloc", "tray_cuda_frame_free", "tray_cuda_ipc_export", "tray_cuda_ipc_open", "tray_cuda_ipc_close",
    "tray_cuda_scene_set_frame_target", "tray_cuda_render_timed", "tray_cuda_trace_any", "tray_cuda_trace_any_device",
    "tray_cuda_scene_build", "tray_cuda_scene_download", "tray_cuda_frame_readback_begin", "tray_cuda_frame_readback_wait",
    "tray_cuda_scene_build_tlas", "tray_cuda_scene_download_instances",
    "tray_cuda_scene_set_variant", "tray_cuda_shard_items", "tray_cuda_scene_set_frames_in_flight", "tray_cuda_scene_fence",
    "tray_cuda_scene_after", "tray_cuda_scene_frame_stream", "tray_cuda_frame_signal", "tray_cuda_frame_wait_flag", "tray_cuda_frame_push", "tray_cuda_untile_shards", "tray_cuda_scene_set_geometry_offsets", "tray_cuda_hits_to_geometry",
    "tray_cuda_group_create", "tray_cuda_group_destroy", "tray_cuda_group_size", "tray_cuda_group_scene",
    "tray_cuda_group_set_frames_in_flight", "tray_cuda_group_set_exchange", "tray_cuda_group_render", "tray_cuda_group_render_timed",
    "tray_cuda_group_readback_begin", "tray_cuda_group_readback_wait", "tray_cuda_group_frame_ptr", "tray_cuda_group_sync",
    "tray_cuda_start_multi",
    "tray_cuda_trace_cost", "tray_cuda_trace_cost_device", "tray_cuda_scene_set_ray_cost", "tray_cuda_frame_download_cost",
    "tray_cuda_scene_refit", "tray_cuda_scene_refit_device", "tray_cuda_scene_exact_node_test",
    "tray_cuda_scene_refit_rebuild_tlas", "tray_cuda_scene_refit_rebuild_tlas_device",
    "tray_cuda_scene_set_instances", "tray_cuda_scene_download_instance_xforms", "tray_cuda_trace_instance",
    "tray_cuda_trace_instance_device", "tray_cuda_frame_download_instance",
    "tray_cuda_hit_attributes", "tray_cuda_hit_attributes_device", "tray_cuda_frame_download_attributes",
)
# semantic switches of tray_cuda_scene_set_variant (include/tray_cuda.h TRAY_VARIANT_*)
VARIANT_BOX_DIVIDE, VARIANT_TIE_LAST, VARIANT_BOX_TMIN_RAY, VARIANT_ZERODIR_BOX_ONLY = 1, 2, 4, 8
# tray_ray_cost (include/tray_cuda.h): one ray's nodes fetched, triangles tested, TLAS leaf entries, peak stack entries
COST_DTYPE = np.dtype([("nodes", "<u4"), ("tris", "<u4"), ("instances", "<u4"), ("stack", "<u4")])
# tray_hit_attr (include/tray_cuda.h): the triangle test's barycentrics of v1 and v2 and its geometric normal (world space, not
# normalised); every byte 0xFF for a miss
ATTR_DTYPE = np.dtype([("u", "<f4"), ("v", "<f4"), ("ng", "<f4", 3)])


class TrayCudaError(RuntimeError):
    pass


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "nodes", "tris", "instances", "hits")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class BuildStats(C.Structure):
    _fields_ = [("n_tris", C.c_uint64), ("n_nodes", C.c_uint64), ("ploc_iterations", C.c_uint32), ("levels", C.c_uint32),
                ("ms_upload", C.c_float), ("ms_sort", C.c_float), ("ms_ploc", C.c_float), ("ms_collapse", C.c_float), ("ms_total", C.c_float),
                ("ms_reinsert", C.c_float), ("reinsert_passes", C.c_uint32), ("reinsert_moves", C.c_uint32),
                ("sah_before", C.c_float), ("sah_after", C.c_float)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class SceneInfo(C.Structure):
    _fields_ = [("n_nodes", C.c_uint64), ("n_tris", C.c_uint64), ("tri_stride", C.c_uint32), ("n_instances", C.c_uint32),
                ("tlas_start", C.c_uint32), ("is_tlas", C.c_uint32), ("device", C.c_int32), ("sm_count", C.c_uint32),
                ("device_bytes", C.c_uint64), ("l2_bytes", C.c_uint64), ("l2_persist_bytes", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_lib = None


def _as_u8(buf) -> np.ndarray:
    if isinstance(buf, (bytes, bytearray, memoryview)):
        return np.frombuffer(buf, dtype=np.uint8)
    return np.ascontiguousarray(buf).view(np.uint8).reshape(-1)


def lib() -> C.CDLL:
    """Load libtray_cuda.so; fail loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TrayCudaError(f"{LIB_PATH} is missing — the CUDA extension is not built and there is no fallback; "
                                "run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(LIB_PATH)
        vp, u64, u32, i32, f32p = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(C.c_float)
        L.tray_cuda_device_count.restype = i32
        L.tray_cuda_abi_version.restype = C.c_uint
        L.tray_cuda_last_error.restype = C.c_char_p
        L.tray_cuda_scene_create.restype = i32
        L.tray_cuda_scene_create.argtypes = [vp, u64, vp, u64, u32, vp, u32, u32, i32, C.POINTER(vp)]
        L.tray_cuda_scene_destroy.argtypes = [vp]
        L.tray_cuda_scene_destroy.restype = None
        L.tray_cuda_scene_info.restype = i32
        L.tray_cuda_scene_info.argtypes = [vp, C.POINTER(SceneInfo)]
        L.tray_cuda_trace.restype = i32
        L.tray_cuda_trace.argtypes = [vp, vp, u64, vp, f32p, f32p]
        L.tray_cuda_trace_device.restype = i32
        L.tray_cuda_trace_device.argtypes = [vp, vp, u64, vp, vp, f32p]
        L.tray_cuda_scene_build.restype = i32
        L.tray_cuda_scene_build.argtypes = [vp, u64, u32, u32, u32, i32, C.POINTER(vp), C.POINTER(BuildStats)]
        L.tray_cuda_scene_build_tlas.restype = i32
        L.tray_cuda_scene_build_tlas.argtypes = [vp, u64, vp, u32, u32, u32, u32, i32, C.POINTER(vp), C.POINTER(BuildStats)]
        L.tray_cuda_scene_download_instances.restype = i32
        L.tray_cuda_scene_download_instances.argtypes = [vp, vp]
        L.tray_cuda_scene_download.restype = i32
        L.tray_cuda_scene_download.argtypes = [vp, vp, vp, vp]
        L.tray_cuda_frame_readback_begin.restype = i32
        L.tray_cuda_frame_readback_begin.argtypes = [vp, vp, u32]
        L.tray_cuda_frame_readback_wait.restype = i32
        L.tray_cuda_frame_readback_wait.argtypes = [vp, u32]
        L.tray_cuda_trace_any.restype = i32
        L.tray_cuda_trace_any.argtypes = [vp, vp, u64, vp, f32p, f32p]
        L.tray_cuda_trace_any_device.restype = i32
        L.tray_cuda_trace_any_device.argtypes = [vp, vp, u64, vp, vp, f32p]
        L.tray_cuda_render.restype = i32
        L.tray_cuda_render.argtypes = [vp, C.POINTER(TrayView), u32, u32, u32, u32, u32, u32, f32p, f32p]
        L.tray_cuda_render_timed.restype = i32
        L.tray_cuda_render_timed.argtypes = [vp, C.POINTER(TrayView), u32, u32, u32, u32, u32, u32, f32p]
        L.tray_cuda_shard_pixels.restype = u64
        L.tray_cuda_shard_pixels.argtypes = [u32, u32, u32, u32]
        L.tray_cuda_frame_download.restype = i32
        L.tray_cuda_frame_download.argtypes = [vp, vp, vp, vp, vp]
        L.tray_cuda_frame_device_ptrs.restype = i32
        L.tray_cuda_frame_device_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
        L.tray_cuda_sync.restype = i32
        L.tray_cuda_sync.argtypes = [vp]
        L.tray_cuda_untile_rgba.restype = i32
        L.tray_cuda_untile_rgba.argtypes = [vp, vp, u32, u32, u32, u32, vp]
        L.tray_cuda_scene_set_stream.restype = i32
        L.tray_cuda_scene_set_stream.argtypes = [vp, vp]
        L.tray_cuda_bandwidth_probe.restype = i32
        L.tray_cuda_bandwidth_probe.argtypes = [i32, u64, i32, f32p]
        L.tray_cuda_l1_gather_probe.restype = i32
        L.tray_cuda_l1_gather_probe.argtypes = [i32, u32, i32, f32p]
        L.tray_cuda_frame_alloc.restype = i32
        L.tray_cuda_frame_alloc.argtypes = [i32, u64, C.POINTER(vp)]
        L.tray_cuda_frame_free.restype = i32
        L.tray_cuda_frame_free.argtypes = [i32, vp]
        L.tray_cuda_ipc_export.restype = i32
        L.tray_cuda_ipc_export.argtypes = [i32, vp, C.c_char_p]
        L.tray_cuda_ipc_open.restype = i32
        L.tray_cuda_ipc_open.argtypes = [i32, C.c_char_p, C.POINTER(vp)]
        L.tray_cuda_ipc_close.restype = i32
        L.tray_cuda_ipc_close.argtypes = [i32, vp]
        L.tray_cuda_scene_set_frame_target.restype = i32
        L.tray_cuda_scene_set_frame_target.argtypes = [vp, vp]
        L.tray_cuda_counters.restype = i32
        L.tray_cuda_counters.argtypes = [vp, C.POINTER(Counters), C.POINTER(Counters)]
        L.tray_cuda_set_counting.restype = i32
        L.tray_cuda_set_counting.argtypes = [vp, i32]
        L.tray_cuda_start.restype = i32
        L.tray_cuda_start.argtypes = [vp, u64, vp, u64, vp, u64, u32, u32, i32, C.POINTER(TrayView), u32, u32,
                                      C.c_float, i32, i32, i32, f32p, f32p, C.POINTER(u32)]
        L.tray_cuda_scene_set_variant.restype = i32
        L.tray_cuda_scene_set_variant.argtypes = [vp, u32]
        L.tray_cuda_shard_items.restype = u64
        L.tray_cuda_shard_items.argtypes = [u32, u32, u32, u32]
        L.tray_cuda_scene_set_frames_in_flight.restype = i32
        L.tray_cuda_scene_set_frames_in_flight.argtypes = [vp, u32]
        L.tray_cuda_scene_fence.restype = i32
        L.tray_cuda_scene_fence.argtypes = [vp, vp]
        L.tray_cuda_scene_after.restype = i32
        L.tray_cuda_scene_after.argtypes = [vp, vp]
        L.tray_cuda_frame_push.restype = i32
        L.tray_cuda_frame_push.argtypes = [vp, vp]
        L.tray_cuda_untile_shards.restype = i32
        L.tray_cuda_untile_shards.argtypes = [vp, vp, u32, u32, u32, vp]
        L.tray_cuda_frame_signal.restype = i32
        L.tray_cuda_frame_signal.argtypes = [vp, vp, u32]
        L.tray_cuda_frame_wait_flag.restype = i32
        L.tray_cuda_frame_wait_flag.argtypes = [vp, vp, u32, i32]
        L.tray_cuda_scene_frame_stream.restype = i32
        L.tray_cuda_scene_frame_stream.argtypes = [vp, i32, C.POINTER(vp)]
        L.tray_cuda_scene_set_geometry_offsets.restype = i32
        L.tray_cuda_scene_set_geometry_offsets.argtypes = [vp, vp, u32]
        L.tray_cuda_hits_to_geometry.restype = i32
        L.tray_cuda_hits_to_geometry.argtypes = [vp, vp, u64, vp, vp]
        L.tray_cuda_group_create.restype = i32
        L.tray_cuda_group_create.argtypes = [vp, u64, vp, u64, u32, vp, u32, u32, vp, i32, C.POINTER(vp)]
        L.tray_cuda_group_destroy.restype = None
        L.tray_cuda_group_destroy.argtypes = [vp]
        L.tray_cuda_group_size.restype = i32
        L.tray_cuda_group_size.argtypes = [vp]
        L.tray_cuda_group_scene.restype = i32
        L.tray_cuda_group_scene.argtypes = [vp, i32, C.POINTER(vp)]
        L.tray_cuda_group_set_frames_in_flight.restype = i32
        L.tray_cuda_group_set_frames_in_flight.argtypes = [vp, u32]
        L.tray_cuda_group_set_exchange.restype = i32
        L.tray_cuda_group_set_exchange.argtypes = [vp, i32]
        L.tray_cuda_group_render.restype = i32
        L.tray_cuda_group_render.argtypes = [vp, C.POINTER(TrayView), u32, u32, u32, u32]
        L.tray_cuda_group_render_timed.restype = i32
        L.tray_cuda_group_render_timed.argtypes = [vp, C.POINTER(TrayView), u32, u32, u32, u32, f32p]
        L.tray_cuda_group_readback_begin.restype = i32
        L.tray_cuda_group_readback_begin.argtypes = [vp, vp, u32]
        L.tray_cuda_group_readback_wait.restype = i32
        L.tray_cuda_group_readback_wait.argtypes = [vp, u32]
        L.tray_cuda_group_frame_ptr.restype = i32
        L.tray_cuda_group_frame_ptr.argtypes = [vp, C.POINTER(vp)]
        L.tray_cuda_group_sync.restype = i32
        L.tray_cuda_group_sync.argtypes = [vp]
        L.tray_cuda_trace_cost.restype = i32
        L.tray_cuda_trace_cost.argtypes = [vp, vp, u64, i32, vp, vp, f32p, f32p]
        L.tray_cuda_trace_cost_device.restype = i32
        L.tray_cuda_trace_cost_device.argtypes = [vp, vp, u64, i32, vp, vp, vp, f32p]
        L.tray_cuda_scene_set_ray_cost.restype = i32
        L.tray_cuda_scene_set_ray_cost.argtypes = [vp, i32]
        L.tray_cuda_frame_download_cost.restype = i32
        L.tray_cuda_frame_download_cost.argtypes = [vp, vp, vp]
        L.tray_cuda_start_multi.restype = i32
        L.tray_cuda_start_multi.argtypes = [vp, i32, vp, u64, vp, u64, vp, u64, u32, u32, i32, C.POINTER(TrayView), u32, u32,
                                            C.c_float, i32, i32, f32p, f32p, C.POINTER(u32)]
        L.tray_cuda_scene_refit.restype = i32
        L.tray_cuda_scene_refit.argtypes = [vp, vp, u64, f32p]
        L.tray_cuda_scene_refit_device.restype = i32
        L.tray_cuda_scene_refit_device.argtypes = [vp, vp, u64, vp, f32p]
        L.tray_cuda_scene_exact_node_test.restype = i32
        L.tray_cuda_scene_exact_node_test.argtypes = [vp, C.POINTER(i32)]
        L.tray_cuda_scene_refit_rebuild_tlas.restype = i32
        L.tray_cuda_scene_refit_rebuild_tlas.argtypes = [vp, vp, u64, u32, u32, f32p]
        L.tray_cuda_scene_refit_rebuild_tlas_device.restype = i32
        L.tray_cuda_scene_refit_rebuild_tlas_device.argtypes = [vp, vp, u64, u32, u32, vp, f32p]
        L.tray_cuda_scene_set_instances.restype = i32
        L.tray_cuda_scene_set_instances.argtypes = [vp, vp, vp, u32, u32, u32, f32p]
        L.tray_cuda_scene_download_instance_xforms.restype = i32
        L.tray_cuda_scene_download_instance_xforms.argtypes = [vp, vp, vp]
        L.tray_cuda_trace_instance.restype = i32
        L.tray_cuda_trace_instance.argtypes = [vp, vp, u64, i32, vp, vp, f32p, f32p]
        L.tray_cuda_trace_instance_device.restype = i32
        L.tray_cuda_trace_instance_device.argtypes = [vp, vp, u64, i32, vp, vp, vp, f32p]
        L.tray_cuda_frame_download_instance.restype = i32
        L.tray_cuda_frame_download_instance.argtypes = [vp, vp, vp]
        L.tray_cuda_hit_attributes.restype = i32
        L.tray_cuda_hit_attributes.argtypes = [vp, vp, vp, vp, u64, vp, f32p]
        L.tray_cuda_hit_attributes_device.restype = i32
        L.tray_cuda_hit_attributes_device.argtypes = [vp, vp, vp, vp, u64, vp, vp, f32p]
        L.tray_cuda_frame_download_attributes.restype = i32
        L.tray_cuda_frame_download_attributes.argtypes = [vp, vp, vp]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise TrayCudaError(f"tray_cuda error {rc}: {lib().tray_cuda_last_error().decode(errors='replace')}")


def device_count() -> int:
    return lib().tray_cuda_device_count()


def l1_gather_probe(nbytes: int = 32 << 10, iters: int = 200, device: int = 0) -> float:
    """GB/s (whole chip) the L1 delivers when every lane gathers its own 16-byte record from a different line of an
    L1-resident `nbytes` table — the access pattern of a traversal warp."""
    g = C.c_float()
    _check(lib().tray_cuda_l1_gather_probe(device, int(nbytes), int(iters), C.byref(g)))
    return g.value


def bandwidth_probe(nbytes: int, iters: int = 20, device: int = 0) -> float:
    """Streaming-read GB/s over an `nbytes` buffer: << L2 size measures L2, >> L2 measures HBM."""
    g = C.c_float()
    _check(lib().tray_cuda_bandwidth_probe(device, int(nbytes), int(iters), C.byref(g)))
    return g.value


def frame_alloc(nbytes: int, device: int = 0) -> int:
    """A zeroed device allocation that can be exported over CUDA IPC (the shared row-major frame of a multi-GPU run)."""
    p = C.c_void_p()
    _check(lib().tray_cuda_frame_alloc(device, int(nbytes), C.byref(p)))
    return p.value


def frame_free(ptr: int, device: int = 0):
    _check(lib().tray_cuda_frame_free(device, C.c_void_p(ptr)))


def ipc_export(ptr: int, device: int = 0) -> bytes:
    h = C.create_string_buffer(64)
    _check(lib().tray_cuda_ipc_export(device, C.c_void_p(ptr), h))
    return h.raw


def ipc_open(handle: bytes, device: int = 0) -> int:
    """Map another process's frame_alloc() allocation (same box) into this process; enables peer access."""
    if len(handle) != 64:
        raise ValueError("a CUDA IPC handle is 64 bytes")
    p = C.c_void_p()
    _check(lib().tray_cuda_ipc_open(device, C.create_string_buffer(handle, 64), C.byref(p)))
    return p.value


def ipc_close(ptr: int, device: int = 0):
    _check(lib().tray_cuda_ipc_close(device, C.c_void_p(ptr)))


def shard_pixels(w: int, h: int, shard: int = 0, shards: int = 1) -> int:
    return lib().tray_cuda_shard_pixels(w, h, shard, shards)


class TrayCudaScene:
    """A CWBVH resident on one GPU.  Batch-grain `Traversable` (reference traversable/src/lib.rs:13-28):
    `traverse(rays) -> hits`, plus the frame operator of the render loop (reference src/rt_cpu/rt_cpu.rs:35-91)."""

    def __init__(self, bvh_bytes, tri_bytes, tri_stride=48, blas_offsets=None, tlas_start=0, device=0):
        nodes = _as_u8(bvh_bytes)
        tris = _as_u8(tri_bytes)
        if nodes.size % 80:
            raise ValueError("bvh_bytes length is not a multiple of 80")        # reference src/rt_gpu/mod.rs:70,105
        if tris.size % tri_stride:
            raise ValueError("tri_bytes length is not a multiple of tri_stride")  # reference src/rt_gpu/mod.rs:86,107
        blas = None if blas_offsets is None else np.ascontiguousarray(blas_offsets, dtype=np.uint32)
        h = C.c_void_p()
        _check(lib().tray_cuda_scene_create(nodes.ctypes.data, nodes.size // 80, tris.ctypes.data, tris.size // tri_stride,
                                            tri_stride, None if blas is None else blas.ctypes.data,
                                            0 if blas is None else blas.size, tlas_start, device, C.byref(h)))
        self._h = h
        self.tri_stride = tri_stride
        self.frame_size = None

    @classmethod
    def build(cls, tris, tri_stride=48, max_prims_per_leaf=3, search_radius=0, device=0, object_offsets=None) -> "TrayCudaScene":
        """Build the CWBVH ON THE GPU from a triangle soup (n x 3 x 3 floats) — tray_cuda_scene_build; the reference's
        `cwbvh_from_tris` (src/cwbvh.rs:24-105) runs on the CPU.  With `object_offsets` (n_objects + 1 triangle offsets):
        one BLAS per object + a TLAS (`tlas_from_blas`, src/cwbvh.rs:108-137) — tray_cuda_scene_build_tlas.
        `build_stats` holds the phase times."""
        t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
        self = cls.__new__(cls)
        h, st = C.c_void_p(), BuildStats()
        if object_offsets is not None:
            off = np.ascontiguousarray(object_offsets, dtype=np.uint64)
            _check(lib().tray_cuda_scene_build_tlas(t.ctypes.data, t.shape[0], off.ctypes.data, off.size - 1, tri_stride,
                                                    max_prims_per_leaf, search_radius, device, C.byref(h), C.byref(st)))
        else:
            _check(lib().tray_cuda_scene_build(t.ctypes.data, t.shape[0], tri_stride, max_prims_per_leaf, search_radius, device,
                                               C.byref(h), C.byref(st)))
        self._h = h
        self.tri_stride = tri_stride
        self.frame_size = None
        self.build_stats = st.as_dict()
        return self

    def download_bvh(self, prim_indices: bool = True):
        """(bvh_bytes, tri_bytes, prim_indices) of the scene, copied back to the host (tray_cuda_scene_download)."""
        i = self.info()
        nodes = np.zeros(i["n_nodes"] * 80, dtype=np.uint8)
        tris = np.zeros(i["n_tris"] * i["tri_stride"], dtype=np.uint8)
        pi = np.zeros(i["n_tris"], dtype=np.uint32) if prim_indices else None
        _check(lib().tray_cuda_scene_download(self._h, nodes.ctypes.data, tris.ctypes.data, None if pi is None else pi.ctypes.data))
        return nodes, tris, pi

    def download_instances(self) -> np.ndarray:
        """blas_offsets of a two-level scene (tray_cuda_scene_download_instances)"""
        out = np.zeros(self.info()["n_instances"], dtype=np.uint32)
        if out.size:
            _check(lib().tray_cuda_scene_download_instances(self._h, out.ctypes.data))
        return out

    def exact_node_test(self) -> bool:
        """Whether traversal takes the unfused node test everywhere (a node scale >= 2^40, or TRAY_CUDA_FORCE_EXACT)."""
        e = C.c_int()
        _check(lib().tray_cuda_scene_exact_node_test(self._h, C.byref(e)))
        return bool(e.value)

    def refit(self, tris, timings: dict | None = None):
        """Same tree, new vertex positions: `tris` (n x 3 x 3 or n x 9 float32) in the scene's triangle order — input order for
        a built scene, BVH slot order for one made from bytes (tray_cuda_scene_refit).  timings["ms_refit"]: the refit launches."""
        t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
        ms = C.c_float()
        _check(lib().tray_cuda_scene_refit(self._h, t.ctypes.data, t.shape[0], C.byref(ms)))
        if timings is not None:
            timings["ms_refit"] = ms.value

    def refit_device(self, d_ptr: int, n: int, stream: int = 0, timed: bool = False):
        """refit() from n x 9 float32 in device memory, after the work enqueued so far on `stream` (tray_cuda_scene_refit_device);
        returns ms_refit when `timed`."""
        ms = C.c_float()
        _check(lib().tray_cuda_scene_refit_device(self._h, d_ptr, n, stream or None, C.byref(ms) if timed else None))
        return ms.value if timed else None

    def refit_rebuild_tlas(self, tris, max_prims_per_leaf=3, search_radius=0, timings: dict | None = None):
        """Two-level scenes whose objects move as a whole: refit every BLAS as refit() does and rebuild the TLAS over the BLAS
        roots' boxes as build() builds it (tray_cuda_scene_refit_rebuild_tlas).  `tris` in the scene's triangle order, as for
        refit().  timings["ms_refit_rebuild_tlas"]: coordinate check to the last TLAS write."""
        t = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 9)
        ms = C.c_float()
        _check(lib().tray_cuda_scene_refit_rebuild_tlas(self._h, t.ctypes.data, t.shape[0], max_prims_per_leaf, search_radius, C.byref(ms)))
        if timings is not None:
            timings["ms_refit_rebuild_tlas"] = ms.value

    def refit_rebuild_tlas_device(self, d_ptr: int, n: int, max_prims_per_leaf=3, search_radius=0, stream: int = 0, timed: bool = False):
        """refit_rebuild_tlas() from n x 9 float32 in device memory, after the work enqueued so far on `stream`
        (tray_cuda_scene_refit_rebuild_tlas_device); returns the call's ms when `timed`."""
        ms = C.c_float()
        _check(lib().tray_cuda_scene_refit_rebuild_tlas_device(self._h, d_ptr, n, max_prims_per_leaf, search_radius, stream or None,
                                                                C.byref(ms) if timed else None))
        return ms.value if timed else None

    def set_instances(self, blas_roots, object_to_world, max_prims_per_leaf=3, search_radius=0, timings: dict | None = None):
        """Place BLAS by transforms (tray_cuda_scene_set_instances): instance k is the BLAS whose root node is blas_roots[k]
        (one of the scene's blas_offsets values), placed by object_to_world[k], a row-major 3 x 4 [R | t].  Only the TLAS is
        built; timings["ms_set_instances"]: upload of the transforms to the last TLAS write."""
        roots = np.asarray(blas_roots)
        xf = np.asarray(object_to_world)
        if roots.ndim != 1 or roots.size == 0 or roots.dtype.kind not in "iu":
            raise ValueError("blas_roots must be a non-empty 1-D integer array")
        if (roots < 0).any() or (roots > 0xFFFFFFFF).any():
            raise ValueError("blas_roots must be node indices (uint32)")
        if xf.dtype.kind != "f" or xf.shape != (roots.size, 3, 4):
            raise ValueError(f"object_to_world must be a float array of shape ({roots.size}, 3, 4), got {xf.dtype} {xf.shape}")
        roots = np.ascontiguousarray(roots, dtype=np.uint32)
        xf = np.ascontiguousarray(xf, dtype=np.float32)
        ms = C.c_float()
        _check(lib().tray_cuda_scene_set_instances(self._h, roots.ctypes.data, xf.ctypes.data, roots.size, max_prims_per_leaf,
                                                    search_radius, C.byref(ms)))
        if timings is not None:
            timings["ms_set_instances"] = ms.value

    def download_instance_xforms(self):
        """(leaf_instance, world_to_object): the instance of every TLAS leaf, and every instance's world_to_object (n, 3, 4)
        as the kernels use it (tray_cuda_scene_download_instance_xforms)."""
        n = self.info()["n_instances"]
        leaf, w2o = np.zeros(n, dtype=np.uint32), np.zeros((n, 3, 4), dtype=np.float32)
        _check(lib().tray_cuda_scene_download_instance_xforms(self._h, leaf.ctypes.data, w2o.ctypes.data))
        return leaf, w2o

    def traverse_instance(self, rays: np.ndarray, any_hit: bool = False, timings: dict | None = None):
        """(hits, instance_ids): traverse() on an instanced scene plus the instance of every hit, 0xFFFFFFFF for a miss
        (tray_cuda_trace_instance)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        ids = np.empty(rays.shape[0], dtype=np.uint32)
        k, t = C.c_float(), C.c_float()
        _check(lib().tray_cuda_trace_instance(self._h, rays.ctypes.data, rays.shape[0], int(any_hit), hits.ctypes.data, ids.ctypes.data,
                                              C.byref(k), C.byref(t)))
        if timings is not None:
            timings["ms_kernel"], timings["ms_total"] = k.value, t.value
        return hits, ids

    def traverse_instance_device(self, d_rays_ptr: int, n: int, d_hits_ptr: int, d_ids_ptr: int, stream: int = 0, timed: bool = False,
                                 any_hit: bool = False):
        """traverse_device() plus a uint32 instance id per ray at `d_ids_ptr` — tray_cuda_trace_instance_device."""
        k = C.c_float()
        _check(lib().tray_cuda_trace_instance_device(self._h, d_rays_ptr, n, int(any_hit), d_hits_ptr, d_ids_ptr, stream or None,
                                                     C.byref(k) if timed else None))
        return k.value if timed else None

    def download_instance(self, primary=True, bounce=False) -> dict:
        """The last frame's instance ids (uint32, row-major, w*h): "primary" and / or "bounce"; 0xFFFFFFFF for misses, other
        shards' pixels and pixels without a bounce ray (tray_cuda_frame_download_instance)."""
        w, h = self.frame_size
        out = {name: np.zeros(w * h, dtype=np.uint32) for name, want in (("primary", primary), ("bounce", bounce)) if want}
        p, b = out.get("primary"), out.get("bounce")
        _check(lib().tray_cuda_frame_download_instance(self._h, None if p is None else p.ctypes.data, None if b is None else b.ctypes.data))
        return out

    def _instanced(self) -> bool:
        """whether set_instances has made the scene instanced (the library accepts its instance-transform download)"""
        h = getattr(self, "_h", None)
        return bool(h is not None and h.value) and lib().tray_cuda_scene_download_instance_xforms(h, None, None) == 0

    def hit_attributes(self, rays, hits, instance_ids=None, timings: dict | None = None) -> np.ndarray:
        """{u, v, ng} (ATTR_DTYPE) of every hit on its ray, as the triangle test computed them (tray_cuda_hit_attributes).
        `instance_ids` (from traverse_instance) is required on an instanced scene and must be None on any other."""
        rays, hits = np.asarray(rays), np.asarray(hits)
        if rays.dtype != RAY_DTYPE or hits.dtype != HIT_DTYPE:
            raise ValueError(f"rays must be RAY_DTYPE and hits HIT_DTYPE, got {rays.dtype} and {hits.dtype}")
        if rays.ndim != 1 or rays.shape != hits.shape:
            raise ValueError(f"rays and hits must be 1-D arrays of one length, got {rays.shape} and {hits.shape}")
        ids = None
        if instance_ids is not None:
            ids = np.asarray(instance_ids)
            if ids.dtype.kind not in "iu" or ids.shape != hits.shape or (ids.size and (ids.min() < 0 or ids.max() > 0xFFFFFFFF)):
                raise ValueError(f"instance_ids must be uint32 of shape {hits.shape}")
            ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if (ids is None) == self._instanced():
            raise ValueError("instance_ids are required on an instanced scene and refused on any other")
        rays, hits = np.ascontiguousarray(rays), np.ascontiguousarray(hits)
        out = np.empty(rays.shape[0], dtype=ATTR_DTYPE)
        k = C.c_float()
        _check(lib().tray_cuda_hit_attributes(self._h, rays.ctypes.data, hits.ctypes.data, None if ids is None else ids.ctypes.data,
                                              rays.shape[0], out.ctypes.data, C.byref(k)))
        if timings is not None:
            timings["ms_kernel"] = k.value
        return out

    def hit_attributes_device(self, d_rays_ptr: int, d_hits_ptr: int, d_ids_ptr: int | None, n: int, d_attrs_ptr: int, stream: int = 0,
                              timed: bool = False):
        """hit_attributes() on device buffers (20-byte records at `d_attrs_ptr`), ordered after the scene stream's traces
        (tray_cuda_hit_attributes_device); returns ms_kernel when `timed`."""
        k = C.c_float()
        _check(lib().tray_cuda_hit_attributes_device(self._h, d_rays_ptr, d_hits_ptr, d_ids_ptr or None, n, d_attrs_ptr, stream or None,
                                                     C.byref(k) if timed else None))
        return k.value if timed else None

    def download_attributes(self, primary=True, bounce=False) -> dict:
        """The last frame's hit attributes (ATTR_DTYPE, row-major, w*h): "primary" and / or "bounce"; every byte 0xFF for misses,
        other shards' pixels and pixels without a bounce ray (tray_cuda_frame_download_attributes)."""
        w, h = self.frame_size
        out = {name: np.zeros(w * h, dtype=ATTR_DTYPE) for name, want in (("primary", primary), ("bounce", bounce)) if want}
        p, b = out.get("primary"), out.get("bounce")
        _check(lib().tray_cuda_frame_download_attributes(self._h, None if p is None else p.ctypes.data, None if b is None else b.ctypes.data))
        return out

    @classmethod
    def from_packed(cls, p, device=0) -> "TrayCudaScene":
        return cls(p.bvh_bytes, p.tri_bytes, p.tri_stride, p.blas_offsets if p.use_tlas else None, p.tlas_start, device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value and _lib is not None:
            if not getattr(self, "_borrowed", False):        # a scene borrowed from a TrayCudaGroup belongs to the group
                _lib.tray_cuda_scene_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def info(self) -> dict:
        i = SceneInfo()
        _check(lib().tray_cuda_scene_info(self._h, C.byref(i)))
        return i.as_dict()

    # ---- Traversable::traverse at batch grain -----------------------------------------------
    def traverse(self, rays: np.ndarray, timings: dict | None = None, any_hit: bool = False) -> np.ndarray:
        """Closest hit per ray (`Traversable::traverse` at batch grain); any_hit=True stops each ray at its first
        accepted triangle (tray_cuda_trace_any)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        k, t = C.c_float(), C.c_float()
        fn = lib().tray_cuda_trace_any if any_hit else lib().tray_cuda_trace
        _check(fn(self._h, rays.ctypes.data, rays.shape[0], hits.ctypes.data, C.byref(k), C.byref(t)))
        if timings is not None:
            timings["ms_kernel"], timings["ms_total"] = k.value, t.value
        return hits

    def traverse_device(self, d_rays_ptr: int, n: int, d_hits_ptr: int, stream: int = 0, timed: bool = False, any_hit: bool = False):
        k = C.c_float()
        fn = lib().tray_cuda_trace_any_device if any_hit else lib().tray_cuda_trace_device
        _check(fn(self._h, d_rays_ptr, n, d_hits_ptr, stream or None, C.byref(k) if timed else None))
        return k.value if timed else None

    def set_counting(self, on: bool):
        _check(lib().tray_cuda_set_counting(self._h, int(on)))

    def traverse_cost(self, rays: np.ndarray, any_hit: bool = False, timings: dict | None = None):
        """(hits, costs): traverse() plus the cost of every ray (COST_DTYPE) — tray_cuda_trace_cost."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        costs = np.empty(rays.shape[0], dtype=COST_DTYPE)
        k, t = C.c_float(), C.c_float()
        _check(lib().tray_cuda_trace_cost(self._h, rays.ctypes.data, rays.shape[0], int(any_hit), hits.ctypes.data, costs.ctypes.data,
                                          C.byref(k), C.byref(t)))
        if timings is not None:
            timings["ms_kernel"], timings["ms_total"] = k.value, t.value
        return hits, costs

    def traverse_cost_device(self, d_rays_ptr: int, n: int, d_hits_ptr: int, d_costs_ptr: int, stream: int = 0, timed: bool = False,
                             any_hit: bool = False):
        """traverse_device() plus 16-byte cost records at `d_costs_ptr` — tray_cuda_trace_cost_device."""
        k = C.c_float()
        _check(lib().tray_cuda_trace_cost_device(self._h, d_rays_ptr, n, int(any_hit), d_hits_ptr, d_costs_ptr, stream or None,
                                                 C.byref(k) if timed else None))
        return k.value if timed else None

    def set_ray_cost(self, on: bool):
        """While on, every render with RENDER_COUNTERS keeps each ray's cost for download_cost()."""
        _check(lib().tray_cuda_scene_set_ray_cost(self._h, int(on)))

    def set_variant(self, flags: int):
        """Run the other reading of the semantics that are sourced from memory of obvhs (VARIANT_* flags; 0 = default)."""
        _check(lib().tray_cuda_scene_set_variant(self._h, int(flags)))

    def set_frames_in_flight(self, n: int):
        """1 (default) or 2: consecutive render() calls alternate between two frame slots / streams (include/tray_cuda.h)."""
        _check(lib().tray_cuda_scene_set_frames_in_flight(self._h, int(n)))

    def fence(self, cuda_stream: int = 0):
        """`cuda_stream` (0 = the scene stream) waits for every frame enqueued so far."""
        _check(lib().tray_cuda_scene_fence(self._h, cuda_stream or None))

    def after(self, cuda_stream: int):
        """Frames enqueued from now on start after the work already enqueued on `cuda_stream`."""
        _check(lib().tray_cuda_scene_after(self._h, cuda_stream))

    def push(self, d_dst: int):
        """One DMA copy of the last frame's compact RGBA shard to `d_dst` (this or a peer device) on the frame's stream."""
        _check(lib().tray_cuda_frame_push(self._h, C.c_void_p(d_dst)))

    def untile_shards(self, d_staging: int, width: int, height: int, shards: int, d_frame: int):
        """All shards' compact RGBA (back to back in `d_staging`) -> the row-major frame, one launch on the frame's stream."""
        _check(lib().tray_cuda_untile_shards(self._h, C.c_void_p(d_staging), width, height, shards, C.c_void_p(d_frame)))

    def signal(self, d_flag: int, value: int):
        """Behind the last frame: write `value` to the 32-bit flag at device address `d_flag` (possibly peer memory) — no kernel."""
        _check(lib().tray_cuda_frame_signal(self._h, C.c_void_p(d_flag), value & 0xFFFFFFFF))

    def wait_flag(self, d_flag: int, value: int, before_next_frame: bool = False):
        """The stream of the last frame (or of the next one) waits until the flag at `d_flag` has reached `value` — no kernel."""
        _check(lib().tray_cuda_frame_wait_flag(self._h, C.c_void_p(d_flag), value & 0xFFFFFFFF, int(before_next_frame)))

    def frame_stream(self, which: int = -1) -> int:
        """cudaStream_t of frame slot `which` (0 / 1), or of the last rendered frame (-1); 0 = the legacy default stream."""
        p = C.c_void_p()
        _check(lib().tray_cuda_scene_frame_stream(self._h, which, C.byref(p)))
        return p.value or 0

    def set_geometry_offsets(self, tri_offsets):
        """First global triangle of every BLAS / object (n + 1 entries) — the runner's running `tri_offset`, rt_gpu/mod.rs:45-47."""
        off = np.ascontiguousarray(tri_offsets, dtype=np.uint32)
        _check(lib().tray_cuda_scene_set_geometry_offsets(self._h, off.ctypes.data if off.size else None, max(0, off.size - 1)))

    def hits_to_geometry(self, hits: np.ndarray):
        """(geometry_id, primitive_id) per hit, as `CwBvhTlasScene::traverse` reports them (src/cwbvh.rs:144-166)."""
        hits = np.ascontiguousarray(hits, dtype=HIT_DTYPE)
        g, pr = np.empty(hits.shape[0], dtype=np.uint32), np.empty(hits.shape[0], dtype=np.uint32)
        _check(lib().tray_cuda_hits_to_geometry(self._h, hits.ctypes.data, hits.shape[0], g.ctypes.data, pr.ctypes.data))
        return g, pr

    def counters(self):
        a, b = Counters(), Counters()
        _check(lib().tray_cuda_counters(self._h, C.byref(a), C.byref(b)))
        return a.as_dict(), b.as_dict()

    # ---- frame operator ------------------------------------------------------------------------
    def render(self, view: TrayView, width: int, height: int, frame_count: int = 0, flags: int = RENDER_BOUNCE | RENDER_RGBA,
               shard: int = 0, shards: int = 1, timed: bool = True):
        a, b = C.c_float(), C.c_float()
        _check(lib().tray_cuda_render(self._h, C.byref(view), width, height, frame_count, flags, shard, shards,
                                      C.byref(a) if timed else None, C.byref(b) if timed else None))
        self.frame_size = (width, height)
        self.frame_shard = (shard, shards)
        return (a.value, b.value) if timed else None

    def render_frame_ms(self, view: TrayView, width: int, height: int, frame_count: int = 0, flags: int = RENDER_BOUNCE | RENDER_RGBA,
                        shard: int = 0, shards: int = 1) -> float:
        """Whole-frame CUDA-event time (ray generation + both traversal launches) — tray_cuda_render_timed."""
        ms = C.c_float()
        _check(lib().tray_cuda_render_timed(self._h, C.byref(view), width, height, frame_count, flags, shard, shards, C.byref(ms)))
        self.frame_size = (width, height)
        self.frame_shard = (shard, shards)
        return ms.value

    def readback_begin(self, rgba: np.ndarray, slot: int):
        """Start the asynchronous copy of the last frame's RGBA8 into `rgba` ((h, w, 4) uint8, pinned for overlap)."""
        w, h = self.frame_size
        assert rgba.dtype == np.uint8 and rgba.size == w * h * 4 and rgba.flags["C_CONTIGUOUS"]
        _check(lib().tray_cuda_frame_readback_begin(self._h, rgba.ctypes.data, slot))

    def readback_wait(self, slot: int):
        _check(lib().tray_cuda_frame_readback_wait(self._h, slot))

    def download(self, primary=False, bounce=False, bounce_rays=False, rgba=False, into: dict | None = None,
                 merge: bool = False) -> dict:
        """Last frame -> host arrays in row-major pixel order.  Pixels of other shards come back as zeros; with
        merge=True only this shard's pixels of the arrays already in `into` are overwritten."""
        w, h = self.frame_size
        out = into if (into is not None and not merge) else {}
        def buf(name, want, dtype, shape):
            if not want:
                return None
            if name not in out:
                out[name] = np.zeros(shape, dtype=dtype)
            return out[name]
        p = buf("primary", primary, HIT_DTYPE, w * h)
        b = buf("bounce", bounce, HIT_DTYPE, w * h)
        r = buf("bounce_rays", bounce_rays, RAY_DTYPE, w * h)
        g = buf("rgba", rgba, np.uint8, (h, w, 4))
        _check(lib().tray_cuda_frame_download(self._h, None if p is None else p.ctypes.data, None if b is None else b.ctypes.data,
                                              None if r is None else r.ctypes.data, None if g is None else g.ctypes.data))
        return self._merged(out, into) if merge and into is not None else out

    def download_cost(self, primary=True, bounce=False, into: dict | None = None, merge: bool = False) -> dict:
        """The last frame's ray costs (COST_DTYPE, row-major, w*h): "primary" and / or "bounce" (zero where a pixel shot no
        bounce ray).  Pixels of other shards come back as zeros; merge=True as in download()."""
        w, h = self.frame_size
        out = into if (into is not None and not merge) else {}
        for name, want in (("primary", primary), ("bounce", bounce)):
            if want and name not in out:
                out[name] = np.zeros(w * h, dtype=COST_DTYPE)
        p, b = out.get("primary") if primary else None, out.get("bounce") if bounce else None
        _check(lib().tray_cuda_frame_download_cost(self._h, None if p is None else p.ctypes.data, None if b is None else b.ctypes.data))
        return self._merged(out, into) if merge and into is not None else out

    def _merged(self, out: dict, into: dict) -> dict:
        """this shard's pixels of `out` written over the arrays of `into` (arrays `into` lacks are taken whole)"""
        w, h = self.frame_size
        shard, shards = self.frame_shard
        own = shard_mask(w, h, shard, shards)
        for k, v in out.items():
            if k not in into:
                into[k] = v
            elif k == "rgba":
                into[k][own.reshape(h, w)] = v[own.reshape(h, w)]
            else:
                into[k][own] = v[own]
        return into

    def frame_device_ptrs(self):
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _check(lib().tray_cuda_frame_device_ptrs(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def sync(self):
        _check(lib().tray_cuda_sync(self._h))

    def set_stream(self, cuda_stream: int):
        """Enqueue this scene's work on a caller-owned cudaStream_t (0 restores the scene's own stream)."""
        _check(lib().tray_cuda_scene_set_stream(self._h, cuda_stream or None))

    def set_frame_target(self, d_frame: int | None):
        """RGBA of later renders goes straight into the row-major frame at `d_frame` (this GPU or a peer mapping from
        ipc_open): the fused framebuffer exchange of include/tray_cuda.h.  None restores the compact local buffer."""
        _check(lib().tray_cuda_scene_set_frame_target(self._h, C.c_void_p(d_frame or 0)))

    def untile_rgba(self, d_compact: int, width: int, height: int, shard: int, shards: int, d_frame: int):
        _check(lib().tray_cuda_untile_rgba(self._h, d_compact, width, height, shard, shards, d_frame))


class TrayCudaGroup:
    """One process, several GPUs (include/tray_cuda.h `tray_group`): BVH replicated on `devices`, tiles dealt round-robin,
    pixels stored straight into one row-major frame on devices[0] over peer access, completion by events."""

    def __init__(self, bvh_bytes, tri_bytes, tri_stride=48, blas_offsets=None, tlas_start=0, devices=(0,)):
        nodes, tris = _as_u8(bvh_bytes), _as_u8(tri_bytes)
        blas = None if blas_offsets is None else np.ascontiguousarray(blas_offsets, dtype=np.uint32)
        dev = np.ascontiguousarray(list(devices), dtype=np.int32)
        h = C.c_void_p()
        _check(lib().tray_cuda_group_create(nodes.ctypes.data, nodes.size // 80, tris.ctypes.data, tris.size // tri_stride, tri_stride,
                                            None if blas is None else blas.ctypes.data, 0 if blas is None else blas.size, tlas_start,
                                            dev.ctypes.data, dev.size, C.byref(h)))
        self._h = h
        self.devices = list(devices)
        self.frame_size = None

    @classmethod
    def from_packed(cls, p, devices=(0,)) -> "TrayCudaGroup":
        return cls(p.bvh_bytes, p.tri_bytes, p.tri_stride, p.blas_offsets if p.use_tlas else None, p.tlas_start, devices)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value and _lib is not None:
            _lib.tray_cuda_group_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def scene(self, i: int) -> "TrayCudaScene":
        """Borrowed scene of devices[i] (do not close it)."""
        h = C.c_void_p()
        _check(lib().tray_cuda_group_scene(self._h, i, C.byref(h)))
        sc = TrayCudaScene.__new__(TrayCudaScene)
        sc._h, sc.tri_stride, sc.frame_size, sc._borrowed = h, None, self.frame_size, True
        sc.frame_shard = (i, len(self.devices))
        return sc

    def set_frames_in_flight(self, n: int):
        _check(lib().tray_cuda_group_set_frames_in_flight(self._h, int(n)))

    def set_exchange(self, push: bool):
        """push (default): one peer DMA copy per shard + one untile launch on devices[0]; else the kernels store pixels into the frame."""
        _check(lib().tray_cuda_group_set_exchange(self._h, int(push)))

    def render(self, view: TrayView, width: int, height: int, frame_count: int = 0, flags: int = RENDER_BOUNCE | RENDER_RGBA, timed: bool = False):
        self.frame_size = (width, height)
        if timed:
            ms = C.c_float()
            _check(lib().tray_cuda_group_render_timed(self._h, C.byref(view), width, height, frame_count, flags, C.byref(ms)))
            return ms.value
        _check(lib().tray_cuda_group_render(self._h, C.byref(view), width, height, frame_count, flags))
        return None

    def readback_begin(self, rgba: np.ndarray, slot: int):
        w, h = self.frame_size
        assert rgba.dtype == np.uint8 and rgba.size == w * h * 4 and rgba.flags["C_CONTIGUOUS"]
        _check(lib().tray_cuda_group_readback_begin(self._h, rgba.ctypes.data, slot))

    def readback_wait(self, slot: int):
        _check(lib().tray_cuda_group_readback_wait(self._h, slot))

    def frame(self) -> np.ndarray:
        """The last frame, (h, w, 4) uint8, synchronously."""
        w, h = self.frame_size
        out = np.zeros((h, w, 4), dtype=np.uint8)
        self.readback_begin(out, 0)
        self.readback_wait(0)
        return out

    def frame_ptr(self) -> int:
        p = C.c_void_p()
        _check(lib().tray_cuda_group_frame_ptr(self._h, C.byref(p)))
        return p.value

    def sync(self):
        _check(lib().tray_cuda_group_sync(self._h))


def start_multi(devices, bvh_bytes, instance_bytes, tri_bytes, tlas_start, view: TrayView, width=1920, height=1080, render_time=1.0,
                benchmark=True, animate=False, use_tlas=False, tri_stride=48):
    """tray_cuda_start on several GPUs in ONE process (tray_cuda_start_multi).  Returns (min_ms, mean_ms, frames)."""
    nodes, inst, tris = _as_u8(bvh_bytes), _as_u8(instance_bytes), _as_u8(tri_bytes)
    dev = np.ascontiguousarray(list(devices), dtype=np.int32)
    mn, mean, frames = C.c_float(), C.c_float(), C.c_uint32()
    _check(lib().tray_cuda_start_multi(dev.ctypes.data, dev.size, nodes.ctypes.data, nodes.size, inst.ctypes.data, inst.size,
                                       tris.ctypes.data, tris.size, tri_stride, tlas_start, int(use_tlas), C.byref(view), width, height,
                                       float(render_time), int(benchmark), int(animate), C.byref(mn), C.byref(mean), C.byref(frames)))
    return mn.value, mean.value, frames.value


def shard_mask(width: int, height: int, shard: int, shards: int) -> np.ndarray:
    """bool[h*w]: pixels owned by `shard` — 32x8-pixel tiles, tile k (row-major) belongs to shard k % shards."""
    y, x = np.divmod(np.arange(width * height), width)
    k = (y // 8) * ((width + 31) // 32) + x // 32
    return (k % shards) == shard


def local_items(width: int, height: int, shard: int = 0, shards: int = 1) -> int:
    """Entries of a shard's compact (tile-ordered) frame buffers: its 32x8 tiles x 256."""
    tiles = ((width + 31) // 32) * ((height + 7) // 8)
    return 0 if shard >= tiles else ((tiles - shard + shards - 1) // shards) * 256


class DeviceArray:
    """Zero-copy view of device memory owned by libtray_cuda for consumers of __cuda_array_interface__
    (torch.as_tensor(DeviceArray(...), device="cuda")) — used to hand shard buffers to NCCL."""

    def __init__(self, ptr: int, shape, typestr: str, owner=None):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}
        self._owner = owner


def start(bvh_bytes, instance_bytes, tri_bytes, tlas_start, view: TrayView, width=1920, height=1080, render_time=1.0,
          benchmark=True, animate=False, use_tlas=False, tri_stride=48, device=0):
    """`rt_gpu_software::start(.., bvh_bytes, instance_bytes, tri_bytes, tlas_start) -> f32`
    (reference src/rt_gpu/rt_gpu_software.rs:24-32).  Returns (min_ms, mean_ms, frames); the reference returns min_ms."""
    nodes = _as_u8(bvh_bytes)
    inst = _as_u8(instance_bytes)
    tris = _as_u8(tri_bytes)
    mn, mean, frames = C.c_float(), C.c_float(), C.c_uint32()
    _check(lib().tray_cuda_start(nodes.ctypes.data, nodes.size, inst.ctypes.data, inst.size, tris.ctypes.data, tris.size,
                                 tri_stride, tlas_start, int(use_tlas), C.byref(view), width, height, float(render_time),
                                 int(benchmark), int(animate), device, C.byref(mn), C.byref(mean), C.byref(frames)))
    return mn.value, mean.value, frames.value
