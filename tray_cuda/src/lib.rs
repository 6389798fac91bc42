//! Thin Rust face of `include/tray_cuda.h`.  Mirrors `rt_gpu_software::start` (tray_racing
//! src/rt_gpu/rt_gpu_software.rs:24-32) so that `cwbvh_cuda_runner` reads like `cwbvh_gpu_runner`.
//! Authored against the header; not compiled in the build image (no Rust toolchain there).
use std::ffi::{c_char, c_int, c_void, CStr};

#[repr(C)]
#[derive(Clone, Copy, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayRay { pub origin: [f32; 3], pub tmin: f32, pub dir: [f32; 3], pub tmax: f32 }

#[repr(C)]
#[derive(Clone, Copy, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayHit { pub t: f32, pub prim: u32 }

/// `tray_hit_attr` of include/tray_cuda.h: the triangle test's barycentrics of v1 and v2 (v0's is 1 - u - v) and its geometric
/// normal in world space, not normalised; every byte 0xFF (NaN) for a miss.  20 bytes.
#[repr(C)]
#[derive(Clone, Copy, Debug, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayHitAttr { pub u: f32, pub v: f32, pub ng: [f32; 3] }

/// `ViewUniform` of tray_racing (src/main.rs:589-597) padded to 160 bytes.
#[repr(C)]
#[derive(Clone, Copy, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayView {
    pub view_inv: [f32; 16], pub proj_inv: [f32; 16], pub eye: [f32; 3], pub exposure: f32,
    pub tlas_start: u32, pub pad: [u32; 3],
}

/// f32 triangle record: obvhs `RtTriangle` without `ng` (48 B) — `(&tri).into()` then copy v0, e1, e2.
#[repr(C)]
#[derive(Clone, Copy, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayTri48 { pub v0: [f32; 3], pub p0: f32, pub e1: [f32; 3], pub p1: f32, pub e2: [f32; 3], pub p2: f32 }

/// `tray_ray_cost` of include/tray_cuda.h: one ray's nodes fetched, triangles tested, TLAS leaf entries and peak stack entries
#[repr(C)]
#[derive(Clone, Copy, Default, Debug, bytemuck::Pod, bytemuck::Zeroable)]
pub struct TrayRayCost { pub nodes: u32, pub tris: u32, pub instances: u32, pub stack: u32 }

#[repr(C)] pub struct TrayScene { _private: [u8; 0] }
#[repr(C)] pub struct TrayGroup { _private: [u8; 0] }

/// `tray_build_stats` of include/tray_cuda.h
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct TrayBuildStats {
    pub n_tris: u64, pub n_nodes: u64, pub ploc_iterations: u32, pub levels: u32,
    pub ms_upload: f32, pub ms_sort: f32, pub ms_ploc: f32, pub ms_collapse: f32, pub ms_total: f32,
    pub ms_reinsert: f32, pub reinsert_passes: u32, pub reinsert_moves: u32, pub sah_before: f32, pub sah_after: f32,
}

/// `tray_counters` of include/tray_cuda.h (the algorithmic bytes per ray come from these)
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct TrayCounters { pub rays: u64, pub nodes: u64, pub tris: u64, pub instances: u64, pub hits: u64 }

/// `tray_scene_info` of include/tray_cuda.h
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct TraySceneInfo {
    pub n_nodes: u64, pub n_tris: u64, pub tri_stride: u32, pub n_instances: u32, pub tlas_start: u32, pub is_tlas: u32,
    pub device: i32, pub sm_count: u32, pub device_bytes: u64, pub l2_bytes: u64, pub l2_persist_bytes: u64,
}

pub const RENDER_BOUNCE: u32 = 0x1;
pub const RENDER_RGBA: u32 = 0x2;
pub const RENDER_COUNTERS: u32 = 0x4;
pub const RENDER_KEEP_RAYS: u32 = 0x8;
pub const RENDER_ANYHIT_AO: u32 = 0x10;
pub const RENDER_OVERLAP: u32 = 0x20;
/// semantic switches of `tray_cuda_scene_set_variant` (include/tray_cuda.h TRAY_VARIANT_*)
pub const VARIANT_BOX_DIVIDE: u32 = 0x1;
pub const VARIANT_TIE_LAST: u32 = 0x2;
pub const VARIANT_BOX_TMIN_RAY: u32 = 0x4;
pub const VARIANT_ZERODIR_BOX_ONLY: u32 = 0x8;

extern "C" {
    pub fn tray_cuda_abi_version() -> u32;
    pub fn tray_cuda_scene_info(scene: *const TrayScene, out_info: *mut TraySceneInfo) -> c_int;
    pub fn tray_cuda_scene_exact_node_test(scene: *const TrayScene, out_exact: *mut c_int) -> c_int;
    pub fn tray_cuda_scene_build_tlas(tris9: *const f32, n_tris: u64, object_offsets: *const u64, n_objects: u32, tri_stride: u32,
        max_prims_per_leaf: u32, search_radius: u32, device: c_int, out: *mut *mut TrayScene, stats: *mut TrayBuildStats) -> c_int;
    pub fn tray_cuda_scene_download_instances(scene: *mut TrayScene, blas_offsets: *mut u32) -> c_int;
    pub fn tray_cuda_trace_device(scene: *mut TrayScene, d_rays: *const TrayRay, n: u64, d_hits: *mut TrayHit,
        stream: *mut c_void, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_trace_any_device(scene: *mut TrayScene, d_rays: *const TrayRay, n: u64, d_hits: *mut TrayHit,
        stream: *mut c_void, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_shard_pixels(width: u32, height: u32, shard_index: u32, shard_count: u32) -> u64;
    pub fn tray_cuda_frame_device_ptrs(scene: *mut TrayScene, d_primary: *mut *mut c_void, d_bounce: *mut *mut c_void,
        d_rgba: *mut *mut c_void) -> c_int;
    pub fn tray_cuda_untile_rgba(scene: *mut TrayScene, d_compact: *const c_void, width: u32, height: u32, shard_index: u32,
        shard_count: u32, d_frame: *mut c_void) -> c_int;
    pub fn tray_cuda_frame_alloc(device: c_int, bytes: u64, d_ptr: *mut *mut c_void) -> c_int;
    pub fn tray_cuda_frame_free(device: c_int, d_ptr: *mut c_void) -> c_int;
    pub fn tray_cuda_ipc_export(device: c_int, d_ptr: *mut c_void, handle: *mut u8) -> c_int;         // handle: [u8; 64]
    pub fn tray_cuda_ipc_open(device: c_int, handle: *const u8, d_ptr: *mut *mut c_void) -> c_int;
    pub fn tray_cuda_ipc_close(device: c_int, d_ptr: *mut c_void) -> c_int;
    pub fn tray_cuda_scene_set_frame_target(scene: *mut TrayScene, d_frame: *mut c_void) -> c_int;
    pub fn tray_cuda_scene_set_stream(scene: *mut TrayScene, stream: *mut c_void) -> c_int;
    pub fn tray_cuda_sync(scene: *mut TrayScene) -> c_int;
    pub fn tray_cuda_counters(scene: *mut TrayScene, primary: *mut TrayCounters, bounce: *mut TrayCounters) -> c_int;
    pub fn tray_cuda_set_counting(scene: *mut TrayScene, enabled: c_int) -> c_int;
    pub fn tray_cuda_trace_cost(scene: *mut TrayScene, rays: *const TrayRay, n: u64, any_hit: c_int, hits: *mut TrayHit,
        costs: *mut TrayRayCost, ms_kernel: *mut f32, ms_total: *mut f32) -> c_int;
    pub fn tray_cuda_trace_cost_device(scene: *mut TrayScene, d_rays: *const TrayRay, n: u64, any_hit: c_int, d_hits: *mut TrayHit,
        d_costs: *mut TrayRayCost, stream: *mut c_void, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_scene_set_ray_cost(scene: *mut TrayScene, enabled: c_int) -> c_int;
    pub fn tray_cuda_frame_download_cost(scene: *mut TrayScene, primary: *mut TrayRayCost, bounce: *mut TrayRayCost) -> c_int;
    pub fn tray_cuda_bandwidth_probe(device: c_int, bytes: u64, iters: c_int, out_gbs: *mut f32) -> c_int;
    pub fn tray_cuda_l1_gather_probe(device: c_int, bytes: u32, iters: c_int, out_gbs: *mut f32) -> c_int;
    pub fn tray_cuda_device_count() -> c_int;
    pub fn tray_cuda_last_error() -> *const c_char;
    pub fn tray_cuda_scene_create(nodes: *const c_void, n_nodes: u64, tris: *const c_void, n_tris: u64, tri_stride: u32,
        blas_offsets: *const u32, n_instances: u32, tlas_start: u32, device: c_int, out: *mut *mut TrayScene) -> c_int;
    pub fn tray_cuda_scene_destroy(scene: *mut TrayScene);
    pub fn tray_cuda_trace(scene: *mut TrayScene, rays: *const TrayRay, n: u64, hits: *mut TrayHit,
        ms_kernel: *mut f32, ms_total: *mut f32) -> c_int;
    pub fn tray_cuda_trace_any(scene: *mut TrayScene, rays: *const TrayRay, n: u64, hits: *mut TrayHit,
        ms_kernel: *mut f32, ms_total: *mut f32) -> c_int;
    pub fn tray_cuda_render(scene: *mut TrayScene, view: *const TrayView, width: u32, height: u32, frame_count: u32,
        flags: u32, shard_index: u32, shard_count: u32, ms_primary: *mut f32, ms_bounce: *mut f32) -> c_int;
    pub fn tray_cuda_render_timed(scene: *mut TrayScene, view: *const TrayView, width: u32, height: u32, frame_count: u32,
        flags: u32, shard_index: u32, shard_count: u32, ms_frame: *mut f32) -> c_int;
    pub fn tray_cuda_frame_readback_begin(scene: *mut TrayScene, rgba_host: *mut u8, slot: u32) -> c_int;
    pub fn tray_cuda_frame_readback_wait(scene: *mut TrayScene, slot: u32) -> c_int;
    pub fn tray_cuda_scene_build(tris9: *const f32, n_tris: u64, tri_stride: u32, max_prims_per_leaf: u32, search_radius: u32,
        device: c_int, out: *mut *mut TrayScene, stats: *mut TrayBuildStats) -> c_int;
    pub fn tray_cuda_scene_download(scene: *mut TrayScene, nodes: *mut c_void, tris: *mut c_void, prim_indices: *mut u32) -> c_int;
    // same tree, new vertex positions (n_tris x 9 f32 in the scene's triangle order); synchronous, after every frame enqueued
    pub fn tray_cuda_scene_refit(scene: *mut TrayScene, tris9: *const f32, n_tris: u64, ms_refit: *mut f32) -> c_int;
    pub fn tray_cuda_scene_refit_device(scene: *mut TrayScene, d_tris9: *const f32, n_tris: u64, stream: *mut c_void,
        ms_refit: *mut f32) -> c_int;
    // two-level scenes whose objects move as a whole: refit every BLAS, rebuild the TLAS over their boxes; synchronous as the refit
    pub fn tray_cuda_scene_refit_rebuild_tlas(scene: *mut TrayScene, tris9: *const f32, n_tris: u64, max_prims_per_leaf: u32,
        search_radius: u32, ms: *mut f32) -> c_int;
    pub fn tray_cuda_scene_refit_rebuild_tlas_device(scene: *mut TrayScene, d_tris9: *const f32, n_tris: u64, max_prims_per_leaf: u32,
        search_radius: u32, stream: *mut c_void, ms: *mut f32) -> c_int;
    // instances: BLAS placed by row-major 3x4 object_to_world transforms, only the TLAS rebuilt; synchronous as the refit
    pub fn tray_cuda_scene_set_instances(scene: *mut TrayScene, blas_roots: *const u32, object_to_world: *const f32, n_instances: u32,
        max_prims_per_leaf: u32, search_radius: u32, ms: *mut f32) -> c_int;
    pub fn tray_cuda_scene_download_instance_xforms(scene: *mut TrayScene, leaf_instance: *mut u32, world_to_object: *mut f32) -> c_int;
    pub fn tray_cuda_trace_instance(scene: *mut TrayScene, rays: *const TrayRay, n: u64, any_hit: c_int, hits: *mut TrayHit,
        instance_ids: *mut u32, ms_kernel: *mut f32, ms_total: *mut f32) -> c_int;
    pub fn tray_cuda_trace_instance_device(scene: *mut TrayScene, d_rays: *const TrayRay, n: u64, any_hit: c_int, d_hits: *mut TrayHit,
        d_instance_ids: *mut u32, stream: *mut c_void, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_frame_download_instance(scene: *mut TrayScene, primary: *mut u32, bounce: *mut u32) -> c_int;
    // hit attributes: u, v and the geometric normal of each hit, as the triangle test computed them
    pub fn tray_cuda_hit_attributes(scene: *mut TrayScene, rays: *const TrayRay, hits: *const TrayHit, instance_ids: *const u32, n: u64,
        attrs: *mut TrayHitAttr, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_hit_attributes_device(scene: *mut TrayScene, d_rays: *const TrayRay, d_hits: *const TrayHit, d_instance_ids: *const u32,
        n: u64, d_attrs: *mut TrayHitAttr, stream: *mut c_void, ms_kernel: *mut f32) -> c_int;
    pub fn tray_cuda_frame_download_attributes(scene: *mut TrayScene, primary: *mut TrayHitAttr, bounce: *mut TrayHitAttr) -> c_int;
    pub fn tray_cuda_frame_download(scene: *mut TrayScene, primary: *mut TrayHit, bounce: *mut TrayHit,
        bounce_rays: *mut TrayRay, rgba: *mut u8) -> c_int;
    pub fn tray_cuda_scene_set_variant(scene: *mut TrayScene, variant_flags: u32) -> c_int;
    pub fn tray_cuda_shard_items(width: u32, height: u32, shard_index: u32, shard_count: u32) -> u64;
    pub fn tray_cuda_scene_set_frames_in_flight(scene: *mut TrayScene, n: u32) -> c_int;
    pub fn tray_cuda_scene_fence(scene: *mut TrayScene, stream: *mut c_void) -> c_int;
    pub fn tray_cuda_scene_after(scene: *mut TrayScene, stream: *mut c_void) -> c_int;
    pub fn tray_cuda_frame_push(scene: *mut TrayScene, d_dst: *mut c_void) -> c_int;
    pub fn tray_cuda_untile_shards(scene: *mut TrayScene, d_staging: *const c_void, width: u32, height: u32, shards: u32,
        d_frame: *mut c_void) -> c_int;
    pub fn tray_cuda_frame_signal(scene: *mut TrayScene, d_flag: *mut c_void, value: u32) -> c_int;
    pub fn tray_cuda_frame_wait_flag(scene: *mut TrayScene, d_flag: *const c_void, value: u32, before_next_frame: c_int) -> c_int;
    pub fn tray_cuda_scene_frame_stream(scene: *mut TrayScene, which: c_int, stream: *mut *mut c_void) -> c_int;
    pub fn tray_cuda_scene_set_geometry_offsets(scene: *mut TrayScene, tri_offsets: *const u32, n_geometries: u32) -> c_int;
    pub fn tray_cuda_hits_to_geometry(scene: *mut TrayScene, hits: *const TrayHit, n: u64, geometry_id: *mut u32,
        primitive_id: *mut u32) -> c_int;
    pub fn tray_cuda_group_create(nodes: *const c_void, n_nodes: u64, tris: *const c_void, n_tris: u64, tri_stride: u32,
        blas_offsets: *const u32, n_instances: u32, tlas_start: u32, devices: *const c_int, n_devices: c_int,
        out: *mut *mut TrayGroup) -> c_int;
    pub fn tray_cuda_group_destroy(group: *mut TrayGroup);
    pub fn tray_cuda_group_size(group: *const TrayGroup) -> c_int;
    pub fn tray_cuda_group_scene(group: *mut TrayGroup, i: c_int, out_scene: *mut *mut TrayScene) -> c_int;
    pub fn tray_cuda_group_set_frames_in_flight(group: *mut TrayGroup, n: u32) -> c_int;
    pub fn tray_cuda_group_set_exchange(group: *mut TrayGroup, push: c_int) -> c_int;
    pub fn tray_cuda_group_render(group: *mut TrayGroup, view: *const TrayView, width: u32, height: u32, frame_count: u32,
        flags: u32) -> c_int;
    pub fn tray_cuda_group_render_timed(group: *mut TrayGroup, view: *const TrayView, width: u32, height: u32, frame_count: u32,
        flags: u32, ms_frame: *mut f32) -> c_int;
    pub fn tray_cuda_group_readback_begin(group: *mut TrayGroup, rgba_host: *mut u8, slot: u32) -> c_int;
    pub fn tray_cuda_group_readback_wait(group: *mut TrayGroup, slot: u32) -> c_int;
    pub fn tray_cuda_group_frame_ptr(group: *mut TrayGroup, d_frame: *mut *mut c_void) -> c_int;
    pub fn tray_cuda_group_sync(group: *mut TrayGroup) -> c_int;
    pub fn tray_cuda_start_multi(devices: *const c_int, n_devices: c_int, bvh: *const c_void, bvh_len: u64, inst: *const c_void,
        inst_len: u64, tris: *const c_void, tri_len: u64, tri_stride: u32, tlas_start: u32, use_tlas: c_int,
        view: *const TrayView, width: u32, height: u32, render_time_s: f32, benchmark: c_int, animate: c_int,
        out_min_ms: *mut f32, out_mean_ms: *mut f32, out_frames: *mut u32) -> c_int;
    pub fn tray_cuda_start(bvh: *const c_void, bvh_len: u64, inst: *const c_void, inst_len: u64, tris: *const c_void,
        tri_len: u64, tri_stride: u32, tlas_start: u32, use_tlas: c_int, view: *const TrayView, width: u32, height: u32,
        render_time_s: f32, benchmark: c_int, animate: c_int, device: c_int,
        out_min_ms: *mut f32, out_mean_ms: *mut f32, out_frames: *mut u32) -> c_int;
}

fn check(rc: c_int) {
    if rc != 0 {
        // the reference panics on every error (src/main.rs:178-180, rt_gpu_software.rs:99,124,307)
        let msg = unsafe { CStr::from_ptr(tray_cuda_last_error()) }.to_string_lossy().into_owned();
        panic!("tray_cuda error {rc}: {msg}");
    }
}

pub struct StartArgs<'a> {
    pub bvh_bytes: &'a [u8], pub instance_bytes: &'a [u8], pub tri_bytes: &'a [u8], pub tlas_start: u32, pub use_tlas: bool,
    pub view: TrayView, pub width: u32, pub height: u32, pub render_time: f32, pub benchmark: bool, pub animate: bool,
    /// bytes per triangle record in `tri_bytes`: 48 / 64 (f32 `RtTriangle`, the parity path) or 24 (`RtCompressedTriangle`)
    pub tri_stride: u32,
    /// CUDA devices to render on; one entry = `tray_cuda_start`, several = `tray_cuda_start_multi` (tiles dealt round-robin)
    pub devices: &'a [i32],
}

/// Drop-in for `rt_gpu_software::start`: returns the min frame time in ms.
pub fn start(a: StartArgs) -> f32 {
    let (mut min_ms, mut mean_ms, mut frames) = (0f32, 0f32, 0u32);
    let devices: &[i32] = if a.devices.is_empty() { &[0] } else { a.devices };
    check(unsafe {
        if devices.len() == 1 {
            tray_cuda_start(a.bvh_bytes.as_ptr().cast(), a.bvh_bytes.len() as u64, a.instance_bytes.as_ptr().cast(),
                a.instance_bytes.len() as u64, a.tri_bytes.as_ptr().cast(), a.tri_bytes.len() as u64, a.tri_stride, a.tlas_start,
                a.use_tlas as c_int, &a.view, a.width, a.height, a.render_time, a.benchmark as c_int, a.animate as c_int,
                devices[0], &mut min_ms, &mut mean_ms, &mut frames)
        } else {
            tray_cuda_start_multi(devices.as_ptr(), devices.len() as c_int, a.bvh_bytes.as_ptr().cast(), a.bvh_bytes.len() as u64,
                a.instance_bytes.as_ptr().cast(), a.instance_bytes.len() as u64, a.tri_bytes.as_ptr().cast(),
                a.tri_bytes.len() as u64, a.tri_stride, a.tlas_start, a.use_tlas as c_int, &a.view, a.width, a.height,
                a.render_time, a.benchmark as c_int, a.animate as c_int, &mut min_ms, &mut mean_ms, &mut frames)
        }
    });
    min_ms
}

/// Owning handle of a device-resident scene: the batch-grain face of `Traversable` (traversable/src/lib.rs:13-28).
/// Like the reference, every error panics.
pub struct Scene { raw: *mut TrayScene }

impl Scene {
    /// Upload the buffers `cwbvh_gpu_runner` builds (src/rt_gpu/mod.rs:16-112); `blas_offsets` empty = single-level.
    pub fn new(bvh_bytes: &[u8], tri_bytes: &[u8], tri_stride: u32, blas_offsets: &[u32], tlas_start: u32, device: i32) -> Scene {
        let mut raw = std::ptr::null_mut();
        check(unsafe {
            tray_cuda_scene_create(bvh_bytes.as_ptr().cast(), (bvh_bytes.len() / 80) as u64, tri_bytes.as_ptr().cast(),
                (tri_bytes.len() / tri_stride as usize) as u64, tri_stride,
                if blas_offsets.is_empty() { std::ptr::null() } else { blas_offsets.as_ptr() }, blas_offsets.len() as u32,
                tlas_start, device, &mut raw)
        });
        Scene { raw }
    }

    /// Build the CWBVH on the device from a triangle soup (9 floats per triangle), the step `cwbvh_from_tris` does on the CPU.
    pub fn build(tris9: &[f32], max_prims_per_leaf: u32, search_radius: u32, device: i32) -> (Scene, TrayBuildStats) {
        let (mut raw, mut stats) = (std::ptr::null_mut(), TrayBuildStats::default());
        check(unsafe { tray_cuda_scene_build(tris9.as_ptr(), (tris9.len() / 9) as u64, 48, max_prims_per_leaf, search_radius, device, &mut raw, &mut stats) });
        (Scene { raw }, stats)
    }

    /// One BLAS per object (`object_offsets[k]..object_offsets[k + 1]` are object k's triangles) plus a TLAS: `--tlas`.
    pub fn build_tlas(tris9: &[f32], object_offsets: &[u64], max_prims_per_leaf: u32, search_radius: u32, device: i32) -> (Scene, TrayBuildStats) {
        let (mut raw, mut stats) = (std::ptr::null_mut(), TrayBuildStats::default());
        check(unsafe {
            tray_cuda_scene_build_tlas(tris9.as_ptr(), (tris9.len() / 9) as u64, object_offsets.as_ptr(), (object_offsets.len() - 1) as u32,
                48, max_prims_per_leaf, search_radius, device, &mut raw, &mut stats)
        });
        (Scene { raw }, stats)
    }

    pub fn info(&self) -> TraySceneInfo {
        let mut i = TraySceneInfo::default();
        check(unsafe { tray_cuda_scene_info(self.raw, &mut i) });
        i
    }

    /// Closest hit per ray (`Traversable::traverse` for a batch); `any_hit` stops each ray at its first accepted triangle.
    pub fn traverse(&mut self, rays: &[TrayRay], any_hit: bool) -> Vec<TrayHit> {
        let mut hits = vec![TrayHit { t: f32::INFINITY, prim: u32::MAX }; rays.len()];
        let f = if any_hit { tray_cuda_trace_any } else { tray_cuda_trace };
        check(unsafe { f(self.raw, rays.as_ptr(), rays.len() as u64, hits.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut()) });
        hits
    }

    /// Place BLAS by transforms: instance k is the BLAS rooted at node `blas_roots[k]`, placed by the row-major 3x4
    /// `object_to_world[k]`; only the TLAS is built.  Returns the call's ms (upload of the transforms to the last TLAS write).
    pub fn set_instances(&mut self, blas_roots: &[u32], object_to_world: &[[f32; 12]], max_prims_per_leaf: u32, search_radius: u32) -> f32 {
        assert_eq!(blas_roots.len(), object_to_world.len(), "one transform per instance");
        let mut ms = 0f32;
        check(unsafe {
            tray_cuda_scene_set_instances(self.raw, blas_roots.as_ptr(), object_to_world.as_ptr().cast(), blas_roots.len() as u32,
                max_prims_per_leaf, search_radius, &mut ms)
        });
        ms
    }

    /// Closest (or any) hit per ray of an instanced scene, with the instance of every hit (u32::MAX for a miss).
    pub fn traverse_instance(&mut self, rays: &[TrayRay], any_hit: bool) -> (Vec<TrayHit>, Vec<u32>) {
        let mut hits = vec![TrayHit { t: f32::INFINITY, prim: u32::MAX }; rays.len()];
        let mut ids = vec![u32::MAX; rays.len()];
        check(unsafe {
            tray_cuda_trace_instance(self.raw, rays.as_ptr(), rays.len() as u64, any_hit as c_int, hits.as_mut_ptr(), ids.as_mut_ptr(),
                std::ptr::null_mut(), std::ptr::null_mut())
        });
        (hits, ids)
    }

    /// u, v and the world-space geometric normal of every hit on its ray (`hits` and `instance_ids` as `traverse` or
    /// `traverse_instance` returned them; `instance_ids` is required on an instanced scene and must be `None` on any other).
    pub fn hit_attributes(&mut self, rays: &[TrayRay], hits: &[TrayHit], instance_ids: Option<&[u32]>) -> Vec<TrayHitAttr> {
        assert_eq!(rays.len(), hits.len(), "one hit per ray");
        if let Some(ids) = instance_ids { assert_eq!(ids.len(), hits.len(), "one instance id per hit"); }
        let mut attrs = vec![TrayHitAttr { u: f32::NAN, v: f32::NAN, ng: [f32::NAN; 3] }; hits.len()];
        check(unsafe {
            tray_cuda_hit_attributes(self.raw, rays.as_ptr(), hits.as_ptr(), instance_ids.map_or(std::ptr::null(), |i| i.as_ptr()),
                hits.len() as u64, attrs.as_mut_ptr(), std::ptr::null_mut())
        });
        attrs
    }

    /// The last frame's hit attributes, row-major (width * height each): (primary, bounce); `bounce` needs a frame rendered with
    /// RENDER_BOUNCE.  Panics when the scene was refit, re-instanced or given other variants since that frame.
    pub fn download_attributes(&mut self, width: u32, height: u32, bounce: bool) -> (Vec<TrayHitAttr>, Vec<TrayHitAttr>) {
        let n = width as usize * height as usize;
        let nan = TrayHitAttr { u: f32::NAN, v: f32::NAN, ng: [f32::NAN; 3] };
        let (mut p, mut b) = (vec![nan; n], if bounce { vec![nan; n] } else { Vec::new() });
        check(unsafe {
            tray_cuda_frame_download_attributes(self.raw, p.as_mut_ptr(), if bounce { b.as_mut_ptr() } else { std::ptr::null_mut() })
        });
        (p, b)
    }

    /// One frame (primary + bounce rays) of shard `shard` of `shards`; returns (ms primary, ms bounce) of the kernels.
    pub fn render(&mut self, view: &TrayView, width: u32, height: u32, frame_count: u32, flags: u32, shard: u32, shards: u32) -> (f32, f32) {
        let (mut a, mut b) = (0f32, 0f32);
        check(unsafe { tray_cuda_render(self.raw, view, width, height, frame_count, flags, shard, shards, &mut a, &mut b) });
        (a, b)
    }

    /// RGBA8 of the last frame, row-major (the reference's PNG input, rt_cpu.rs:102-112).
    pub fn download_rgba(&mut self, width: u32, height: u32) -> Vec<u8> {
        let mut px = vec![0u8; width as usize * height as usize * 4];
        check(unsafe { tray_cuda_frame_download(self.raw, std::ptr::null_mut(), std::ptr::null_mut(), std::ptr::null_mut(), px.as_mut_ptr()) });
        px
    }

    /// CPU-style hit records of a `--tlas` scene (`CwBvhTlasScene::traverse`, src/cwbvh.rs:144-166): `tri_offsets` is the runner's
    /// running `tri_offset` per object (src/rt_gpu/mod.rs:45-47) plus the total; returns (geometry_id, primitive_id) per hit.
    pub fn set_geometry_offsets(&mut self, tri_offsets: &[u32]) {
        check(unsafe { tray_cuda_scene_set_geometry_offsets(self.raw, tri_offsets.as_ptr(), (tri_offsets.len().max(1) - 1) as u32) });
    }
    pub fn hits_to_geometry(&mut self, hits: &[TrayHit]) -> (Vec<u32>, Vec<u32>) {
        let (mut g, mut p) = (vec![u32::MAX; hits.len()], vec![u32::MAX; hits.len()]);
        check(unsafe { tray_cuda_hits_to_geometry(self.raw, hits.as_ptr(), hits.len() as u64, g.as_mut_ptr(), p.as_mut_ptr()) });
        (g, p)
    }

    pub fn counters(&mut self) -> (TrayCounters, TrayCounters) {
        let (mut p, mut b) = (TrayCounters::default(), TrayCounters::default());
        check(unsafe { tray_cuda_counters(self.raw, &mut p, &mut b) });
        (p, b)
    }

    pub fn as_raw(&self) -> *mut TrayScene { self.raw }
}

impl Drop for Scene {
    fn drop(&mut self) { unsafe { tray_cuda_scene_destroy(self.raw) } }
}
