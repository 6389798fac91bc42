// tray_cuda.cu — the C ABI of include/tray_cuda.h over the sm_100a kernels in traverse.cuh.
// No CPU fallback exists: without a CUDA device every compute entry point fails with TRAY_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

#include "build_gpu.h"
#include "host_copy.h"
#include "traverse.cuh"

static_assert(sizeof(tray_cwbvh_node) == 80, "CwBvhNode is 80 bytes (bvh_embree_to_cwbvh.rs:91, rt_gpu/mod.rs:70)");
static_assert(sizeof(tray_tri48) == 48 && sizeof(tray_tri64) == 64 && sizeof(tray_tri24) == 24, "triangle record strides");
static_assert(sizeof(tray_ray) == 32 && sizeof(tray_hit) == 8, "ray / hit records");
static_assert(sizeof(tray_ray_cost) == 16 && alignof(tray_ray_cost) == 4, "ray cost record: one 16-byte store per ray");
static_assert(sizeof(tray_view) == 160, "ViewUniform is padded to 160 bytes (main.rs:589-597)");

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(TRAY_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// whether a scene takes the unfused node test everywhere: some node scale is >= 2^40 (tray::node_needs_exact), or
// TRAY_CUDA_FORCE_EXACT asks for it
bool scene_force_exact(bool nodes_need_it) { return env_int("TRAY_CUDA_FORCE_EXACT", 0) != 0 || nodes_need_it; }

}  // namespace

// Everything one frame in flight owns: its compact (tile-ordered) buffers, its work cursors and its stream.  Slot 0 runs on
// tray_scene::stream (the scene's own, or the caller's: tray_cuda_scene_set_stream), slot 1 on a stream of its own, so that
// the kernels of frame k+1 fill the SM slots the drain phase of frame k leaves empty.
struct FrameSlot {
    cudaStream_t own_stream = nullptr;       // slot 1 only
    unsigned long long* d_cursor = nullptr;  // cursor block (tray::CURSOR_WORDS)
    uint32_t* d_units = nullptr;             // FRAME kernel: cursor over the 32-item groups of bounce work
    cudaEvent_t ev[4] = { nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t done = nullptr;              // recorded behind the frame's last launch (fences, group completion)
    uint64_t f_cap = 0;
    bool f_has_bounce = false, f_has_rgba = false, f_has_rays = false;
    uchar4* f_target = nullptr;              // the frame target the last frame was rendered into (NULL: compact d_rgba)
    tray_hit* d_primary = nullptr; tray_hit* d_bounce = nullptr; uchar4* d_rgba = nullptr;
    tray_ray* d_prays = nullptr;             // generated primary rays, local order
    tray_ray* d_brays = nullptr;             // generated bounce rays, COMPACT (hit pixels only)
    uint32_t* d_bitem = nullptr;             // local item of compact bounce ray i
    tray_ray* d_brays_item = nullptr;        // optional: bounce rays by local item (TRAY_RENDER_KEEP_RAYS)
    tray_ray_cost* d_cost = nullptr;         // optional: ray costs by local item, 2 x f_cap: primary [0, n_items), bounce from n_items
    bool f_has_cost = false;                 // the last frame kept ray costs (tray_cuda_scene_set_ray_cost + TRAY_RENDER_COUNTERS)
    uint32_t* d_flag = nullptr;              // the device error word of this slot's launches (a word of tray_scene::d_overflow)
    tray::FrameParams last_frame{};          // width 0: no frame rendered yet
};

struct tray_scene {
    int device = 0;
    int sm_count = 0;
    uint64_t n_nodes = 0, n_tris = 0;
    uint32_t tri_stride = 48, n_instances = 0, tlas_start = 0;
    bool tlas = false;
    bool force_exact = false;                // some node scale >= 2^40: 2^23 * adj_inv could overflow in the fused node test
    uint4* d_nodes = nullptr;
    uint4* d_tris = nullptr;
    uint32_t* d_blas = nullptr;
    uint32_t* d_prim_indices = nullptr;      // BVH slot -> input triangle (scenes made by tray_cuda_scene_build)
    tray_build::RefitTopology* refit = nullptr;   // the topology walk of the first tray_cuda_scene_refit, kept for the next
    uint32_t* d_geom_offsets = nullptr; uint32_t n_geometries = 0;   // first global triangle of BLAS / object g (tray_cuda_scene_set_geometry_offsets)
    unsigned long long* d_cursor = nullptr;     // cursor block of batch traces (tray::CURSOR_WORDS)
    // device error words (TraceParams::overflow): [0] batch traces, [1 + k] the launches of frame slot k — one word per slot, so
    // that a frame's error is reported for that frame and cleared in the order of that slot's stream
    uint32_t* d_overflow = nullptr;
    cudaStream_t stream = nullptr;          // the stream work is enqueued on
    cudaStream_t own_stream = nullptr;      // created with the scene
    cudaEvent_t ev[2] = { nullptr, nullptr };
    bool have_window = false;                // persisting-L2 access-policy window over the node array, applied per launch
    cudaAccessPolicyWindow window{};
    uint64_t device_bytes = 0, l2_bytes = 0, l2_persist = 0;
    bool counting = false;                   // tray_cuda_set_counting: batch traces count (a render counts with TRAY_RENDER_COUNTERS alone)
    bool ray_cost = false;                   // tray_cuda_scene_set_ray_cost: counted renders keep every ray's cost
    uint32_t variant = 0;                    // TRAY_VARIANT_* (tray_cuda_scene_set_variant): the MODE 1 kernels
    uint32_t refill_min = 6, tri_weight = 3, gen_min = 4;
    bool overlap_default = false;            // TRAY_CUDA_OVERLAP=1: tray_cuda_render always takes the one-launch frame kernel
    int blocks_per_sm[3] = { 0, 0, 0 };      // resident CTAs per SM of the lane kernel [0], the MODE 1 kernel [1], the counting lane kernel [2]
    // ray-batch staging
    tray_ray* d_rays = nullptr; tray_hit* d_hits = nullptr; uint64_t batch_cap = 0;
    tray_ray_cost* d_costs = nullptr; uint64_t cost_cap = 0;   // tray_cuda_trace_cost: allocated on first use
    // host <-> device pipeline of tray_cuda_trace: two pinned staging slots per direction, copy streams, events
    tray_ray* h_rays[2] = { nullptr, nullptr }; tray_hit* h_hits[2] = { nullptr, nullptr };
    tray_ray_cost* h_costs[2] = { nullptr, nullptr };          // pinned cost slots, allocated by the first pipelined cost call
    cudaStream_t s_in = nullptr, s_out = nullptr; bool pipeline_ready = false;
    cudaEvent_t e_in[2] = { nullptr, nullptr }, e_k[2] = { nullptr, nullptr }, e_out[2] = { nullptr, nullptr };
    // frame state: one FrameSlot per frame in flight (tray_cuda_scene_set_frames_in_flight); `cur` = the slot of the last frame
    FrameSlot slot[TRAY_MAX_FRAMES_IN_FLIGHT];
    int n_slots = 1, cur = 0;
    void* d_untiled = nullptr; uint64_t untiled_cap = 0;
    // asynchronous RGBA readback: double-buffered row-major staging, copies on their own stream
    cudaStream_t copy_stream = nullptr;
    uchar4* d_stage[TRAY_READBACK_SLOTS] = {}; uint64_t stage_cap[TRAY_READBACK_SLOTS] = {}; bool stage_busy[TRAY_READBACK_SLOTS] = {};
    cudaEvent_t ev_untiled[TRAY_READBACK_SLOTS] = {}, ev_copied[TRAY_READBACK_SLOTS] = {};
    cudaEvent_t ev_after = nullptr;          // tray_cuda_scene_after
    uint32_t* h_flag = nullptr;              // pinned, one word per staging slot: the error word of the frame staging slot i was filled from
    uchar4* frame_target = nullptr;          // borrowed: row-major RGBA8 frame (this or a peer device), see tray_cuda_scene_set_frame_target
    tray_counters cnt_primary{}, cnt_bounce{};
};

namespace {

using namespace tray;

void free_pipeline(tray_scene* s) {
    for (int i = 0; i < 2; i++) {
        if (s->h_rays[i]) cudaFreeHost(s->h_rays[i]);
        if (s->h_hits[i]) cudaFreeHost(s->h_hits[i]);
        if (s->h_costs[i]) cudaFreeHost(s->h_costs[i]);
        s->h_costs[i] = nullptr;
        if (s->e_in[i]) cudaEventDestroy(s->e_in[i]);
        if (s->e_k[i]) cudaEventDestroy(s->e_k[i]);
        if (s->e_out[i]) cudaEventDestroy(s->e_out[i]);
        s->h_rays[i] = nullptr; s->h_hits[i] = nullptr; s->e_in[i] = s->e_k[i] = s->e_out[i] = nullptr;
    }
    if (s->s_in) cudaStreamDestroy(s->s_in);
    if (s->s_out) cudaStreamDestroy(s->s_out);
    s->s_in = s->s_out = nullptr;
    s->pipeline_ready = false;
}


typedef void (*kernel_fn)(const TraceParams);

// The trace_kernel instantiation of a launch. MODE 0: every (tlas, count, stride) x {closest hit, any hit, frame}.
// MODE 1 (variant) exists without counters only, so it ignores `count` (launch() rejects that combination).
template <bool TLAS, bool COUNT, int STRIDE>
kernel_fn pick_kernel(bool anyhit, bool frame, bool variant) {
    if (variant) return (kernel_fn)trace_kernel<TLAS, false, STRIDE, false, false, 1>;
    if (frame) return (kernel_fn)trace_kernel<TLAS, COUNT, STRIDE, false, true>;
    return anyhit ? (kernel_fn)trace_kernel<TLAS, COUNT, STRIDE, true> : (kernel_fn)trace_kernel<TLAS, COUNT, STRIDE, false>;
}
template <bool TLAS, bool COUNT>
kernel_fn pick_kernel(uint32_t stride, bool anyhit, bool frame, bool variant) {
    return stride == 64 ? pick_kernel<TLAS, COUNT, 64>(anyhit, frame, variant)
         : stride == 24 ? pick_kernel<TLAS, COUNT, 24>(anyhit, frame, variant) : pick_kernel<TLAS, COUNT, 48>(anyhit, frame, variant);
}
kernel_fn pick_kernel(bool tlas, bool count, uint32_t stride, bool anyhit, bool frame, bool variant) {
    if (tlas) return count ? pick_kernel<true, true>(stride, anyhit, frame, variant) : pick_kernel<true, false>(stride, anyhit, frame, variant);
    return count ? pick_kernel<false, true>(stride, anyhit, frame, variant) : pick_kernel<false, false>(stride, anyhit, frame, variant);
}

uint64_t local_items(uint32_t w, uint32_t h, uint32_t shard, uint32_t shards) {
    const uint64_t tiles = (uint64_t)((w + 31) / 32) * ((h + 7) / 8);
    if (shard >= tiles) return 0;
    return ((tiles - shard + shards - 1) / shards) * 256ull;
}

void base_params(const tray_scene* s, TraceParams& P) {
    memset(&P, 0, sizeof P);
    P.nodes = s->d_nodes; P.tris = s->d_tris; P.blas_offsets = s->d_blas; P.tlas_start = s->tlas_start;
    P.cursor = (uint32_t*)s->d_cursor; P.overflow = s->d_overflow;
    P.refill_min = s->refill_min; P.tri_weight = s->tri_weight; P.k4b = 0x4B000000u; P.force_exact = s->force_exact ? 1u : 0u;
    P.variant = s->variant; P.one = 1u;
}

const char* const VARIANT_REFUSAL = "semantic variants (tray_cuda_scene_set_variant) cover the closest-hit kernels without counters only";

// one launch: reset the cursor, run the persistent grid (sized to the chip, or to the work if that is smaller)
// `cur` = the cursor block the launch works on; its counters go to slot `counter_slot` (and the next, for the frame kernel).
// `count`: the counting kernels (tray_scene::counting for batch traces, TRAY_RENDER_COUNTERS for the launches of one frame)
int launch(tray_scene* s, TraceParams& P, cudaStream_t st, unsigned long long* cur, int counter_slot, bool count, bool anyhit = false, bool keep_counters = false, bool frame = false) {
    if (s->variant && (anyhit || frame || count)) return fail(TRAY_ERR_ARG, "%s", VARIANT_REFUSAL);
    kernel_fn k = pick_kernel(s->tlas, count, s->tri_stride, anyhit, frame, s->variant != 0);
    int& bps = s->blocks_per_sm[s->variant ? 1 : count ? 2 : 0];
    if (bps == 0) {
        int nb = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, BLOCK_THREADS, 0));
        bps = nb > 0 ? nb : 1;
    }
    P.cursor = (uint32_t*)cur;
    P.counters = cur + CURSOR_COUNTERS + N_COUNTERS * counter_slot;
    CU(cudaMemsetAsync(cur, 0, sizeof(unsigned long long), st));
    if (count && !keep_counters) CU(cudaMemsetAsync(P.counters, 0, (frame ? 2 : 1) * N_COUNTERS * sizeof(unsigned long long), st));
    const uint64_t blocks_needed = ((uint64_t)P.n_work + BLOCK_THREADS - 1) / BLOCK_THREADS;
    uint64_t grid = (uint64_t)s->sm_count * bps;
    if (blocks_needed < grid) grid = blocks_needed;
    if (grid == 0) return TRAY_OK;
    // the persisting-L2 window over the node array travels with the launch, so it holds on any stream
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)BLOCK_THREADS); cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (s->have_window) {
        attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[0].val.accessPolicyWindow = s->window;
        cfg.attrs = attr; cfg.numAttrs = 1;
    }
    void* args[1] = { (void*)&P };
    CU(cudaLaunchKernelExC(&cfg, (const void*)k, args));
    return TRAY_OK;
}

cudaStream_t slot_stream(const tray_scene* s, int k) { return k == 0 ? s->stream : s->slot[k].own_stream; }
int next_slot(const tray_scene* s) { return (s->cur + 1) % s->n_slots; }     // the slot the next tray_cuda_render takes
// waits for the scene stream and the scene's own frame streams (slot 0 runs on tray_scene::stream), in the order asked for
int sync_streams(const tray_scene* s, bool scene_stream_first) {
    if (scene_stream_first) CU(cudaStreamSynchronize(s->stream));
    for (int k = 1; k < TRAY_MAX_FRAMES_IN_FLIGHT; k++) CU(cudaStreamSynchronize(s->slot[k].own_stream));
    if (!scene_stream_first) CU(cudaStreamSynchronize(s->stream));
    return TRAY_OK;
}

// the per-frame buffers of a slot (not its cursor block); the caller has synchronised the slot's stream
void free_frame_buffers(FrameSlot& f) {
    cudaFree(f.d_primary); cudaFree(f.d_bounce); cudaFree(f.d_brays); cudaFree(f.d_rgba);
    cudaFree(f.d_prays); cudaFree(f.d_bitem); cudaFree(f.d_brays_item); cudaFree(f.d_cost);
    f.d_primary = nullptr; f.d_bounce = nullptr; f.d_brays = nullptr; f.d_rgba = nullptr;
    f.d_prays = nullptr; f.d_bitem = nullptr; f.d_brays_item = nullptr; f.d_cost = nullptr; f.f_cap = 0;
}

int check_tri_stride(uint32_t tri_stride) {
    if (tri_stride != 48 && tri_stride != 64 && tri_stride != 24) return fail(TRAY_ERR_ARG, "tri_stride must be 48, 64 or 24 (got %u)", tri_stride);
    return TRAY_OK;
}
// after the argument checks, so that a bad argument is reported as such on a machine without a GPU too
int select_device(int device) {
    const int ndev = tray_cuda_device_count();
    if (ndev == 0) return fail(TRAY_ERR_NO_DEVICE, "no CUDA device (tray_cuda has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(TRAY_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);
    CU(cudaSetDevice(device));
    return TRAY_OK;
}

void frame_params(FrameParams& F, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t shard, uint32_t shards) {
    memset(&F, 0, sizeof F);
    if (view) F.view = *view;
    F.width = w; F.height = h; F.frame_count = frame_count;
    F.shard_index = shard; F.shard_count = shards; F.tiles_x = (w + 31) / 32;
    F.n_items = (uint32_t)local_items(w, h, shard, shards);
}

int read_counters(const unsigned long long* cur, cudaStream_t st, int slot, tray_counters* out) {
    unsigned long long c[N_COUNTERS];
    CU(cudaMemcpyAsync(c, cur + CURSOR_COUNTERS + N_COUNTERS * slot, sizeof c, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    out->rays = c[0]; out->nodes = c[1]; out->tris = c[2]; out->instances = c[3]; out->hits = c[4];
    return TRAY_OK;
}

// An empty scene is uploaded as one zeroed placeholder root (scene_create_impl), which every ray fetches and misses.  It is not
// a node of the scene: its visits are not counted, as the reference visits no node there.
void drop_placeholder_root(tray_scene* s) {
    if (s->n_nodes == 0) { s->cnt_primary.nodes = 0; s->cnt_bounce.nodes = 0; }
}
// The same for the cost records of n rays at d: a ray of an empty scene fetches the placeholder root and nothing else (no
// triangle, no instance, no push), so its whole record is zero.
int drop_placeholder_costs(const tray_scene* s, tray_ray_cost* d, uint64_t n, cudaStream_t st) {
    if (s->n_nodes == 0 && d && n) CU(cudaMemsetAsync(d, 0, n * sizeof(tray_ray_cost), st));
    return TRAY_OK;
}

// a device error word as a status
int flag_status(uint32_t f) {
    if (!f) return TRAY_OK;
    if (f & ERR_WATCHDOG) return fail(TRAY_ERR_CUDA, "frame kernel watchdog: a group of primary hits never arrived (the frame is incomplete)");
    return fail(TRAY_ERR_OVERFLOW, "traversal stack overflow: BVH needs more than %d stack entries", STACK_SMEM + STACK_SPILL);
}
// the error word `flag` behind the work enqueued on `st`, as a status; a set word is cleared there, in stream order, so that an
// error is reported once, by the first synchronising call that covers the launch that raised it
int check_overflow(uint32_t* flag, cudaStream_t st) {
    uint32_t f = 0;
    CU(cudaMemcpyAsync(&f, flag, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (f) cudaMemsetAsync(flag, 0, 4, st);
    return flag_status(f);
}

// the start protocol's arguments (the reference asserts these strides at src/rt_gpu/mod.rs:70,86,105,107)
int check_start_args(const tray_view* view, uint64_t bvh_len, uint64_t tri_len, uint32_t tri_stride, uint64_t instance_len) {
    if (!view) return fail(TRAY_ERR_ARG, "NULL view");
    if (bvh_len % 80 != 0) return fail(TRAY_ERR_ARG, "bvh_bytes length %llu is not a multiple of 80", (unsigned long long)bvh_len);
    if (tri_stride == 0 || tri_len % tri_stride != 0) return fail(TRAY_ERR_ARG, "tri_bytes length is not a multiple of tri_stride");
    if (instance_len % 4 != 0) return fail(TRAY_ERR_ARG, "instance_bytes length is not a multiple of 4");
    return TRAY_OK;
}

// the timed loop of the start protocol over one scene or a group: render(frame_count), render_timed(frame_count, &ms), sync()
template <typename Render, typename RenderTimed, typename Sync>
int start_loop(Render render, RenderTimed render_timed, Sync sync, float render_time_s, int benchmark, int animate,
               float* out_min_ms, float* out_mean_ms, uint32_t* out_frames) {
    float min_ms = 3.402823466e+38f; double sum = 0; uint32_t frames = 0, frame_count = 0;
    const auto t0 = std::chrono::steady_clock::now();
    for (;;) {
        if (benchmark) {   // untimed warm-up dispatch right before the timed one (rt_gpu_software.rs:289-295)
            if (const int rc = render(frame_count)) return rc;
        }
        float ms = 0.f;       // the whole dispatch, as the reference's timestamp queries bracket it (rt_gpu_software.rs:296-301)
        if (const int rc = render_timed(frame_count, &ms)) return rc;
        if (ms < min_ms) min_ms = ms;
        sum += ms; frames++;
        if (animate) frame_count = frames;                                   // rt_cpu.rs:95-97
        const float el = std::chrono::duration<float>(std::chrono::steady_clock::now() - t0).count();
        if (el > render_time_s) break;                                       // rt_cpu.rs:98-100, rt_gpu_software.rs:354-359
    }
    if (const int rc = sync()) return rc;
    if (out_min_ms) *out_min_ms = min_ms;
    if (out_mean_ms) *out_mean_ms = frames ? (float)(sum / frames) : 0.f;
    if (out_frames) *out_frames = frames;
    return TRAY_OK;
}

}  // namespace

namespace {
__global__ void __launch_bounds__(512) bandwidth_kernel(const uint4* __restrict__ buf, uint64_t n16, int iters, uint32_t* out) {
    uint4 acc = make_uint4(0, 0, 0, 0);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (int it = 0; it < iters; it++)
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
            const uint4 v = __ldcg(buf + i);                // L2-cached, bypass L1: this measures the L2 / HBM pipe
            acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
        }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345678u) out[0] = acc.x;   // never true in practice; keeps the loads alive
}
// every lane gathers 16-byte records from its own pseudo-random line of a small (L1-resident) table
__global__ void __launch_bounds__(128, 8) l1_gather_kernel(const uint4* __restrict__ buf, uint32_t n_lines, int iters, uint32_t* out) {
    uint32_t x = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x = x * 1664525u + 1013904223u;
            const uint32_t line = __umulhi(x, n_lines), quad = (x >> 3) & 7u;      // 128-byte line, 16-byte record inside it
            const uint4 v = __ldg(buf + (size_t)line * 8u + quad);
            acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
        }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345678u) out[0] = acc.x;
}
}  // namespace

extern "C" {

int tray_cuda_l1_gather_probe(int device, uint32_t bytes, int iters, float* out_gbs) {
    if (!out_gbs || bytes < 1024 || bytes > (64u << 10) || iters < 1) return fail(TRAY_ERR_ARG, "bad argument");
    if (tray_cuda_device_count() == 0) return fail(TRAY_ERR_NO_DEVICE, "no CUDA device");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, device));
    uint4* buf = nullptr; uint32_t* out = nullptr;
    const uint32_t n_lines = bytes / 128;
    CU(cudaMalloc(&buf, (size_t)n_lines * 128)); CU(cudaMalloc(&out, 4));
    CU(cudaMemset(buf, 0x5a, (size_t)n_lines * 128));
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    const int grid = prop.multiProcessorCount * 8;
    l1_gather_kernel<<<grid, 128>>>(buf, n_lines, 2, out);
    CU(cudaEventRecord(e0));
    l1_gather_kernel<<<grid, 128>>>(buf, n_lines, iters, out);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f; CU(cudaEventElapsedTime(&ms, e0, e1));
    *out_gbs = (float)((double)grid * 128.0 * 8.0 * iters * 16.0 / (ms * 1e-3) / 1e9);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf); cudaFree(out);
    return TRAY_OK;
}

int tray_cuda_bandwidth_probe(int device, uint64_t bytes, int iters, float* out_gbs) {
    if (!out_gbs || bytes < 4096 || iters < 1) return fail(TRAY_ERR_ARG, "bad argument");
    if (tray_cuda_device_count() == 0) return fail(TRAY_ERR_NO_DEVICE, "no CUDA device");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, device));
    uint4* buf = nullptr; uint32_t* out = nullptr;
    const uint64_t n16 = bytes / 16;
    CU(cudaMalloc(&buf, n16 * 16)); CU(cudaMalloc(&out, 4));
    CU(cudaMemset(buf, 0x5a, n16 * 16));
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    const int grid = prop.multiProcessorCount * 4;
    bandwidth_kernel<<<grid, 512>>>(buf, n16, 2, out);      // warm-up: brings the buffer into L2 when it fits
    CU(cudaEventRecord(e0));
    bandwidth_kernel<<<grid, 512>>>(buf, n16, iters, out);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f; CU(cudaEventElapsedTime(&ms, e0, e1));
    *out_gbs = (float)((double)n16 * 16.0 * iters / (ms * 1e-3) / 1e9);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf); cudaFree(out);
    return TRAY_OK;
}

const char* tray_cuda_last_error(void) { return g_err; }
unsigned tray_cuda_abi_version(void) { return TRAY_CUDA_ABI_VERSION; }

int tray_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void tray_cuda_scene_destroy(tray_scene* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    cudaFree(s->d_nodes); cudaFree(s->d_tris); cudaFree(s->d_blas); cudaFree(s->d_prim_indices); cudaFree(s->d_cursor); cudaFree(s->d_overflow);
    cudaFree(s->d_rays); cudaFree(s->d_hits); cudaFree(s->d_costs); cudaFree(s->d_geom_offsets);
    delete s->refit;
    free_pipeline(s);
    cudaFree(s->d_untiled);
    for (auto& f : s->slot) {
        if (f.own_stream) cudaStreamSynchronize(f.own_stream);
        free_frame_buffers(f);
        cudaFree(f.d_cursor); cudaFree(f.d_units);
        for (auto& e : f.ev) if (e) cudaEventDestroy(e);
        if (f.done) cudaEventDestroy(f.done);
        if (f.own_stream) cudaStreamDestroy(f.own_stream);
    }
    for (auto& e : s->ev) if (e) cudaEventDestroy(e);
    for (int i = 0; i < TRAY_READBACK_SLOTS; i++) {
        if (s->stage_busy[i]) cudaEventSynchronize(s->ev_copied[i]);
        cudaFree(s->d_stage[i]);
        if (s->ev_untiled[i]) cudaEventDestroy(s->ev_untiled[i]);
        if (s->ev_copied[i]) cudaEventDestroy(s->ev_copied[i]);
    }
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    if (s->h_flag) cudaFreeHost(s->h_flag);
    if (s->ev_after) cudaEventDestroy(s->ev_after);
    delete s;
}

}  // extern "C"

namespace {
// `built` != NULL: adopt the device buffers of the device-side builder instead of uploading host arrays
int scene_create_impl(const void* nodes, uint64_t n_nodes, const void* tris, uint64_t n_tris, uint32_t tri_stride,
                      const uint32_t* blas_offsets, uint32_t n_instances, uint32_t tlas_start,
                      int device, tray_build::Result* built, tray_scene** out) {
    if (!out) return fail(TRAY_ERR_ARG, "out_scene is NULL");
    *out = nullptr;
    if (!built && ((n_nodes && !nodes) || (n_tris && !tris))) return fail(TRAY_ERR_ARG, "NULL node / triangle buffer");
    if (const int rc = check_tri_stride(tri_stride)) return rc;
    if (n_instances && !blas_offsets && !built) return fail(TRAY_ERR_ARG, "n_instances > 0 but blas_offsets is NULL");
    if (n_instances && tlas_start >= n_nodes) return fail(TRAY_ERR_ARG, "tlas_start %u outside %llu nodes", tlas_start, (unsigned long long)n_nodes);
    if (n_nodes >= 0xffffffffull || n_tris >= 0xffffffffull) return fail(TRAY_ERR_ARG, "node / triangle indices are 32-bit");
    if (const int rc = select_device(device)) return rc;
    tray_scene* s = new (std::nothrow) tray_scene();
    if (!s) return fail(TRAY_ERR_ARG, "out of host memory");
    s->device = device; s->n_nodes = n_nodes; s->n_tris = n_tris; s->tri_stride = tri_stride;
    s->n_instances = n_instances; s->tlas_start = tlas_start; s->tlas = n_instances > 0;
    s->refill_min = (uint32_t)env_int("TRAY_CUDA_REFILL_MIN", 6);       // 6: +0.3 % (C3) ... +2 % (C1) over 4 with the r2 kernel (profiles/experiments/r2_refill_min_ab.log)
    s->force_exact = scene_force_exact(built && built->force_exact);
    for (uint64_t i = 0; !built && i < n_nodes && !s->force_exact; i++) {
        const uint8_t* e = (const uint8_t*)nodes + i * 80 + 12;
        if (tray::node_needs_exact(e[0] | (uint32_t)e[1] << 8 | (uint32_t)e[2] << 16)) s->force_exact = true;   // scale = 2^(e-127) >= 2^40
    }
    s->tri_weight = (uint32_t)env_int("TRAY_CUDA_TRI_WEIGHT", 3);     // 3: +0.6 ... 1.2 % over 4 with two triangles per step (profiles/experiments/r2_triweight_ab.log)
    s->gen_min = (uint32_t)env_int("TRAY_CUDA_GEN_MIN", 4);
    s->overlap_default = env_int("TRAY_CUDA_OVERLAP", 0) != 0;
    const bool adopted = built && built->d_nodes;
    auto body = [&]() -> int {
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, device));
        s->sm_count = prop.multiProcessorCount;
        s->l2_bytes = (uint64_t)prop.l2CacheSize;
        CU(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
        s->stream = s->own_stream;
        for (auto& e : s->ev) CU(cudaEventCreate(&e));
        CU(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&s->ev_after, cudaEventDisableTiming));
        CU(cudaMallocHost(&s->h_flag, TRAY_READBACK_SLOTS * sizeof(uint32_t)));
        for (int i = 0; i < TRAY_READBACK_SLOTS; i++) {
            s->h_flag[i] = 0u;
            CU(cudaEventCreateWithFlags(&s->ev_untiled[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s->ev_copied[i], cudaEventDisableTiming));
        }
        const size_t nb = (size_t)(n_nodes ? n_nodes : 1) * 80, tb = (size_t)(n_tris ? n_tris : 1) * tri_stride;
        if (adopted) {
            s->d_nodes = (uint4*)built->d_nodes; s->d_tris = (uint4*)built->d_tris; s->d_prim_indices = built->d_prim_indices;
            s->d_blas = built->d_blas_offsets;
            // ownership moves to the scene HERE: from now on tray_cuda_scene_destroy is the one place that frees them
            built->d_nodes = nullptr; built->d_tris = nullptr; built->d_prim_indices = nullptr; built->d_blas_offsets = nullptr;
        } else {
            CU(cudaMalloc(&s->d_nodes, nb));
            CU(cudaMalloc(&s->d_tris, tb));
        }
        if (!s->d_blas) CU(cudaMalloc(&s->d_blas, (size_t)(n_instances ? n_instances : 1) * 4));
        CU(cudaMalloc(&s->d_cursor, CURSOR_WORDS * sizeof(unsigned long long)));
        CU(cudaMalloc(&s->d_overflow, (1 + TRAY_MAX_FRAMES_IN_FLIGHT) * sizeof(uint32_t)));
        CU(cudaMemsetAsync(s->d_cursor, 0, CURSOR_WORDS * sizeof(unsigned long long), s->stream));
        for (int k = 0; k < TRAY_MAX_FRAMES_IN_FLIGHT; k++) {
            FrameSlot& f = s->slot[k];
            if (k >= 1) CU(cudaStreamCreateWithFlags(&f.own_stream, cudaStreamNonBlocking));
            CU(cudaMalloc(&f.d_cursor, CURSOR_WORDS * sizeof(unsigned long long)));
            CU(cudaMalloc(&f.d_units, sizeof(uint32_t)));
            f.d_flag = s->d_overflow + 1 + k;
            CU(cudaMemsetAsync(f.d_cursor, 0, CURSOR_WORDS * sizeof(unsigned long long), s->stream));
            for (auto& e : f.ev) CU(cudaEventCreate(&e));
            CU(cudaEventCreateWithFlags(&f.done, cudaEventDisableTiming));
        }
        CU(cudaMemsetAsync(s->d_overflow, 0, (1 + TRAY_MAX_FRAMES_IN_FLIGHT) * sizeof(uint32_t), s->stream));
        s->device_bytes = nb + tb + (size_t)n_instances * 4;
        if (!adopted) {
            if (n_nodes) CU(tray::upload_pipelined(s->d_nodes, nodes, (size_t)n_nodes * 80, s->stream));
            else CU(cudaMemsetAsync(s->d_nodes, 0, 80, s->stream));   // empty scene: a root with no children, every ray misses
            if (n_tris) CU(tray::upload_pipelined(s->d_tris, tris, (size_t)n_tris * tri_stride, s->stream));
        }
        if (n_instances && blas_offsets) CU(cudaMemcpyAsync(s->d_blas, blas_offsets, (size_t)n_instances * 4, cudaMemcpyHostToDevice, s->stream));
        // keep the node array hot in the 126 MB L2: persisting access-policy window, attached to every traversal launch
        if (prop.persistingL2CacheMaxSize > 0 && n_nodes) {
            size_t want = (size_t)prop.persistingL2CacheMaxSize;
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
                size_t win = (size_t)n_nodes * 80;
                if (win > (size_t)prop.accessPolicyMaxWindowSize) win = (size_t)prop.accessPolicyMaxWindowSize;
                memset(&s->window, 0, sizeof s->window);
                s->window.base_ptr = s->d_nodes;
                s->window.num_bytes = win;
                double ratio = (double)want / (double)win;
                s->window.hitRatio = (float)(ratio > 1.0 ? 1.0 : ratio);
                s->window.hitProp = cudaAccessPropertyPersisting;
                s->window.missProp = cudaAccessPropertyStreaming;
                s->have_window = true;
                s->l2_persist = win < want ? win : want;
            } else cudaGetLastError();
        }
        CU(cudaStreamSynchronize(s->stream));
        return TRAY_OK;
    };
    const int rc = body();
    if (rc != TRAY_OK) { tray_cuda_scene_destroy(s); return rc; }
    *out = s;
    return TRAY_OK;
}
}  // namespace

extern "C" {

int tray_cuda_scene_create(const void* nodes, uint64_t n_nodes, const void* tris, uint64_t n_tris, uint32_t tri_stride,
                           const uint32_t* blas_offsets, uint32_t n_instances, uint32_t tlas_start,
                           int device, tray_scene** out) {
    return scene_create_impl(nodes, n_nodes, tris, n_tris, tri_stride, blas_offsets, n_instances, tlas_start, device, nullptr, out);
}

}  // extern "C"

namespace {
int scene_build_impl(const float* tris9, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects, uint32_t tri_stride,
                     uint32_t max_prims_per_leaf, uint32_t search_radius, int device, tray_scene** out, tray_build_stats* out_stats) {
    if (!out) return fail(TRAY_ERR_ARG, "out_scene is NULL");
    *out = nullptr;
    if (n_tris && !tris9) return fail(TRAY_ERR_ARG, "NULL triangle buffer");
    if (const int rc = check_tri_stride(tri_stride)) return rc;
    if (max_prims_per_leaf < 1 || max_prims_per_leaf > 3) return fail(TRAY_ERR_ARG, "max_prims_per_leaf must be 1..3");
    if (search_radius > 64) return fail(TRAY_ERR_ARG, "search_radius must be 0 (default 14) or 1..64");
    if (object_offsets && n_tris == 0) return fail(TRAY_ERR_ARG, "a two-level scene needs triangles");
    if (const int rc = select_device(device)) return rc;
    tray_build::Result r;
    char msg[400] = "";
    const int brc = tray_build::build_tlas(tris9, n_tris, object_offsets, n_objects, tri_stride, max_prims_per_leaf,
                                           search_radius ? search_radius : 14u, nullptr, &r, msg, sizeof msg);
    if (brc) return fail(brc == -1 ? TRAY_ERR_ARG : TRAY_ERR_CUDA, "device build failed: %s", msg);
    const int rc = scene_create_impl(nullptr, r.n_nodes, nullptr, n_tris, tri_stride, nullptr, r.n_instances, r.tlas_start, device, &r, out);
    // whatever scene_create_impl did not adopt is still ours (adopted pointers are nulled in `r`): freed exactly once
    if (rc) { cudaFree(r.d_nodes); cudaFree(r.d_tris); cudaFree(r.d_prim_indices); cudaFree(r.d_blas_offsets); return rc; }
    if (out_stats) *out_stats = r.stats;
    return TRAY_OK;
}
}  // namespace

extern "C" {

int tray_cuda_scene_build(const float* tris9, uint64_t n_tris, uint32_t tri_stride, uint32_t max_prims_per_leaf,
                          uint32_t search_radius, int device, tray_scene** out, tray_build_stats* out_stats) {
    return scene_build_impl(tris9, n_tris, nullptr, 0, tri_stride, max_prims_per_leaf, search_radius, device, out, out_stats);
}

int tray_cuda_scene_build_tlas(const float* tris9, uint64_t n_tris, const uint64_t* object_offsets, uint32_t n_objects, uint32_t tri_stride,
                               uint32_t max_prims_per_leaf, uint32_t search_radius, int device, tray_scene** out, tray_build_stats* out_stats) {
    if (!object_offsets || n_objects == 0) return fail(TRAY_ERR_ARG, "object_offsets is NULL / no objects");
    return scene_build_impl(tris9, n_tris, object_offsets, n_objects, tri_stride, max_prims_per_leaf, search_radius, device, out, out_stats);
}

int tray_cuda_scene_download_instances(tray_scene* s, uint32_t* blas_offsets) {
    if (!s || !blas_offsets) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    if (s->n_instances) CU(cudaMemcpy(blas_offsets, s->d_blas, (size_t)s->n_instances * 4, cudaMemcpyDeviceToHost));
    return TRAY_OK;
}

int tray_cuda_scene_download(tray_scene* s, void* nodes, void* tris, uint32_t* prim_indices) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    if (prim_indices && !s->d_prim_indices && s->n_tris) return fail(TRAY_ERR_ARG, "this scene was not built on the device: it has no primitive index array");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    if (nodes && s->n_nodes) CU(cudaMemcpy(nodes, s->d_nodes, (size_t)s->n_nodes * 80, cudaMemcpyDeviceToHost));
    if (tris && s->n_tris) CU(cudaMemcpy(tris, s->d_tris, (size_t)s->n_tris * s->tri_stride, cudaMemcpyDeviceToHost));
    if (prim_indices && s->n_tris) CU(cudaMemcpy(prim_indices, s->d_prim_indices, (size_t)s->n_tris * 4, cudaMemcpyDeviceToHost));
    return TRAY_OK;
}

int tray_cuda_scene_info(const tray_scene* s, tray_scene_info* o) {
    if (!s || !o) return fail(TRAY_ERR_ARG, "NULL argument");
    memset(o, 0, sizeof *o);
    o->n_nodes = s->n_nodes; o->n_tris = s->n_tris; o->tri_stride = s->tri_stride; o->n_instances = s->n_instances;
    o->tlas_start = s->tlas_start; o->is_tlas = s->tlas; o->device = s->device; o->sm_count = (uint32_t)s->sm_count;
    o->device_bytes = s->device_bytes; o->l2_bytes = s->l2_bytes; o->l2_persist_bytes = s->l2_persist;
    return TRAY_OK;
}

int tray_cuda_scene_exact_node_test(const tray_scene* s, int* out_exact) {
    if (!s || !out_exact) return fail(TRAY_ERR_ARG, "NULL argument");
    *out_exact = s->force_exact ? 1 : 0;
    return TRAY_OK;
}

int tray_cuda_set_counting(tray_scene* s, int enabled) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    s->counting = enabled != 0;
    return TRAY_OK;
}

int tray_cuda_scene_set_ray_cost(tray_scene* s, int enabled) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    s->ray_cost = enabled != 0;
    return TRAY_OK;
}

int tray_cuda_scene_set_variant(tray_scene* s, uint32_t flags) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    if (flags & ~0xfu) return fail(TRAY_ERR_ARG, "unknown variant flags 0x%x", flags);
    s->variant = flags;
    return TRAY_OK;
}

int tray_cuda_scene_set_stream(tray_scene* s, void* stream) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    CU(cudaSetDevice(s->device));
    if (const int rc = sync_streams(s, /*scene_stream_first=*/true)) return rc;
    s->stream = stream ? (cudaStream_t)stream : s->own_stream;
    return TRAY_OK;
}

int tray_cuda_untile_rgba(tray_scene* s, const void* d_compact, uint32_t w, uint32_t h, uint32_t shard, uint32_t shards, void* d_frame) {
    if (!s || !d_compact || !d_frame) return fail(TRAY_ERR_ARG, "NULL argument");
    if (shards == 0) shards = 1;
    if (w == 0 || h == 0 || shard >= shards) return fail(TRAY_ERR_ARG, "bad frame size / shard");
    CU(cudaSetDevice(s->device));
    FrameParams F; frame_params(F, nullptr, w, h, 0, shard, shards);
    if (F.n_items == 0) return TRAY_OK;
    // on the stream of the last rendered frame (its compact buffer is the usual source); with one frame in flight: the scene stream
    tray::untile_kernel<uchar4><<<(F.n_items + 255) / 256, 256, 0, slot_stream(s, s->cur)>>>(F, (const uchar4*)d_compact, (uchar4*)d_frame);
    CU(cudaGetLastError());
    return TRAY_OK;
}

int tray_cuda_frame_push(tray_scene* s, void* d_dst) {
    if (!s || !d_dst) return fail(TRAY_ERR_ARG, "NULL argument");
    const FrameSlot& f = s->slot[s->cur];
    if (f.last_frame.width == 0 || !f.f_has_rgba) return fail(TRAY_ERR_ARG, "last frame was rendered without TRAY_RENDER_RGBA (or into a frame target)");
    CU(cudaSetDevice(s->device));
    if (f.last_frame.n_items) CU(cudaMemcpyAsync(d_dst, f.d_rgba, (size_t)f.last_frame.n_items * sizeof(uchar4), cudaMemcpyDeviceToDevice, slot_stream(s, s->cur)));
    return TRAY_OK;
}

int tray_cuda_untile_shards(tray_scene* s, const void* d_staging, uint32_t w, uint32_t h, uint32_t shards, void* d_frame) {
    if (!s || !d_staging || !d_frame) return fail(TRAY_ERR_ARG, "NULL argument");
    if (shards == 0) shards = 1;
    if (w == 0 || h == 0) return fail(TRAY_ERR_ARG, "bad frame size");
    CU(cudaSetDevice(s->device));
    const dim3 grid((w + 255) / 256, h);
    tray::untile_shards_kernel<<<grid, 256, 0, slot_stream(s, s->cur)>>>((const uchar4*)d_staging, w, h, (w + 31) / 32, shards,
                                                                        local_items(w, h, 0, shards), (uchar4*)d_frame);
    CU(cudaGetLastError());
    return TRAY_OK;
}

int tray_cuda_frame_alloc(int device, uint64_t bytes, void** d_ptr) {
    if (!d_ptr || bytes == 0) return fail(TRAY_ERR_ARG, "bad argument");
    if (tray_cuda_device_count() == 0) return fail(TRAY_ERR_NO_DEVICE, "no CUDA device");
    CU(cudaSetDevice(device));
    CU(cudaMalloc(d_ptr, bytes));
    CU(cudaMemset(*d_ptr, 0, bytes));
    return TRAY_OK;
}

int tray_cuda_frame_free(int device, void* d_ptr) {
    if (!d_ptr) return TRAY_OK;
    CU(cudaSetDevice(device));
    CU(cudaFree(d_ptr));
    return TRAY_OK;
}

int tray_cuda_ipc_export(int device, void* d_ptr, uint8_t handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    if (!d_ptr || !handle) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, d_ptr));
    memcpy(handle, &h, 64);
    return TRAY_OK;
}

int tray_cuda_ipc_open(int device, const uint8_t handle[64], void** d_ptr) {
    if (!d_ptr || !handle) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return TRAY_OK;
}

int tray_cuda_ipc_close(int device, void* d_ptr) {
    if (!d_ptr) return TRAY_OK;
    CU(cudaSetDevice(device));
    CU(cudaIpcCloseMemHandle(d_ptr));
    return TRAY_OK;
}

int tray_cuda_scene_set_frame_target(tray_scene* s, void* d_frame) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    // launches already enqueued carry the old target in their parameters: no synchronisation needed to switch
    s->frame_target = (uchar4*)d_frame;
    return TRAY_OK;
}

int tray_cuda_sync(tray_scene* s) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    CU(cudaSetDevice(s->device));
    if (const int rc = sync_streams(s, /*scene_stream_first=*/false)) return rc;
    // every error word a launch of the scene can have set: batch traces and each frame slot; a set word is cleared on its own
    // stream, ahead of whatever is enqueued there next
    uint32_t f[1 + TRAY_MAX_FRAMES_IN_FLIGHT];
    CU(cudaMemcpyAsync(f, s->d_overflow, sizeof f, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    uint32_t all = 0;
    for (int k = 0; k <= TRAY_MAX_FRAMES_IN_FLIGHT; k++)
        if (f[k]) { all |= f[k]; cudaMemsetAsync(s->d_overflow + k, 0, 4, k ? slot_stream(s, k - 1) : s->stream); }
    return flag_status(all);
}

}  // extern "C"

namespace {
// tray_cuda_scene_refit(_device): `tris9` is host memory unless `device_ptr`.  Every check runs before the first write, so a
// refused call leaves nodes, records and force_exact as they were.
int refit_impl(tray_scene* s, const float* tris9, uint64_t n_tris, bool device_ptr, void* stream, float* ms_refit) {
    if (ms_refit) *ms_refit = 0.f;
    if (!s || !tris9) return fail(TRAY_ERR_ARG, "NULL argument");
    if (n_tris != s->n_tris) return fail(TRAY_ERR_ARG, "refit with %llu triangles, the scene has %llu", (unsigned long long)n_tris, (unsigned long long)s->n_tris);
    CU(cudaSetDevice(s->device));
    // after every frame and batch enqueued so far: frames rendered before the refit keep their old-geometry results
    if (stream) CU(cudaStreamSynchronize((cudaStream_t)stream));
    if (const int rc = sync_streams(s, /*scene_stream_first=*/false)) return rc;
    CU(cudaStreamSynchronize(s->copy_stream));
    if (s->pipeline_ready) { CU(cudaStreamSynchronize(s->s_in)); CU(cudaStreamSynchronize(s->s_out)); }
    if (n_tris == 0) return TRAY_OK;
    char msg[400] = "";
    if (!s->refit) {
        tray_build::RefitTopology t;
        const int rc = tray_build::refit_walk(s->d_nodes, s->n_nodes, s->n_tris, s->tlas ? s->d_blas : nullptr, s->tlas ? s->n_instances : 0u,
                                              s->tlas_start, s->stream, &t, msg, sizeof msg);
        if (rc) return fail(rc == -1 ? TRAY_ERR_ARG : TRAY_ERR_CUDA, "refit: %s", msg);
        s->refit = new (std::nothrow) tray_build::RefitTopology(std::move(t));
        if (!s->refit) return fail(TRAY_ERR_ARG, "out of host memory");
        s->device_bytes += s->refit->bytes;
    }
    const float* d_tris9 = tris9;
    float* d_upload = nullptr;
    if (!device_ptr) {
        CU(cudaMalloc(&d_upload, (size_t)n_tris * 36));
        const cudaError_t e = tray::upload_pipelined(d_upload, tris9, (size_t)n_tris * 36, s->stream);
        if (e != cudaSuccess) { cudaFree(d_upload); return fail(TRAY_ERR_CUDA, "refit upload failed: %s", cudaGetErrorString(e)); }
        d_tris9 = d_upload;
    }
    auto body = [&]() -> int {
        float ms_check = 0.f, ms_run = 0.f;
        bool bad = false, exact = false;
        CU(cudaEventRecord(s->ev[0], s->stream));
        if (tray_build::refit_check(*s->refit, d_tris9, n_tris, s->stream, &bad, msg, sizeof msg)) return fail(TRAY_ERR_CUDA, "refit: %s", msg);
        CU(cudaEventRecord(s->ev[1], s->stream));
        CU(cudaEventSynchronize(s->ev[1]));
        CU(cudaEventElapsedTime(&ms_check, s->ev[0], s->ev[1]));
        if (bad) return fail(TRAY_ERR_ARG, "refit: a coordinate is not finite, or the triangles' extent on some axis overflows f32");
        CU(cudaEventRecord(s->ev[0], s->stream));
        if (tray_build::refit_run(*s->refit, d_tris9, n_tris, s->d_prim_indices, s->tri_stride, s->d_nodes, s->d_tris, s->d_blas, s->stream,
                                  &exact, msg, sizeof msg)) return fail(TRAY_ERR_CUDA, "refit: %s", msg);
        CU(cudaEventRecord(s->ev[1], s->stream));
        CU(cudaEventSynchronize(s->ev[1]));
        CU(cudaEventElapsedTime(&ms_run, s->ev[0], s->ev[1]));
        s->force_exact = scene_force_exact(exact);
        if (ms_refit) *ms_refit = ms_check + ms_run;
        return TRAY_OK;
    };
    const int rc = body();
    cudaFree(d_upload);
    return rc;
}
}  // namespace

extern "C" {

int tray_cuda_scene_refit(tray_scene* s, const float* tris9, uint64_t n_tris, float* ms_refit) {
    return refit_impl(s, tris9, n_tris, false, nullptr, ms_refit);
}
int tray_cuda_scene_refit_device(tray_scene* s, const float* d_tris9, uint64_t n_tris, void* stream, float* ms_refit) {
    return refit_impl(s, d_tris9, n_tris, true, stream, ms_refit);
}

}  // extern "C"

namespace {
// d_costs != NULL: the cost calls — the counting kernels whatever tray_scene::counting says, the counters read under it alone
int trace_device_impl(tray_scene* s, const tray_ray* d_rays, uint64_t n, tray_hit* d_hits, tray_ray_cost* d_costs, void* stream,
                      float* ms_kernel, bool anyhit) {
    if (!s || (n && (!d_rays || !d_hits))) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (ms_kernel) CU(cudaEventRecord(s->ev[0], st));
    const uint64_t chunk = INDEX_MASK + 1ull;             // inside the kernel a ray index keeps two tag bits above INDEX_MASK
    for (uint64_t off = 0; off < n; off += chunk) {
        TraceParams P; base_params(s, P);
        P.rays = d_rays + off; P.n_work = (uint32_t)(n - off < chunk ? n - off : chunk); P.hits_out = d_hits + off;
        P.ray_cost = d_costs ? d_costs + off : nullptr;
        int rc = launch(s, P, st, s->d_cursor, 0, s->counting || d_costs, anyhit, /*keep_counters=*/off > 0);      // counters accumulate over the chunks of one batch
        if (rc) return rc;
    }
    if (const int rc = drop_placeholder_costs(s, d_costs, n, st)) return rc;
    if (ms_kernel) {
        CU(cudaEventRecord(s->ev[1], st));
        CU(cudaEventSynchronize(s->ev[1]));
        CU(cudaEventElapsedTime(ms_kernel, s->ev[0], s->ev[1]));
        if (s->counting) {                                // synchronised: the batch's counters, summed over its launches
            const int rc = read_counters(s->d_cursor, st, 0, &s->cnt_primary); if (rc) return rc;
            memset(&s->cnt_bounce, 0, sizeof s->cnt_bounce);
            drop_placeholder_root(s);
        }
        return check_overflow(s->d_overflow, st);         // synchronised: an overflow of this batch is reported by this call
    }
    return TRAY_OK;
}

constexpr uint64_t CHUNK_MAX = 1ull << 20;        // rays per pipeline stage (32 MiB in, 8 MiB out)
constexpr uint64_t PIPE_MIN = 1ull << 18;         // smaller batches take the plain copy-launch-copy path

int ensure_pipeline(tray_scene* s) {
    if (s->pipeline_ready) return TRAY_OK;
    auto body = [&]() -> int {
        CU(cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaMallocHost(&s->h_rays[i], CHUNK_MAX * sizeof(tray_ray)));
            CU(cudaMallocHost(&s->h_hits[i], CHUNK_MAX * sizeof(tray_hit)));
            CU(cudaEventCreateWithFlags(&s->e_in[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s->e_k[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s->e_out[i], cudaEventDisableTiming));
        }
        return TRAY_OK;
    };
    const int rc = body();
    if (rc) { free_pipeline(s); return rc; }      // a half-built pipeline must not look ready to the next call
    s->pipeline_ready = true;
    return TRAY_OK;
}

// Batch operator with HOST buffers (Traversable::traverse for a slice of rays).  Large batches run as a three-stage pipeline
// over chunks of up to CHUNK_MAX rays: [host threads: caller's rays -> pinned slot] [copy stream: H2D] [scene stream: traversal]
// [copy stream: D2H into a pinned slot] [host threads: -> caller's hits]; chunk i+1 is staged and uploaded while chunk i is
// traced and chunk i-1 is read back.  The caller's memory is only borrowed for the call and never registered.
// costs != NULL: the cost calls (see trace_device_impl); the records travel like the hits
int trace_impl(tray_scene* s, const tray_ray* rays, uint64_t n, tray_hit* hits, tray_ray_cost* costs, float* ms_kernel, float* ms_total,
               bool anyhit) {
    if (!s || (n && (!rays || !hits))) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    const auto t0 = std::chrono::steady_clock::now();
    if (n > s->batch_cap) {
        cudaFree(s->d_rays); cudaFree(s->d_hits); s->d_rays = nullptr; s->d_hits = nullptr; s->batch_cap = 0;
        CU(cudaMalloc(&s->d_rays, n * sizeof(tray_ray)));
        CU(cudaMalloc(&s->d_hits, n * sizeof(tray_hit)));
        s->batch_cap = n;
    }
    if (costs && n > s->cost_cap) {
        cudaFree(s->d_costs); s->d_costs = nullptr; s->cost_cap = 0;
        CU(cudaMalloc(&s->d_costs, n * sizeof(tray_ray_cost)));
        s->cost_cap = n;
    }
    tray_ray_cost* const d_costs = costs ? s->d_costs : nullptr;
    float k = 0.f;
    int rc = TRAY_OK;
    if (n < PIPE_MIN) {
        if (n) CU(cudaMemcpyAsync(s->d_rays, rays, n * sizeof(tray_ray), cudaMemcpyHostToDevice, s->stream));
        rc = trace_device_impl(s, s->d_rays, n, s->d_hits, d_costs, s->stream, &k, anyhit);
        if (rc) return rc;
        if (n) CU(cudaMemcpyAsync(hits, s->d_hits, n * sizeof(tray_hit), cudaMemcpyDeviceToHost, s->stream));
        if (n && costs) CU(cudaMemcpyAsync(costs, d_costs, n * sizeof(tray_ray_cost), cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
    } else {
        rc = ensure_pipeline(s);
        if (rc) return rc;
        for (int i = 0; costs && i < 2; i++)
            if (!s->h_costs[i]) CU(cudaMallocHost(&s->h_costs[i], CHUNK_MAX * sizeof(tray_ray_cost)));
        // chunk size: the pipeline only pays once it has a few stages, and every stage is a kernel launch with its own
        // drain phase — 2^19 rays below 4 M rays, 2^20 above
        const uint64_t chunk = n < (4ull << 20) ? (CHUNK_MAX >> 1) : CHUNK_MAX;
        const uint64_t n_chunks = (n + chunk - 1) / chunk;
        auto chunk_len = [&](uint64_t i) { return i + 1 < n_chunks ? chunk : n - i * chunk; };
        if (s->counting) CU(cudaMemsetAsync(s->d_cursor + CURSOR_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), s->stream));
        CU(cudaEventRecord(s->ev[0], s->stream));
        for (uint64_t i = 0; i < n_chunks + 2; i++) {
            const int slot = (int)(i & 1);
            if (i < n_chunks) {
                const uint64_t off = i * chunk, len = chunk_len(i);
                if (i >= 2) CU(cudaEventSynchronize(s->e_in[slot]));                 // the slot's previous upload has left it
                tray::par_copy(s->h_rays[slot], rays + off, len * sizeof(tray_ray));
                CU(cudaMemcpyAsync(s->d_rays + off, s->h_rays[slot], len * sizeof(tray_ray), cudaMemcpyHostToDevice, s->s_in));
                CU(cudaEventRecord(s->e_in[slot], s->s_in));
                CU(cudaStreamWaitEvent(s->stream, s->e_in[slot], 0));
                TraceParams P; base_params(s, P);
                P.rays = s->d_rays + off; P.n_work = (uint32_t)len; P.hits_out = s->d_hits + off;
                P.ray_cost = d_costs ? d_costs + off : nullptr;
                rc = launch(s, P, s->stream, s->d_cursor, 0, s->counting || costs, anyhit, /*keep_counters=*/true);
                if (rc) return rc;
                rc = drop_placeholder_costs(s, P.ray_cost, len, s->stream);
                if (rc) return rc;
                CU(cudaEventRecord(s->e_k[slot], s->stream));
            }
            if (i >= 1 && i - 1 < n_chunks) {                                           // chunk i-1: start its read-back
                const uint64_t j = i - 1; const int ps = (int)(j & 1);
                CU(cudaStreamWaitEvent(s->s_out, s->e_k[ps], 0));
                CU(cudaMemcpyAsync(s->h_hits[ps], s->d_hits + j * chunk, chunk_len(j) * sizeof(tray_hit), cudaMemcpyDeviceToHost, s->s_out));
                if (costs) CU(cudaMemcpyAsync(s->h_costs[ps], d_costs + j * chunk, chunk_len(j) * sizeof(tray_ray_cost), cudaMemcpyDeviceToHost, s->s_out));
                CU(cudaEventRecord(s->e_out[ps], s->s_out));
            }
            if (i >= 2) {                                                               // chunk i-2: hand its hits to the caller
                const uint64_t j = i - 2; const int ps = (int)(j & 1);
                CU(cudaEventSynchronize(s->e_out[ps]));
                tray::par_copy(hits + j * chunk, s->h_hits[ps], chunk_len(j) * sizeof(tray_hit));
                if (costs) tray::par_copy(costs + j * chunk, s->h_costs[ps], chunk_len(j) * sizeof(tray_ray_cost));
            }
        }
        CU(cudaEventRecord(s->ev[1], s->stream));
        CU(cudaStreamSynchronize(s->stream));
        CU(cudaEventElapsedTime(&k, s->ev[0], s->ev[1]));       // span of the GPU work, uploads it waited for included
    }
    if (s->counting) {
        rc = read_counters(s->d_cursor, s->stream, 0, &s->cnt_primary); if (rc) return rc;
        memset(&s->cnt_bounce, 0, sizeof s->cnt_bounce);
        drop_placeholder_root(s);
    }
    rc = check_overflow(s->d_overflow, s->stream);
    if (rc) return rc;
    if (ms_kernel) *ms_kernel = k;
    if (ms_total) *ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return TRAY_OK;
}
}  // namespace

extern "C" {

int tray_cuda_trace_device(tray_scene* s, const tray_ray* d_rays, uint64_t n, tray_hit* d_hits, void* stream, float* ms_kernel) {
    return trace_device_impl(s, d_rays, n, d_hits, nullptr, stream, ms_kernel, false);
}
int tray_cuda_trace(tray_scene* s, const tray_ray* rays, uint64_t n, tray_hit* hits, float* ms_kernel, float* ms_total) {
    return trace_impl(s, rays, n, hits, nullptr, ms_kernel, ms_total, false);
}
int tray_cuda_trace_any_device(tray_scene* s, const tray_ray* d_rays, uint64_t n, tray_hit* d_hits, void* stream, float* ms_kernel) {
    return trace_device_impl(s, d_rays, n, d_hits, nullptr, stream, ms_kernel, true);
}
int tray_cuda_trace_any(tray_scene* s, const tray_ray* rays, uint64_t n, tray_hit* hits, float* ms_kernel, float* ms_total) {
    return trace_impl(s, rays, n, hits, nullptr, ms_kernel, ms_total, true);
}
int tray_cuda_trace_cost_device(tray_scene* s, const tray_ray* d_rays, uint64_t n, int any_hit, tray_hit* d_hits, tray_ray_cost* d_costs,
                                void* stream, float* ms_kernel) {
    if (!s || (n && (!d_rays || !d_hits || !d_costs))) return fail(TRAY_ERR_ARG, "NULL argument");
    if ((uintptr_t)d_costs & 15u) return fail(TRAY_ERR_ARG, "d_costs must be 16-byte aligned (one vector store per record)");
    if (s->variant) return fail(TRAY_ERR_ARG, "%s", VARIANT_REFUSAL);     // before any change of state
    return trace_device_impl(s, d_rays, n, d_hits, d_costs, stream, ms_kernel, any_hit != 0);
}
int tray_cuda_trace_cost(tray_scene* s, const tray_ray* rays, uint64_t n, int any_hit, tray_hit* hits, tray_ray_cost* costs,
                         float* ms_kernel, float* ms_total) {
    if (!s || (n && (!rays || !hits || !costs))) return fail(TRAY_ERR_ARG, "NULL argument");
    if (s->variant) return fail(TRAY_ERR_ARG, "%s", VARIANT_REFUSAL);
    return trace_impl(s, rays, n, hits, costs, ms_kernel, ms_total, any_hit != 0);
}

uint64_t tray_cuda_shard_pixels(uint32_t w, uint32_t h, uint32_t shard, uint32_t shards) {
    if (shards == 0) shards = 1;
    const uint32_t tx = (w + 31) / 32, ty = (h + 7) / 8;
    uint64_t n = 0;
    for (uint64_t k = shard; k < (uint64_t)tx * ty; k += shards) {
        const uint32_t x0 = (uint32_t)(k % tx) * 32, y0 = (uint32_t)(k / tx) * 8;
        const uint32_t cw = x0 + 32 <= w ? 32 : w - x0, ch = y0 + 8 <= h ? 8 : h - y0;
        n += (uint64_t)cw * ch;
    }
    return n;
}

uint64_t tray_cuda_shard_items(uint32_t w, uint32_t h, uint32_t shard, uint32_t shards) {
    return local_items(w, h, shard, shards ? shards : 1);
}

int tray_cuda_scene_set_frames_in_flight(tray_scene* s, uint32_t n) {
    if (!s || n < 1 || n > TRAY_MAX_FRAMES_IN_FLIGHT) return fail(TRAY_ERR_ARG, "frames in flight must be 1 .. %d", TRAY_MAX_FRAMES_IN_FLIGHT);
    CU(cudaSetDevice(s->device));
    if (const int rc = sync_streams(s, /*scene_stream_first=*/false)) return rc;
    if (s->cur >= (int)n) {
        // The last frame's slot does not survive the switch: its frame moves to slot n - 1, and that slot's older frame moves
        // out, so that "the last frame" is still the latest render; the next render takes slot 0.  Every stream is idle here, so
        // buffers, cursors and events move freely.  The streams stay with their slots, and the error word follows the frame.
        FrameSlot& a = s->slot[s->cur];
        FrameSlot& b = s->slot[n - 1];
        std::swap(a, b);
        std::swap(a.own_stream, b.own_stream);
        std::swap(a.d_flag, b.d_flag);
        uint32_t wa = 0, wb = 0;
        CU(cudaMemcpy(&wa, a.d_flag, 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(&wb, b.d_flag, 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(a.d_flag, &wb, 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(b.d_flag, &wa, 4, cudaMemcpyHostToDevice));
        s->cur = (int)n - 1;
    }
    s->n_slots = (int)n;
    return TRAY_OK;
}

int tray_cuda_scene_fence(tray_scene* s, void* stream) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    CU(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    for (int k = 0; k < s->n_slots; k++) {
        cudaStream_t fs = slot_stream(s, k);
        if (fs == st) continue;
        CU(cudaEventRecord(s->slot[k].done, fs));
        CU(cudaStreamWaitEvent(st, s->slot[k].done, 0));
    }
    return TRAY_OK;
}

int tray_cuda_scene_frame_stream(tray_scene* s, int which, void** stream) {
    if (!s || !stream || which < -1 || which >= TRAY_MAX_FRAMES_IN_FLIGHT) return fail(TRAY_ERR_ARG, "bad argument");
    *stream = (void*)slot_stream(s, which < 0 ? s->cur : which);
    return TRAY_OK;
}

// ---- frame completion across GPUs without a kernel: stream memory operations ---------------------------------------------
// cuStreamWriteValue32 / cuStreamWaitValue32 are executed by the stream front-end, so they need no SM slot — unlike a collective
// kernel, which cannot start while the persistent grid of the NEXT frame fills every slot of the chip.  They are driver-API
// entry points: resolved at run time (cudaGetDriverEntryPoint), the library does not link libcuda.
namespace {
typedef int (*stream_memop32_fn)(void* stream, unsigned long long addr, unsigned int value, unsigned int flags);
stream_memop32_fn g_write32 = nullptr, g_wait32 = nullptr;
int resolve_memops() {
    if (g_write32 && g_wait32) return TRAY_OK;
    void* w = nullptr; void* q = nullptr;
    cudaDriverEntryPointQueryResult st;
    CU(cudaGetDriverEntryPoint("cuStreamWriteValue32", &w, cudaEnableDefault, &st));
    if (st != cudaDriverEntryPointSuccess || !w) return fail(TRAY_ERR_CUDA, "cuStreamWriteValue32 is not available in this driver");
    CU(cudaGetDriverEntryPoint("cuStreamWaitValue32", &q, cudaEnableDefault, &st));
    if (st != cudaDriverEntryPointSuccess || !q) return fail(TRAY_ERR_CUDA, "cuStreamWaitValue32 is not available in this driver");
    g_write32 = (stream_memop32_fn)w; g_wait32 = (stream_memop32_fn)q;
    return TRAY_OK;
}
}  // namespace

int tray_cuda_frame_signal(tray_scene* s, void* d_flag, uint32_t value) {
    if (!s || !d_flag) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    int rc = resolve_memops(); if (rc) return rc;
    const int e = g_write32((void*)slot_stream(s, s->cur), (unsigned long long)(uintptr_t)d_flag, value, 0u /* CU_STREAM_WRITE_VALUE_DEFAULT */);
    if (e) return fail(TRAY_ERR_CUDA, "cuStreamWriteValue32 failed (CUresult %d)", e);
    return TRAY_OK;
}

int tray_cuda_frame_wait_flag(tray_scene* s, const void* d_flag, uint32_t value, int before_next_frame) {
    if (!s || !d_flag) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    int rc = resolve_memops(); if (rc) return rc;
    const int k = before_next_frame ? next_slot(s) : s->cur;
    const int e = g_wait32((void*)slot_stream(s, k), (unsigned long long)(uintptr_t)d_flag, value, 0u /* CU_STREAM_WAIT_VALUE_GEQ */);
    if (e) return fail(TRAY_ERR_CUDA, "cuStreamWaitValue32 failed (CUresult %d)", e);
    return TRAY_OK;
}

int tray_cuda_scene_after(tray_scene* s, void* stream) {
    if (!s || !stream) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    CU(cudaEventRecord(s->ev_after, (cudaStream_t)stream));
    for (int k = 0; k < TRAY_MAX_FRAMES_IN_FLIGHT; k++)
        if (slot_stream(s, k) != (cudaStream_t)stream) CU(cudaStreamWaitEvent(slot_stream(s, k), s->ev_after, 0));
    return TRAY_OK;
}

}  // extern "C"

namespace {
// the frame of tray_cuda_render in slot s->cur, its arguments checked; it writes the slot's frame record before its launches
int render_slot(tray_scene* s, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t flags,
                uint32_t shard, uint32_t shards, float* ms_primary, float* ms_bounce) {
    FrameSlot& f = s->slot[s->cur];
    cudaStream_t st = slot_stream(s, s->cur);
    const uint64_t items_cap = local_items(w, h, 0, shards);   // every shard's buffers have the size of the largest (gather)
    const bool want_count = (flags & TRAY_RENDER_COUNTERS) != 0;
    const bool bounce = (flags & TRAY_RENDER_BOUNCE) != 0, rgba = (flags & TRAY_RENDER_RGBA) != 0;
    const bool keep_rays = (flags & TRAY_RENDER_KEEP_RAYS) != 0;
    const bool any_ao = (flags & TRAY_RENDER_ANYHIT_AO) != 0;
    const bool overlap = bounce && !any_ao && !s->variant && ((flags & TRAY_RENDER_OVERLAP) != 0 || s->overlap_default);
    const bool keep_cost = want_count && s->ray_cost;
    if (items_cap > f.f_cap || (keep_rays && !f.d_brays_item) || (keep_cost && !f.d_cost)) {
        const uint64_t cap = items_cap > f.f_cap ? items_cap : f.f_cap;
        CU(cudaStreamSynchronize(st));
        free_frame_buffers(f);
        const uint64_t c1 = cap ? cap : 1;
        CU(cudaMalloc(&f.d_primary, c1 * sizeof(tray_hit)));
        CU(cudaMalloc(&f.d_bounce, c1 * sizeof(tray_hit)));
        CU(cudaMalloc(&f.d_rgba, c1 * sizeof(uchar4)));
        CU(cudaMalloc(&f.d_prays, c1 * sizeof(tray_ray)));
        CU(cudaMalloc(&f.d_brays, c1 * sizeof(tray_ray)));
        CU(cudaMalloc(&f.d_bitem, c1 * sizeof(uint32_t)));
        if (keep_rays) CU(cudaMalloc(&f.d_brays_item, c1 * sizeof(tray_ray)));
        if (keep_cost) CU(cudaMalloc(&f.d_cost, 2 * c1 * sizeof(tray_ray_cost)));
        CU(cudaMemsetAsync(f.d_primary, 0xff, c1 * sizeof(tray_hit), st));
        CU(cudaMemsetAsync(f.d_bounce, 0xff, c1 * sizeof(tray_hit), st));
        CU(cudaMemsetAsync(f.d_rgba, 0, c1 * sizeof(uchar4), st));
        f.f_cap = cap;
    }
    FrameParams F; frame_params(F, view, w, h, frame_count, shard, shards);
    f.f_has_bounce = bounce; f.f_has_rgba = rgba && !s->frame_target; f.f_has_rays = keep_rays && bounce;
    f.f_target = rgba ? s->frame_target : nullptr;
    f.f_has_cost = keep_cost;
    f.last_frame = F;
    if (F.n_items == 0) {                        // a shard without tiles: no launch, and nothing to count
        if (ms_primary) *ms_primary = 0.f;
        if (ms_bounce) *ms_bounce = 0.f;
        if (want_count) { memset(&s->cnt_primary, 0, sizeof s->cnt_primary); memset(&s->cnt_bounce, 0, sizeof s->cnt_bounce); }
        return TRAY_OK;
    }
    const unsigned gen_grid = (F.n_items + 255) / 256;
    uint32_t* d_nbrays = (uint32_t*)(f.d_cursor + CURSOR_N_BOUNCE);
    const bool timed = ms_primary || ms_bounce;

    // ---- primary: generate rays, trace ----
    // ray costs: primary records at d_cost[item], bounce records at d_cost[n_items + item]; a pixel that shoots no bounce ray
    // writes no bounce record, so that half starts zeroed
    tray_ray_cost* const d_cost_bounce = keep_cost ? f.d_cost + F.n_items : nullptr;
    if (keep_cost && bounce) CU(cudaMemsetAsync(d_cost_bounce, 0, (size_t)F.n_items * sizeof(tray_ray_cost), st));
    if (timed) CU(cudaEventRecord(f.ev[0], st));
    tray::raygen_primary_kernel<<<gen_grid, 256, 0, st>>>(F, f.d_prays);
    CU(cudaGetLastError());
    TraceParams P; base_params(s, P);
    P.rays = f.d_prays; P.n_work = F.n_items; P.hits_out = f.d_primary; P.overflow = f.d_flag;
    P.frame = F; P.row_major = s->frame_target ? 1u : 0u;
    uchar4* const rgba_dst = s->frame_target ? s->frame_target : f.d_rgba;
    P.rgba_out = (rgba && !bounce) ? rgba_dst : nullptr; P.shade_mode = SHADE_PRIMARY;
    P.ray_cost = keep_cost ? f.d_cost : nullptr;
    if (overlap) {
        // one launch for the whole frame (trace_kernel<FRAME>): the bounce rays of finished tiles fill the primary pass's drain
        CU(cudaMemsetAsync(f.d_units, 0, sizeof(uint32_t), st));
        CU(cudaMemsetAsync(f.d_primary, 0xff, (size_t)F.n_items * sizeof(tray_hit), st));     // "not there yet" for every primary hit
        P.rgba_out = rgba ? rgba_dst : nullptr;
        P.bounce_out = f.d_bounce; P.rays_by_item = keep_rays ? f.d_brays_item : nullptr; P.gen_min = s->gen_min;
        P.gen_rays = f.d_brays;
        P.unit_cursor = f.d_units; P.n_units = (uint32_t)(F.n_items / 32);
    }
    int rc = launch(s, P, st, f.d_cursor, 0, want_count, false, false, overlap);
    if (rc) return rc;
    if (timed) CU(cudaEventRecord(f.ev[1], st));
    if (overlap && timed) CU(cudaEventRecord(f.ev[2], st));

    // ---- bounce: generate + compact rays of hit pixels, trace ----
    if (bounce && !overlap) {
        CU(cudaMemsetAsync(d_nbrays, 0, sizeof(uint32_t), st));
        auto gen = s->tri_stride == 64 ? tray::raygen_bounce_kernel<64> : s->tri_stride == 24 ? tray::raygen_bounce_kernel<24> : tray::raygen_bounce_kernel<48>;
        gen<<<(F.n_items + BOUNCE_BLOCK - 1) / BOUNCE_BLOCK, BOUNCE_BLOCK, 0, st>>>(F, s->d_tris, f.d_primary, f.d_brays, f.d_bitem, d_nbrays, f.d_bounce,
                                             rgba ? rgba_dst : nullptr, keep_rays ? f.d_brays_item : nullptr, P.row_major);
        CU(cudaGetLastError());
        TraceParams B; base_params(s, B);
        B.rays = f.d_brays; B.ray_item = f.d_bitem; B.n_work = F.n_items; B.n_work_dev = d_nbrays;   // count stays on the device
        B.overflow = f.d_flag; B.frame = F; B.row_major = P.row_major;
        B.hits_out = f.d_bounce; B.rgba_out = rgba ? rgba_dst : nullptr; B.shade_mode = any_ao ? SHADE_OCCLUSION : SHADE_BOUNCE;
        B.ray_cost = d_cost_bounce;
        rc = launch(s, B, st, f.d_cursor, 1, want_count, any_ao);
        if (rc) return rc;
        if (timed) CU(cudaEventRecord(f.ev[2], st));
    }
    if (keep_cost) { rc = drop_placeholder_costs(s, f.d_cost, F.n_items, st); if (rc) return rc; }   // (an empty scene shoots no bounce ray)
    if (timed) {
        CU(cudaStreamSynchronize(st));
        float a = 0.f, b = 0.f;
        CU(cudaEventElapsedTime(&a, f.ev[0], f.ev[1]));
        if (bounce) CU(cudaEventElapsedTime(&b, f.ev[1], f.ev[2]));
        if (ms_primary) *ms_primary = a;
        if (ms_bounce) *ms_bounce = b;
        rc = check_overflow(f.d_flag, st); if (rc) return rc;
    }
    if (want_count) {
        rc = read_counters(f.d_cursor, st, 0, &s->cnt_primary); if (rc) return rc;
        if (bounce) { rc = read_counters(f.d_cursor, st, 1, &s->cnt_bounce); if (rc) return rc; }
        else memset(&s->cnt_bounce, 0, sizeof s->cnt_bounce);
        // rays generated for pixels outside the frame (tmax = 0) are not rays of the workload
        const uint64_t pad = (uint64_t)F.n_items - tray_cuda_shard_pixels(w, h, shard, shards);
        s->cnt_primary.rays -= pad; s->cnt_primary.nodes -= pad;
        drop_placeholder_root(s);
    }
    return TRAY_OK;
}
}  // namespace

extern "C" {

int tray_cuda_render(tray_scene* s, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t flags,
                     uint32_t shard, uint32_t shards, float* ms_primary, float* ms_bounce) {
    // every refusal comes before the first change of state: a refused render leaves the last frame, the slot the next render
    // takes and the counting state of batch traces as they were
    if (!s || !view) return fail(TRAY_ERR_ARG, "NULL argument");
    if (shards == 0) shards = 1;
    if (w == 0 || h == 0 || shard >= shards) return fail(TRAY_ERR_ARG, "bad frame size / shard (%ux%u, %u of %u)", w, h, shard, shards);
    if ((uint64_t)((w + 31) / 32) * ((h + 7) / 8) * 256ull > INDEX_MASK) return fail(TRAY_ERR_ARG, "frame too large");
    // the launches' own check (launch()), made here: the primary launch counts with TRAY_RENDER_COUNTERS, the bounce launch is an
    // any-hit launch with TRAY_RENDER_ANYHIT_AO (TRAY_RENDER_OVERLAP is ignored under a variant)
    if (s->variant && ((flags & TRAY_RENDER_COUNTERS) || ((flags & TRAY_RENDER_BOUNCE) && (flags & TRAY_RENDER_ANYHIT_AO))))
        return fail(TRAY_ERR_ARG, "%s", VARIANT_REFUSAL);
    CU(cudaSetDevice(s->device));
    s->cur = next_slot(s);
    const int rc = render_slot(s, view, w, h, frame_count, flags, shard, shards, ms_primary, ms_bounce);
    // A frame that failed on its way is no frame: downloads of it fail rather than return what the slot held before.  A stack
    // overflow is reported for a frame whose launches ran to the end.
    if (rc != TRAY_OK && rc != TRAY_ERR_OVERFLOW) s->slot[s->cur].last_frame.width = 0;
    return rc;
}

int tray_cuda_render_timed(tray_scene* s, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t flags,
                           uint32_t shard, uint32_t shards, float* ms_frame) {
    if (!s || !view || !ms_frame) return fail(TRAY_ERR_ARG, "NULL argument");
    CU(cudaSetDevice(s->device));
    const int k = next_slot(s);                                               // the slot tray_cuda_render is about to take
    cudaStream_t st = slot_stream(s, k);
    CU(cudaEventRecord(s->slot[k].ev[0], st));
    int rc = tray_cuda_render(s, view, w, h, frame_count, flags, shard, shards, nullptr, nullptr);
    if (rc) return rc;
    CU(cudaEventRecord(s->slot[k].ev[3], st));
    CU(cudaEventSynchronize(s->slot[k].ev[3]));
    CU(cudaEventElapsedTime(ms_frame, s->slot[k].ev[0], s->slot[k].ev[3]));
    return check_overflow(s->slot[k].d_flag, st);    // synchronising point: a stack overflow / watchdog flag must not pass as TRAY_OK
}

int tray_cuda_counters(tray_scene* s, tray_counters* primary, tray_counters* bounce) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    if (primary) *primary = s->cnt_primary;
    if (bounce) *bounce = s->cnt_bounce;
    return TRAY_OK;
}

int tray_cuda_frame_device_ptrs(tray_scene* s, void** d_primary, void** d_bounce, void** d_rgba) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    const FrameSlot& f = s->slot[s->cur];
    if (d_primary) *d_primary = f.d_primary;
    if (d_bounce) *d_bounce = f.d_bounce;
    if (d_rgba) *d_rgba = f.d_rgba;
    return TRAY_OK;
}

}  // extern "C"

namespace {
// the last frame's compact buffer `d_src`, untiled into the row-major `d_dst` on the frame's stream
template <typename T>
int untile_last_frame(tray_scene* s, const T* d_src, T* d_dst) {
    const FrameParams& F = s->slot[s->cur].last_frame;
    cudaStream_t st = slot_stream(s, s->cur);
    if (F.shard_count > 1) CU(cudaMemsetAsync(d_dst, 0, (uint64_t)F.width * F.height * sizeof(T), st));   // pixels of other shards read as zero
    if (F.n_items) {
        tray::untile_kernel<T><<<(F.n_items + 255) / 256, 256, 0, st>>>(F, d_src, d_dst);
        CU(cudaGetLastError());
    }
    return TRAY_OK;
}

template <typename T>
int download(tray_scene* s, const T* d_src, T* host_dst) {
    const FrameParams& F = s->slot[s->cur].last_frame;
    cudaStream_t st = slot_stream(s, s->cur);
    const uint64_t bytes = (uint64_t)F.width * F.height * sizeof(T);
    if (bytes > s->untiled_cap) {
        cudaFree(s->d_untiled); s->d_untiled = nullptr; s->untiled_cap = 0;
        CU(cudaMalloc(&s->d_untiled, bytes));
        s->untiled_cap = bytes;
    }
    if (const int rc = untile_last_frame(s, d_src, (T*)s->d_untiled)) return rc;
    CU(cudaMemcpyAsync(host_dst, s->d_untiled, bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return TRAY_OK;
}
}  // namespace

extern "C" {

int tray_cuda_frame_download(tray_scene* s, tray_hit* primary, tray_hit* bounce, tray_ray* bounce_rays, uint8_t* rgba) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    const FrameSlot& f = s->slot[s->cur];
    if (f.last_frame.width == 0) return fail(TRAY_ERR_ARG, "no frame has been rendered");
    CU(cudaSetDevice(s->device));
    int rc;
    if (primary) { rc = download<tray_hit>(s, f.d_primary, primary); if (rc) return rc; }
    if (bounce) {
        if (!f.f_has_bounce) return fail(TRAY_ERR_ARG, "last frame was rendered without TRAY_RENDER_BOUNCE");
        rc = download<tray_hit>(s, f.d_bounce, bounce); if (rc) return rc;
    }
    if (bounce_rays) {
        if (!f.f_has_rays) return fail(TRAY_ERR_ARG, "last frame was rendered without the keep-bounce-rays flag (0x8)");
        rc = download<tray_ray>(s, f.d_brays_item, bounce_rays); if (rc) return rc;
    }
    if (rgba) {
        if (!f.f_has_rgba) return fail(TRAY_ERR_ARG, "last frame was rendered without TRAY_RENDER_RGBA");
        rc = download<uchar4>(s, f.d_rgba, (uchar4*)rgba); if (rc) return rc;
    }
    return check_overflow(f.d_flag, slot_stream(s, s->cur));
}

int tray_cuda_frame_download_cost(tray_scene* s, tray_ray_cost* primary, tray_ray_cost* bounce) {
    if (!s) return fail(TRAY_ERR_ARG, "NULL scene");
    const FrameSlot& f = s->slot[s->cur];
    if (f.last_frame.width == 0) return fail(TRAY_ERR_ARG, "no frame has been rendered");
    if (!f.f_has_cost) return fail(TRAY_ERR_ARG, "last frame kept no ray costs (it needs tray_cuda_scene_set_ray_cost and TRAY_RENDER_COUNTERS)");
    if (bounce && !f.f_has_bounce) return fail(TRAY_ERR_ARG, "last frame was rendered without TRAY_RENDER_BOUNCE");
    CU(cudaSetDevice(s->device));
    int rc;
    if (primary) { rc = download<tray_ray_cost>(s, f.d_cost, primary); if (rc) return rc; }
    if (bounce) { rc = download<tray_ray_cost>(s, f.d_cost + f.last_frame.n_items, bounce); if (rc) return rc; }
    return check_overflow(f.d_flag, slot_stream(s, s->cur));
}

int tray_cuda_frame_readback_begin(tray_scene* s, uint8_t* rgba, uint32_t slot) {
    if (!s || !rgba || slot >= TRAY_READBACK_SLOTS) return fail(TRAY_ERR_ARG, "bad argument");
    const FrameSlot& f = s->slot[s->cur];
    cudaStream_t st = slot_stream(s, s->cur);
    if (f.last_frame.width == 0 || (!f.f_has_rgba && !f.f_target)) return fail(TRAY_ERR_ARG, "last frame was rendered without TRAY_RENDER_RGBA");
    CU(cudaSetDevice(s->device));
    const uint64_t bytes = (uint64_t)f.last_frame.width * f.last_frame.height * sizeof(uchar4);
    if (s->stage_busy[slot]) {                       // the previous copy out of this staging buffer must have landed
        CU(cudaEventSynchronize(s->ev_copied[slot]));
        s->stage_busy[slot] = false;
    }
    if (bytes > s->stage_cap[slot]) {
        cudaFree(s->d_stage[slot]); s->d_stage[slot] = nullptr; s->stage_cap[slot] = 0;
        CU(cudaMalloc(&s->d_stage[slot], bytes));
        s->stage_cap[slot] = bytes;
    }
    if (f.f_target) {
        // the frame was rendered into a row-major frame target (all shards' pixels, once the caller's barrier has passed):
        // snapshot it, so that the next frame may overwrite the target while this one travels to the host
        CU(cudaMemcpyAsync(s->d_stage[slot], f.f_target, bytes, cudaMemcpyDeviceToDevice, st));
    } else if (const int rc = untile_last_frame(s, f.d_rgba, s->d_stage[slot])) {
        return rc;
    }
    // the error word travels with the frame (a stream synchronise here would undo the overlap): taken on the frame's stream,
    // behind the frame's launches and ahead of the next frame on that slot, and reported by _wait
    CU(cudaMemcpyAsync(s->h_flag + slot, f.d_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemsetAsync(f.d_flag, 0, sizeof(uint32_t), st));
    CU(cudaEventRecord(s->ev_untiled[slot], st));
    CU(cudaStreamWaitEvent(s->copy_stream, s->ev_untiled[slot], 0));
    CU(cudaMemcpyAsync(rgba, s->d_stage[slot], bytes, cudaMemcpyDeviceToHost, s->copy_stream));
    CU(cudaEventRecord(s->ev_copied[slot], s->copy_stream));
    s->stage_busy[slot] = true;
    return TRAY_OK;
}

int tray_cuda_frame_readback_wait(tray_scene* s, uint32_t slot) {
    if (!s || slot >= TRAY_READBACK_SLOTS) return fail(TRAY_ERR_ARG, "bad argument");
    if (!s->stage_busy[slot]) return TRAY_OK;
    CU(cudaSetDevice(s->device));
    CU(cudaEventSynchronize(s->ev_copied[slot]));
    s->stage_busy[slot] = false;
    const uint32_t fl = s->h_flag[slot];
    s->h_flag[slot] = 0u;
    return flag_status(fl);
}

int tray_cuda_start(const void* bvh_bytes, uint64_t bvh_len, const void* instance_bytes, uint64_t instance_len,
                    const void* tri_bytes, uint64_t tri_len, uint32_t tri_stride, uint32_t tlas_start, int use_tlas,
                    const tray_view* view, uint32_t width, uint32_t height, float render_time_s, int benchmark,
                    int animate, int device, float* out_min_ms, float* out_mean_ms, uint32_t* out_frames) {
    if (const int rc = check_start_args(view, bvh_len, tri_len, tri_stride, instance_len)) return rc;
    tray_scene* s = nullptr;
    int rc = tray_cuda_scene_create(bvh_bytes, bvh_len / 80, tri_bytes, tri_len / tri_stride, tri_stride,
                                    use_tlas ? (const uint32_t*)instance_bytes : nullptr,
                                    use_tlas ? (uint32_t)(instance_len / 4) : 0u, tlas_start, device, &s);
    if (rc) return rc;
    uint32_t flags = TRAY_RENDER_BOUNCE | TRAY_RENDER_RGBA;
    // Two bit-identical ways to render the frame (two launches, or the one-launch frame kernel): which is faster depends on
    // how long the scene's drain phases are, so a short untimed calibration picks one (TRAY_CUDA_OVERLAP=0/1 forces it).
    if (!getenv("TRAY_CUDA_OVERLAP")) {
        float best[2] = { 3.402823466e+38f, 3.402823466e+38f };
        for (int rep = 0; rep < 4 && !rc; rep++)
            for (int path = 0; path < 2 && !rc; path++) {
                float ms = 0.f;
                rc = tray_cuda_render_timed(s, view, width, height, 0, flags | (path ? TRAY_RENDER_OVERLAP : 0u), 0, 1, &ms);
                if (!rc && rep > 0 && ms < best[path]) best[path] = ms;          // the first frame of each path allocates
            }
        if (rc) { tray_cuda_scene_destroy(s); return rc; }
        if (best[1] < best[0]) flags |= TRAY_RENDER_OVERLAP;
    }
    rc = start_loop([&](uint32_t fc) { return tray_cuda_render(s, view, width, height, fc, flags, 0, 1, nullptr, nullptr); },
                    [&](uint32_t fc, float* ms) { return tray_cuda_render_timed(s, view, width, height, fc, flags, 0, 1, ms); },
                    [&] { return tray_cuda_sync(s); },
                    render_time_s, benchmark, animate, out_min_ms, out_mean_ms, out_frames);
    tray_cuda_scene_destroy(s);
    return rc;
}

}  // extern "C"

// ---- CPU-style hit records: (geometry_id, primitive_id) -----------------------------------------------------------------
namespace {
// global triangle index -> (object whose range holds it, index inside that object's BVH-ordered triangle array)
__global__ void hits_to_geometry_kernel(const tray_hit* __restrict__ hits, uint64_t n, const uint32_t* __restrict__ offsets, uint32_t n_geom,
                                        uint32_t* __restrict__ geometry_id, uint32_t* __restrict__ primitive_id) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t prim = hits[i].prim;
    uint32_t g = 0xffffffffu, local = prim;                  // miss: RayHit::none()
    if (prim != 0xffffffffu && n_geom) {
        uint32_t lo = 0, hi = n_geom;                        // last g with offsets[g] <= prim
        while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(offsets + mid) <= prim) lo = mid; else hi = mid; }
        g = lo; local = prim - __ldg(offsets + lo);
    }
    geometry_id[i] = g; primitive_id[i] = local;
}
}  // namespace

extern "C" {

int tray_cuda_scene_set_geometry_offsets(tray_scene* s, const uint32_t* tri_offsets, uint32_t n_geometries) {
    if (!s || (n_geometries && !tri_offsets)) return fail(TRAY_ERR_ARG, "NULL argument");
    if (n_geometries) {
        if (tri_offsets[0] != 0u || tri_offsets[n_geometries] != (uint32_t)s->n_tris) return fail(TRAY_ERR_ARG, "tri_offsets must run from 0 to n_tris (%llu)", (unsigned long long)s->n_tris);
        for (uint32_t g = 0; g < n_geometries; g++)
            if (tri_offsets[g] > tri_offsets[g + 1]) return fail(TRAY_ERR_ARG, "tri_offsets must ascend (entry %u)", g);
    }
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    cudaFree(s->d_geom_offsets); s->d_geom_offsets = nullptr; s->n_geometries = 0;
    if (n_geometries) {
        CU(cudaMalloc(&s->d_geom_offsets, (size_t)(n_geometries + 1) * 4));
        CU(cudaMemcpy(s->d_geom_offsets, tri_offsets, (size_t)(n_geometries + 1) * 4, cudaMemcpyHostToDevice));
        s->n_geometries = n_geometries;
    }
    return TRAY_OK;
}

int tray_cuda_hits_to_geometry(tray_scene* s, const tray_hit* hits, uint64_t n, uint32_t* geometry_id, uint32_t* primitive_id) {
    if (!s || (n && (!hits || !geometry_id || !primitive_id))) return fail(TRAY_ERR_ARG, "NULL argument");
    if (n == 0) return TRAY_OK;
    CU(cudaSetDevice(s->device));
    tray_hit* d_h = nullptr; uint32_t* d_o = nullptr;
    CU(cudaMalloc(&d_h, n * sizeof(tray_hit)));
    if (cudaMalloc(&d_o, n * 8) != cudaSuccess) { cudaFree(d_h); return fail(TRAY_ERR_CUDA, "cudaMalloc failed"); }
    auto body = [&]() -> int {
        CU(cudaMemcpyAsync(d_h, hits, n * sizeof(tray_hit), cudaMemcpyHostToDevice, s->stream));
        hits_to_geometry_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(d_h, n, s->d_geom_offsets, s->n_geometries, d_o, d_o + n);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(geometry_id, d_o, n * 4, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemcpyAsync(primitive_id, d_o + n, n * 4, cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
        return TRAY_OK;
    };
    const int rc = body();
    cudaFree(d_h); cudaFree(d_o);
    return rc;
}

}  // extern "C"

// ---- one process, several GPUs -----------------------------------------------------------------------------------------
// The reference's slot is ONE call from ONE host thread (rt_gpu_software.rs:24-32).  A tray_group keeps that shape on a box
// with several GPUs: the BVH is replicated (one tray_scene per device), the frame's 32x8 tiles are dealt round-robin to the
// devices, and every device's traversal kernels store their finished pixels straight into ONE row-major frame on devices[0]
// through peer access (cudaDeviceEnablePeerAccess: no IPC, no NCCL, no torch).  "Frame complete" is a set of events: device
// 0's stream waits for the event each other device records behind its last launch.
struct tray_group {
    std::vector<tray_scene*> scenes;
    std::vector<int> devices;
    uchar4* target[TRAY_MAX_FRAMES_IN_FLIGHT] = {};    // row-major frames on devices[0], one per frame in flight
    uint64_t target_bytes = 0;
    int in_flight = 1, cur = 0;
    cudaEvent_t ev_snap[TRAY_MAX_FRAMES_IN_FLIGHT] = {};   // devices[0]: the frame in target[i] has been copied out (readback)
    bool snap_pending[TRAY_MAX_FRAMES_IN_FLIGHT] = {};
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;      // devices[0]: frame timing
    // exchange 1 ("push", default): every device keeps its compact shard and moves it with one peer DMA copy into staging[] on
    // devices[0], which untiles all shards in one launch; exchange 0: the kernels store pixels straight into the frame
    int exchange = 1;
    uchar4* staging[TRAY_MAX_FRAMES_IN_FLIGHT] = {};
    uint64_t staging_bytes = 0;
    cudaEvent_t ev_staged[TRAY_MAX_FRAMES_IN_FLIGHT] = {};  // devices[0]: staging[i] has been untiled (it may be overwritten)
    bool staged_pending[TRAY_MAX_FRAMES_IN_FLIGHT] = {};
};

namespace {
int group_ensure_target(tray_group* g, uint32_t w, uint32_t h) {
    const uint64_t bytes = (uint64_t)w * h * 4;
    if (bytes <= g->target_bytes) return TRAY_OK;
    CU(cudaSetDevice(g->devices[0]));
    for (auto* sc : g->scenes) { int rc = tray_cuda_sync(sc); if (rc) return rc; }
    CU(cudaSetDevice(g->devices[0]));
    for (int i = 0; i < TRAY_MAX_FRAMES_IN_FLIGHT; i++) {
        cudaFree(g->target[i]); g->target[i] = nullptr;
        CU(cudaMalloc(&g->target[i], bytes));
        CU(cudaMemset(g->target[i], 0, bytes));
    }
    g->target_bytes = bytes;
    return TRAY_OK;
}
int group_ensure_staging(tray_group* g, uint32_t w, uint32_t h) {
    const uint64_t bytes = (uint64_t)g->scenes.size() * local_items(w, h, 0, (uint32_t)g->scenes.size()) * 4;
    if (bytes <= g->staging_bytes) return TRAY_OK;
    for (auto* sc : g->scenes) { int rc = tray_cuda_sync(sc); if (rc) return rc; }
    CU(cudaSetDevice(g->devices[0]));
    for (int i = 0; i < TRAY_MAX_FRAMES_IN_FLIGHT; i++) {
        cudaFree(g->staging[i]); g->staging[i] = nullptr;
        CU(cudaMalloc(&g->staging[i], bytes));
        g->staged_pending[i] = false;
    }
    g->staging_bytes = bytes;
    return TRAY_OK;
}
}  // namespace

extern "C" {

void tray_cuda_group_destroy(tray_group* g) {
    if (!g) return;
    for (auto* sc : g->scenes) tray_cuda_scene_destroy(sc);
    if (!g->devices.empty()) {
        cudaSetDevice(g->devices[0]);
        for (int i = 0; i < TRAY_MAX_FRAMES_IN_FLIGHT; i++) {
            cudaFree(g->target[i]); cudaFree(g->staging[i]);
            if (g->ev_snap[i]) cudaEventDestroy(g->ev_snap[i]);
            if (g->ev_staged[i]) cudaEventDestroy(g->ev_staged[i]);
        }
        if (g->ev_t0) cudaEventDestroy(g->ev_t0);
        if (g->ev_t1) cudaEventDestroy(g->ev_t1);
    }
    delete g;
}

int tray_cuda_group_create(const void* nodes, uint64_t n_nodes, const void* tris, uint64_t n_tris, uint32_t tri_stride,
                           const uint32_t* blas_offsets, uint32_t n_instances, uint32_t tlas_start,
                           const int* devices, int n_devices, tray_group** out) {
    if (!out) return fail(TRAY_ERR_ARG, "out_group is NULL");
    *out = nullptr;
    const int ndev = tray_cuda_device_count();
    if (ndev == 0) return fail(TRAY_ERR_NO_DEVICE, "no CUDA device (tray_cuda has no CPU fallback)");
    if (n_devices < 1 || n_devices > ndev) return fail(TRAY_ERR_ARG, "n_devices %d out of range (1..%d)", n_devices, ndev);
    tray_group* g = new (std::nothrow) tray_group();
    if (!g) return fail(TRAY_ERR_ARG, "out of host memory");
    for (int i = 0; i < n_devices; i++) {
        const int d = devices ? devices[i] : i;
        for (int j = 0; j < i; j++)
            if (g->devices[j] == d) { tray_cuda_group_destroy(g); return fail(TRAY_ERR_ARG, "device %d listed twice", d); }
        g->devices.push_back(d);
    }
    auto body = [&]() -> int {
        for (int i = 0; i < n_devices; i++) {
            tray_scene* sc = nullptr;
            int rc = tray_cuda_scene_create(nodes, n_nodes, tris, n_tris, tri_stride, blas_offsets, n_instances, tlas_start, g->devices[i], &sc);
            if (rc) return rc;
            g->scenes.push_back(sc);
            if (i > 0) {        // device i stores pixels into device 0's frame
                int can = 0;
                CU(cudaDeviceCanAccessPeer(&can, g->devices[i], g->devices[0]));
                if (!can) return fail(TRAY_ERR_CUDA, "device %d has no peer access to device %d", g->devices[i], g->devices[0]);
                CU(cudaSetDevice(g->devices[i]));
                const cudaError_t e = cudaDeviceEnablePeerAccess(g->devices[0], 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else if (e != cudaSuccess) return fail(TRAY_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d) failed: %s", g->devices[i], g->devices[0], cudaGetErrorString(e));
            }
        }
        CU(cudaSetDevice(g->devices[0]));
        for (int i = 0; i < TRAY_MAX_FRAMES_IN_FLIGHT; i++) {
            CU(cudaEventCreateWithFlags(&g->ev_snap[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&g->ev_staged[i], cudaEventDisableTiming));
        }
        g->exchange = env_int("TRAY_CUDA_GROUP_EXCHANGE", 1) ? 1 : 0;
        CU(cudaEventCreate(&g->ev_t0)); CU(cudaEventCreate(&g->ev_t1));
        return TRAY_OK;
    };
    const int rc = body();
    if (rc) { tray_cuda_group_destroy(g); return rc; }
    *out = g;
    return TRAY_OK;
}

int tray_cuda_group_size(const tray_group* g) { return g ? (int)g->scenes.size() : 0; }

int tray_cuda_group_scene(tray_group* g, int i, tray_scene** out) {
    if (!g || !out || i < 0 || i >= (int)g->scenes.size()) return fail(TRAY_ERR_ARG, "bad argument");
    *out = g->scenes[i];
    return TRAY_OK;
}

int tray_cuda_group_set_frames_in_flight(tray_group* g, uint32_t n) {
    if (!g || n < 1 || n > TRAY_MAX_FRAMES_IN_FLIGHT) return fail(TRAY_ERR_ARG, "frames in flight must be 1 .. %d", TRAY_MAX_FRAMES_IN_FLIGHT);
    for (auto* sc : g->scenes) { int rc = tray_cuda_scene_set_frames_in_flight(sc, n); if (rc) return rc; }
    g->in_flight = (int)n; g->cur = 0;
    return TRAY_OK;
}

int tray_cuda_group_set_exchange(tray_group* g, int push) {
    if (!g) return fail(TRAY_ERR_ARG, "NULL group");
    int rc = tray_cuda_group_sync(g); if (rc) return rc;
    g->exchange = push ? 1 : 0;
    return TRAY_OK;
}

int tray_cuda_group_render(tray_group* g, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t flags) {
    if (!g || !view) return fail(TRAY_ERR_ARG, "NULL argument");
    int rc = group_ensure_target(g, w, h);
    if (rc) return rc;
    const int n = (int)g->scenes.size();
    const bool push = g->exchange == 1 && n > 1;
    if (push) { rc = group_ensure_staging(g, w, h); if (rc) return rc; }
    g->cur = (g->cur + 1) % g->in_flight;
    uchar4* const target = g->target[g->cur];
    const uint64_t items = local_items(w, h, 0, (uint32_t)n);
    const bool snap = g->snap_pending[g->cur];             // the frame this target held last is still being copied out
    for (int i = 0; i < n; i++) {
        tray_scene* sc = g->scenes[i];
        const int k = next_slot(sc);                       // the slot this frame will take on device i
        if (!push && i > 0 && snap) {                      // the previous frame in this target must have been copied out first
            CU(cudaSetDevice(sc->device));
            CU(cudaStreamWaitEvent(slot_stream(sc, k), g->ev_snap[g->cur], 0));
        }
        sc->frame_target = push ? nullptr : target;
        rc = tray_cuda_render(sc, view, w, h, frame_count, flags | TRAY_RENDER_RGBA, (uint32_t)i, (uint32_t)n, nullptr, nullptr);
        if (rc) return rc;
        cudaStream_t st = slot_stream(sc, sc->cur);
        if (push) {
            // one DMA copy of the compact shard into devices[0]'s staging (behind the untile of the frame that used it last)
            if (g->staged_pending[g->cur]) CU(cudaStreamWaitEvent(st, g->ev_staged[g->cur], 0));
            const FrameSlot& f = sc->slot[sc->cur];
            if (f.last_frame.n_items)
                CU(cudaMemcpyPeerAsync(g->staging[g->cur] + (uint64_t)i * items, g->devices[0], f.d_rgba, sc->device, (size_t)f.last_frame.n_items * sizeof(uchar4), st));
        }
        if (i > 0) CU(cudaEventRecord(sc->slot[sc->cur].done, st));
    }
    g->snap_pending[g->cur] = false;
    // frame complete on devices[0]: its stream waits for every other device's last launch / copy
    tray_scene* s0 = g->scenes[0];
    cudaStream_t st0 = slot_stream(s0, s0->cur);
    CU(cudaSetDevice(s0->device));
    for (int i = 1; i < n; i++) CU(cudaStreamWaitEvent(st0, g->scenes[i]->slot[g->scenes[i]->cur].done, 0));
    if (push) {
        if (snap) CU(cudaStreamWaitEvent(st0, g->ev_snap[g->cur], 0));
        tray::untile_shards_kernel<<<dim3((w + 255) / 256, h), 256, 0, st0>>>(g->staging[g->cur], w, h, (w + 31) / 32, (uint32_t)n, items, target);
        CU(cudaGetLastError());
        CU(cudaEventRecord(g->ev_staged[g->cur], st0));
        g->staged_pending[g->cur] = true;
        FrameSlot& f0 = s0->slot[s0->cur];               // the readback of devices[0]'s scene reads the assembled frame
        f0.f_target = target; f0.f_has_rgba = false;
    }
    return TRAY_OK;
}

int tray_cuda_group_render_timed(tray_group* g, const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count, uint32_t flags, float* ms_frame) {
    if (!g || !view || !ms_frame) return fail(TRAY_ERR_ARG, "NULL argument");
    int rc = group_ensure_target(g, w, h);
    if (rc) return rc;
    tray_scene* s0 = g->scenes[0];
    CU(cudaSetDevice(s0->device));
    CU(cudaEventRecord(g->ev_t0, slot_stream(s0, next_slot(s0))));
    for (size_t i = 1; i < g->scenes.size(); i++) {      // nobody starts before the clock does
        tray_scene* sc = g->scenes[i];
        CU(cudaSetDevice(sc->device));
        CU(cudaStreamWaitEvent(slot_stream(sc, next_slot(sc)), g->ev_t0, 0));
    }
    rc = tray_cuda_group_render(g, view, w, h, frame_count, flags);
    if (rc) return rc;
    CU(cudaSetDevice(s0->device));
    CU(cudaEventRecord(g->ev_t1, slot_stream(s0, s0->cur)));
    CU(cudaEventSynchronize(g->ev_t1));
    CU(cudaEventElapsedTime(ms_frame, g->ev_t0, g->ev_t1));
    for (auto* sc : g->scenes) { CU(cudaSetDevice(sc->device)); rc = check_overflow(sc->slot[sc->cur].d_flag, slot_stream(sc, sc->cur)); if (rc) return rc; }
    return TRAY_OK;
}

int tray_cuda_group_readback_begin(tray_group* g, uint8_t* rgba_host, uint32_t slot) {
    if (!g || slot >= TRAY_READBACK_SLOTS) return fail(TRAY_ERR_ARG, "bad argument");
    tray_scene* s0 = g->scenes[0];
    int rc = tray_cuda_frame_readback_begin(s0, rgba_host, slot);       // snapshots the frame target on devices[0], D2H on the copy stream
    if (rc) return rc;
    CU(cudaEventRecord(g->ev_snap[g->cur], slot_stream(s0, s0->cur)));
    g->snap_pending[g->cur] = true;
    return TRAY_OK;
}

int tray_cuda_group_readback_wait(tray_group* g, uint32_t slot) {
    if (!g) return fail(TRAY_ERR_ARG, "NULL group");
    return tray_cuda_frame_readback_wait(g->scenes[0], slot);
}

int tray_cuda_group_frame_ptr(tray_group* g, void** d_frame) {
    if (!g || !d_frame) return fail(TRAY_ERR_ARG, "NULL argument");
    *d_frame = g->target[g->cur];
    return TRAY_OK;
}

int tray_cuda_group_sync(tray_group* g) {
    if (!g) return fail(TRAY_ERR_ARG, "NULL group");
    for (auto* sc : g->scenes) { int rc = tray_cuda_sync(sc); if (rc) return rc; }
    return TRAY_OK;
}

int tray_cuda_start_multi(const int* devices, int n_devices,
                          const void* bvh_bytes, uint64_t bvh_len, const void* instance_bytes, uint64_t instance_len,
                          const void* tri_bytes, uint64_t tri_len, uint32_t tri_stride, uint32_t tlas_start, int use_tlas,
                          const tray_view* view, uint32_t width, uint32_t height, float render_time_s, int benchmark,
                          int animate, float* out_min_ms, float* out_mean_ms, uint32_t* out_frames) {
    if (const int rc = check_start_args(view, bvh_len, tri_len, tri_stride, instance_len)) return rc;
    tray_group* g = nullptr;
    int rc = tray_cuda_group_create(bvh_bytes, bvh_len / 80, tri_bytes, tri_len / tri_stride, tri_stride,
                                    use_tlas ? (const uint32_t*)instance_bytes : nullptr, use_tlas ? (uint32_t)(instance_len / 4) : 0u,
                                    tlas_start, devices, n_devices, &g);
    if (rc) return rc;
    const uint32_t flags = TRAY_RENDER_BOUNCE | TRAY_RENDER_RGBA;
    rc = start_loop([&](uint32_t fc) { return tray_cuda_group_render(g, view, width, height, fc, flags); },
                    [&](uint32_t fc, float* ms) { return tray_cuda_group_render_timed(g, view, width, height, fc, flags, ms); },
                    [&] { return tray_cuda_group_sync(g); },
                    render_time_s, benchmark, animate, out_min_ms, out_mean_ms, out_frames);
    tray_cuda_group_destroy(g);
    return rc;
}

}  // extern "C"
