// device_probe.cu — batch entry points onto the traversal's device primitives, one thread per case.  TEST INFRASTRUCTURE ONLY:
// built by `make -C tray_racing_b200/csrc probe` into libtray_probe.so, loaded by tests/test_device_primitives.py, never linked by
// the product.  Every kernel calls the product's own tray:: functions from traverse.cuh and build_gpu.h (no copies), with k4b, zero
// and one passed at run time as TraceParams passes them.  The host wrappers take host arrays, copy them to the device, launch, copy
// the results back and return a cudaError_t (0 = success).
#include <cstring>

#include "build_gpu.h"
#include "traverse.cuh"

namespace {

// a ray as the oracle's orc_ray / tray_ray: {o[3], tmin, d[3], tmax}
struct ProbeRay { float ox, oy, oz, tmin, dx, dy, dz, tmax; };

__device__ void prep(tray::RayConst& r, const ProbeRay& q, uint32_t variant) {
    tray::prepare_ray(r, q.ox, q.oy, q.oz, q.dx, q.dy, q.dz, q.tmin, variant);
}

// {dx, dy, dz, ix, iy, iz, tdx, tdy, tdz, box_tmin, oct_inv4, wide} per ray
__global__ void k_prepare_ray(const ProbeRay* rays, uint32_t n, uint32_t variant, uint32_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    tray::RayConst r; prep(r, rays[i], variant);
    const float f[10] = {r.dx, r.dy, r.dz, r.ix, r.iy, r.iz, r.tdx, r.tdy, r.tdz, r.box_tmin};
    uint32_t* o = out + 12u * i;
    for (int k = 0; k < 10; k++) o[k] = __float_as_uint(f[k]);
    o[10] = r.oct_inv4; o[11] = r.wide ? 1u : 0u;
}

// which: 0 node_test with its default arguments; 1 node_test as MODE 1 calls it (box_tmin = r.box_tmin, divide per the variant);
// 2 node_test_fast; 3 what a MODE 0 trace_kernel runs (node_test for wide rays or nodes past the exponent guard, else the fast form)
__global__ void k_node_test(const uint4* nodes, const ProbeRay* rays, uint32_t n, uint32_t which, uint32_t variant,
                            uint32_t k4b, float zero, uint32_t one, uint32_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    tray::RayConst r; prep(r, rays[i], which == 1u ? variant : 0u);
    const uint4* np = nodes + 5u * i;
    const uint4 n0 = np[0], n1 = np[1], n2 = np[2], n3 = np[3], n4 = np[4];
    const float tmax = rays[i].tmax;
    uint32_t m;
    if (which == 0u) m = tray::node_test(r, tmax, n0, n1, n2, n3, n4, k4b);
    else if (which == 1u) m = tray::node_test(r, tmax, n0, n1, n2, n3, n4, k4b, r.box_tmin, (variant & TRAY_VARIANT_BOX_DIVIDE) != 0u);
    else if (which == 2u) m = tray::node_test_fast(r, tmax, n0, n1, n2, n3, n4, k4b, zero, one);
    else m = (r.wide || tray::node_needs_exact(n0.w)) ? tray::node_test(r, tmax, n0, n1, n2, n3, n4, k4b)
                                                       : tray::node_test_fast(r, tmax, n0, n1, n2, n3, n4, k4b, zero, one);
    out[i] = m;
}

// record i against ray i, tmax = ray.tmax
template <int S, bool VD>
__global__ void k_tri_test(const uint4* tris, const ProbeRay* rays, uint32_t n, uint32_t variant, float* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    tray::RayConst r; prep(r, rays[i], variant);
    out[i] = tray::tri_test<S, VD>(r, rays[i].tmax, tris, i);
}

__global__ void k_primary_dir(tray::FrameParams F, const uint32_t* px, const uint32_t* py, uint32_t n, float* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    tray::primary_dir(F, px[i], py[i], out[3 * i], out[3 * i + 1], out[3 * i + 2]);
}

// case i: record prim[i] of `tris`, primary direction pd[3i..], hit distance t[i], pixel (px[i], py[i]), frame F.frame_count + fc[i];
// with `inst` (64-byte InstanceRecords, one per case), the instanced form with record i
template <int S>
__global__ void k_bounce_ray(tray::FrameParams F, const uint4* tris, const uint32_t* px, const uint32_t* py, const float* pd,
                             const float* t, const uint32_t* prim, const uint32_t* fc, const uint4* inst, uint32_t n, float* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F.frame_count = fc[i];
    float* o = out + 6u * i;
    if (inst)
        tray::bounce_ray<S, true>(F, tris, px[i], py[i], pd[3 * i], pd[3 * i + 1], pd[3 * i + 2], t[i], prim[i], o[0], o[1], o[2], o[3], o[4],
                                  o[5], inst + tray::INST_RECORD_U4 * i);
    else
        tray::bounce_ray<S>(F, tris, px[i], py[i], pd[3 * i], pd[3 * i + 1], pd[3 * i + 2], t[i], prim[i], o[0], o[1], o[2], o[3], o[4], o[5]);
}

__global__ void k_uhash(const uint32_t* a, const uint32_t* b, uint32_t n, uint32_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tray::uhash(a[i], b[i]);
}
__global__ void k_hash_noise(const uint32_t* x, const uint32_t* y, const uint32_t* f, uint32_t n, float* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tray::hash_noise(x[i], y[i], f[i]);
}
__global__ void k_sincos_tau(const float* u, uint32_t n, float* s, float* c) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tray::sincos_tau(u[i], s[i], c[i]);
}
__global__ void k_shade(uint32_t mode, const float* t, uint32_t n, uint8_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tray::shade(mode, t[i]).x;
}
// the child-order table as trace_kernel builds it (one block), rows LUT_ROW bytes apart
__global__ void k_child_order(uint8_t* out) {
    __shared__ uint8_t lut[tray::LUT_BYTES];
    for (unsigned k = threadIdx.x; k < tray::LUT_BYTES; k += blockDim.x) lut[k] = 0xeeu;
    __syncthreads();
    tray::child_order_fill(lut, threadIdx.x, blockDim.x);
    __syncthreads();
    for (unsigned k = threadIdx.x; k < tray::LUT_BYTES; k += blockDim.x) out[k] = lut[k];
}

// device copies of the host arrays of one call, freed when it returns
struct Dev {
    void* p[12] = {};
    int k = 0;
    cudaError_t err = cudaSuccess;
    template <typename T> T* in(const void* src, size_t bytes) {
        void* d = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&d, bytes ? bytes : 16);
        if (err == cudaSuccess && bytes) err = cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice);
        p[k++] = d;
        return static_cast<T*>(d);
    }
    template <typename T> T* alloc(size_t bytes) {
        void* d = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&d, bytes ? bytes : 16);
        p[k++] = d;
        return static_cast<T*>(d);
    }
    void back(void* dst, const void* src, size_t bytes) {
        if (err == cudaSuccess) err = cudaGetLastError();
        if (err == cudaSuccess) err = cudaDeviceSynchronize();
        if (err == cudaSuccess && bytes) err = cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
    }
    ~Dev() { for (int i = 0; i < k; i++) if (p[i]) cudaFree(p[i]); }
};
inline unsigned blocks(uint32_t n) { return (n + 127u) / 128u; }
constexpr uint32_t K4B = 0x4B000000u;

tray::FrameParams frame(const tray_view* view, uint32_t w, uint32_t h, uint32_t frame_count) {
    tray::FrameParams F;
    std::memset(&F, 0, sizeof(F));
    F.view = *view; F.width = w; F.height = h; F.frame_count = frame_count;
    return F;
}

}  // namespace

extern "C" {

int probe_prepare_ray(const void* rays, uint32_t n, uint32_t variant, uint32_t* out) {
    Dev d;
    const ProbeRay* r = d.in<ProbeRay>(rays, n * sizeof(ProbeRay));
    uint32_t* o = d.alloc<uint32_t>(n * 12u * 4u);
    if (d.err == cudaSuccess && n) k_prepare_ray<<<blocks(n), 128>>>(r, n, variant, o);
    d.back(out, o, n * 12u * 4u);
    return (int)d.err;
}

int probe_node_test(const void* nodes80, const void* rays, uint32_t n, uint32_t which, uint32_t variant, uint32_t* out) {
    Dev d;
    const uint4* nd = d.in<uint4>(nodes80, (size_t)n * 80u);
    const ProbeRay* r = d.in<ProbeRay>(rays, n * sizeof(ProbeRay));
    uint32_t* o = d.alloc<uint32_t>(n * 4u);
    if (d.err == cudaSuccess && n) k_node_test<<<blocks(n), 128>>>(nd, r, n, which, variant, K4B, 0.0f, 1u, o);
    d.back(out, o, n * 4u);
    return (int)d.err;
}

// records: n x stride bytes (24, 48 or 64); variant_dir: tri_test<S, true> (the direction MODE 1 hands the triangle test)
int probe_tri_test(const void* records, uint32_t stride, const void* rays, uint32_t n, uint32_t variant, uint32_t variant_dir, float* out) {
    Dev d;
    const uint4* t = d.in<uint4>(records, (size_t)n * stride);
    const ProbeRay* r = d.in<ProbeRay>(rays, n * sizeof(ProbeRay));
    float* o = d.alloc<float>(n * 4u);
    if (d.err == cudaSuccess && n) {
        const unsigned g = blocks(n);
        if (stride == 24) variant_dir ? k_tri_test<24, true><<<g, 128>>>(t, r, n, variant, o) : k_tri_test<24, false><<<g, 128>>>(t, r, n, variant, o);
        else if (stride == 48) variant_dir ? k_tri_test<48, true><<<g, 128>>>(t, r, n, variant, o) : k_tri_test<48, false><<<g, 128>>>(t, r, n, variant, o);
        else if (stride == 64) variant_dir ? k_tri_test<64, true><<<g, 128>>>(t, r, n, variant, o) : k_tri_test<64, false><<<g, 128>>>(t, r, n, variant, o);
        else return (int)cudaErrorInvalidValue;
    }
    d.back(out, o, n * 4u);
    return (int)d.err;
}

int probe_primary_dir(const tray_view* view, uint32_t w, uint32_t h, const uint32_t* px, const uint32_t* py, uint32_t n, float* out) {
    Dev d;
    const uint32_t* x = d.in<uint32_t>(px, n * 4u);
    const uint32_t* y = d.in<uint32_t>(py, n * 4u);
    float* o = d.alloc<float>(n * 12u);
    if (d.err == cudaSuccess && n) k_primary_dir<<<blocks(n), 128>>>(frame(view, w, h, 0), x, y, n, o);
    d.back(out, o, n * 12u);
    return (int)d.err;
}

// out: n x {ox, oy, oz, dx, dy, dz}; inst_records: NULL, or n x 64 B (case i's instance)
static int bounce_ray_cases(uint32_t stride, const void* records, uint32_t n_records, const tray_view* view, const uint32_t* px,
                            const uint32_t* py, const float* pd, const float* t, const uint32_t* prim, const uint32_t* frame_count,
                            const void* inst_records, uint32_t n, float* out) {
    Dev d;
    const uint4* tr = d.in<uint4>(records, (size_t)n_records * stride);
    const uint32_t* x = d.in<uint32_t>(px, n * 4u);
    const uint32_t* y = d.in<uint32_t>(py, n * 4u);
    const float* dd = d.in<float>(pd, n * 12u);
    const float* tt = d.in<float>(t, n * 4u);
    const uint32_t* pp = d.in<uint32_t>(prim, n * 4u);
    const uint32_t* fc = d.in<uint32_t>(frame_count, n * 4u);
    const uint4* ir = inst_records ? d.in<uint4>(inst_records, (size_t)n * 64u) : nullptr;
    float* o = d.alloc<float>(n * 24u);
    const tray::FrameParams F = frame(view, 1, 1, 0);
    if (d.err == cudaSuccess && n) {
        const unsigned g = blocks(n);
        if (stride == 24) k_bounce_ray<24><<<g, 128>>>(F, tr, x, y, dd, tt, pp, fc, ir, n, o);
        else if (stride == 48) k_bounce_ray<48><<<g, 128>>>(F, tr, x, y, dd, tt, pp, fc, ir, n, o);
        else if (stride == 64) k_bounce_ray<64><<<g, 128>>>(F, tr, x, y, dd, tt, pp, fc, ir, n, o);
        else return (int)cudaErrorInvalidValue;
    }
    d.back(out, o, n * 24u);
    return (int)d.err;
}

int probe_bounce_ray(uint32_t stride, const void* records, uint32_t n_records, const tray_view* view, const uint32_t* px,
                     const uint32_t* py, const float* pd, const float* t, const uint32_t* prim, const uint32_t* frame_count,
                     uint32_t n, float* out) {
    return bounce_ray_cases(stride, records, n_records, view, px, py, pd, t, prim, frame_count, nullptr, n, out);
}

// the instanced form (bounce_ray<S, true>): inst_records = n x 64-byte InstanceRecords, case i takes record i
int probe_bounce_ray_inst(uint32_t stride, const void* records, uint32_t n_records, const tray_view* view, const uint32_t* px,
                          const uint32_t* py, const float* pd, const float* t, const uint32_t* prim, const uint32_t* frame_count,
                          const void* inst_records, uint32_t n, float* out) {
    return bounce_ray_cases(stride, records, n_records, view, px, py, pd, t, prim, frame_count, inst_records, n, out);
}

int probe_uhash(const uint32_t* a, const uint32_t* b, uint32_t n, uint32_t* out) {
    Dev d;
    const uint32_t* x = d.in<uint32_t>(a, n * 4u);
    const uint32_t* y = d.in<uint32_t>(b, n * 4u);
    uint32_t* o = d.alloc<uint32_t>(n * 4u);
    if (d.err == cudaSuccess && n) k_uhash<<<blocks(n), 128>>>(x, y, n, o);
    d.back(out, o, n * 4u);
    return (int)d.err;
}

int probe_hash_noise(const uint32_t* x, const uint32_t* y, const uint32_t* frame_count, uint32_t n, float* out) {
    Dev d;
    const uint32_t* a = d.in<uint32_t>(x, n * 4u);
    const uint32_t* b = d.in<uint32_t>(y, n * 4u);
    const uint32_t* f = d.in<uint32_t>(frame_count, n * 4u);
    float* o = d.alloc<float>(n * 4u);
    if (d.err == cudaSuccess && n) k_hash_noise<<<blocks(n), 128>>>(a, b, f, n, o);
    d.back(out, o, n * 4u);
    return (int)d.err;
}

int probe_sincos_tau(const float* u, uint32_t n, float* s, float* c) {
    Dev d;
    const float* x = d.in<float>(u, n * 4u);
    float* so = d.alloc<float>(n * 4u);
    float* co = d.alloc<float>(n * 4u);
    if (d.err == cudaSuccess && n) k_sincos_tau<<<blocks(n), 128>>>(x, n, so, co);
    d.back(s, so, n * 4u);
    d.back(c, co, n * 4u);
    return (int)d.err;
}

int probe_shade(uint32_t mode, const float* t, uint32_t n, uint8_t* out) {
    Dev d;
    const float* x = d.in<float>(t, n * 4u);
    uint8_t* o = d.alloc<uint8_t>(n);
    if (d.err == cudaSuccess && n) k_shade<<<blocks(n), 128>>>(mode, x, n, o);
    d.back(out, o, n);
    return (int)d.err;
}

// out: LUT_BYTES (8 rows of LUT_ROW bytes)
int probe_child_order(uint8_t* out) {
    Dev d;
    uint8_t* o = d.alloc<uint8_t>(tray::LUT_BYTES);
    if (d.err == cudaSuccess) k_child_order<<<1, tray::BLOCK_THREADS>>>(o);
    d.back(out, o, tray::LUT_BYTES);
    return (int)d.err;
}

uint32_t probe_lut_row(void) { return tray::LUT_ROW; }

}  // extern "C"
