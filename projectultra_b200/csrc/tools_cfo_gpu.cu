// projectultra_b200/csrc/tools_cfo_gpu.cu — the tools' FFT-Hilbert CFO injector (tools_cfo.cpp) for batches of rows on the GPU
// (pu_tools_cfo_*): what the sweep driver runs on every fresh-payload frame of a mode with a tuning error.
//
// Bit-exactness comes from the butterfly DAG, not from a schedule: the host is a radix-2 DIT over the bit-reversed, zero-padded row of
// P = 2^p points; each butterfly of stage s (len = 2^s) is t = w * b in GCC's complex<float> form (cmul of ofdm_dev.cuh under
// -fmad=false), then a - t and a + t, with w = tw[k * P / len].  Every butterfly sees the same inputs and twiddle in any order, so any
// schedule of them reproduces the host's bits; the payload-independent tables (twiddles, rotator of the float phase recurrence) come
// from the host function's own builders; the twiddles of stage s are stored contiguously (tw[k * P / 2^s] at 2^(s-1) - 1 + k), so that
// every stage reads them coalesced.  No butterfly on a zero input is pruned: signed zeros are part of the result.
//
// Schedule, per direction, with tiles of 2^13 complex values (64 KB of shared memory):
//   pass A  one CTA per 2^13 consecutive positions of the bit-reversed array: stages 1..13;
//   pass B  one CTA per 2^(p-13) x (2^13 / 2^(p-13)) tile of the columns 2^13 apart: stages 14..p.
// Forward pass A gathers the row bit-reversed; forward pass B applies the x2 / zero step and writes its output bit-reversed, so that
// the inverse pass A reads consecutive positions; inverse pass B applies 1/P, the rotation and the real part and writes the row.
// p <= 13 runs everything in one CTA per row (forward, x2 / zero, bit reversal in shared memory, inverse, rotation).
#include <algorithm>
#include <cmath>
#include <complex>
#include <vector>

#include "ofdm_dev.cuh"
#include "pu_internal.h"

namespace pu {
namespace {

constexpr int kLogTile = 13, kTile = 1 << kLogTile, kThreads = 512;
constexpr int kMaxLog2 = 20;
constexpr size_t kScratchBytes = size_t(64) << 20;      // both ping-pong buffers of one chunk of rows

__device__ __forceinline__ uint32_t bitrev(uint32_t x, int bits) { return __brev(x) >> (32 - bits); }

__device__ __forceinline__ float2 twiddle(const float2* __restrict__ tw, uint32_t idx, bool inverse) {
    const float2 w = __ldg(tw + idx);
    return inverse ? cconj(w) : w;
}

// stages s_lo..s_hi on a shared-memory tile of consecutive positions (s_hi <= log2 of the tile): k = position mod 2^(s-1)
__device__ __forceinline__ void stages_consecutive(float2* a, int log2n, int s_lo, int s_hi, int p, const float2* __restrict__ tw, bool inverse) {
    const uint32_t half_n = 1u << (log2n - 1);
    for (int s = s_lo; s <= s_hi; ++s) {
        const uint32_t hm = (1u << (s - 1)) - 1;
        for (uint32_t t = threadIdx.x; t < half_n; t += blockDim.x) {
            const uint32_t k = t & hm, i0 = ((t >> (s - 1)) << s) | k, i1 = i0 + hm + 1;
            const float2 w = twiddle(tw, hm + k, inverse);
            const float2 u = a[i0], v = cmul(w, a[i1]);
            a[i1] = csub(u, v);
            a[i0] = cadd(u, v);
        }
        __syncthreads();
    }
}

__device__ __forceinline__ float2 fwd_epilogue(float2 v, uint32_t g, uint32_t P) {      // x2 on (0, P/2), zero on (P/2, P)
    if (g > P / 2) return make_float2(0.0f, 0.0f);
    if (g > 0 && g < P / 2) return cscale(2.0f, v);
    return v;
}

__device__ __forceinline__ float inv_epilogue(float2 v, float scale, float2 r) {          // 1/P, rotation, real part
    v = cscale(scale, v);
    return __fsub_rn(__fmul_rn(v.x, r.x), __fmul_rn(v.y, r.y));
}

// p <= 13: the whole transform pair in one CTA per row
__global__ void __launch_bounds__(kThreads) cfo_row_kernel(float* __restrict__ x, size_t stride, uint32_t n, int p, const float2* __restrict__ tw,
                                                          const float2* __restrict__ rot, float scale) {
    extern __shared__ float2 a[];
    const uint32_t P = 1u << p;
    float* row = x + blockIdx.x * stride;
    for (uint32_t j = threadIdx.x; j < P; j += blockDim.x) {
        const uint32_t src = bitrev(j, p);
        a[j] = make_float2(src < n ? row[src] : 0.0f, 0.0f);
    }
    __syncthreads();
    stages_consecutive(a, p, 1, p, p, tw, false);
    for (uint32_t g = threadIdx.x; g < P; g += blockDim.x) a[g] = fwd_epilogue(a[g], g, P);
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < P; j += blockDim.x) {
        const uint32_t q = bitrev(j, p);
        if (j < q) { const float2 t = a[j]; a[j] = a[q]; a[q] = t; }
    }
    __syncthreads();
    stages_consecutive(a, p, 1, p, p, tw, true);
    for (uint32_t g = threadIdx.x; g < n; g += blockDim.x) row[g] = inv_epilogue(a[g], scale, rot[g]);
}

// pass A, p > 13: forward gathers the row bit-reversed and zero-padded (x -> s1), inverse reads consecutive positions (s2 -> s1)
template <bool kInverse>
__global__ void __launch_bounds__(kThreads) cfo_pass_a_kernel(const float* __restrict__ x, size_t stride, uint32_t n, const float2* __restrict__ s2,
                                                             float2* __restrict__ s1, int p, const float2* __restrict__ tw) {
    extern __shared__ float2 a[];
    const uint32_t base = blockIdx.x * kTile;
    const size_t r = blockIdx.y, P = size_t(1) << p;
    for (uint32_t e = threadIdx.x; e < kTile; e += blockDim.x) {
        if (kInverse) {
            a[e] = s2[r * P + base + e];
        } else {
            const uint32_t src = bitrev(base + e, p);
            a[e] = make_float2(src < n ? x[r * stride + src] : 0.0f, 0.0f);
        }
    }
    __syncthreads();
    stages_consecutive(a, kLogTile, 1, kLogTile, p, tw, kInverse);
    for (uint32_t e = threadIdx.x; e < kTile; e += blockDim.x) s1[r * P + base + e] = a[e];
}

// pass B, p > 13: stages 14..p on a tile of R = 2^(p-13) rows x CB = 2^13 / R columns of the [R][2^13] view of s1; tile element
// (rr, cc) is transform position g = c0 + cc + rr * 2^13.  Forward: x2 / zero, written to s2 at bitrev(g).  Inverse: 1/P, rotation,
// real part, written to the row.
template <bool kInverse>
__global__ void __launch_bounds__(kThreads) cfo_pass_b_kernel(const float2* __restrict__ s1, float2* __restrict__ s2, float* __restrict__ x, size_t stride,
                                                             uint32_t n, int p, const float2* __restrict__ tw, const float2* __restrict__ rot, float scale) {
    extern __shared__ float2 a[];
    const int lr = p - kLogTile, lc = kLogTile - lr;      // log2 R, log2 CB
    const uint32_t CB = 1u << lc, c0 = blockIdx.x << lc, P = 1u << p;
    const size_t r = blockIdx.y;
    const float2* src = s1 + r * P;
    for (uint32_t e = threadIdx.x; e < kTile; e += blockDim.x) a[e] = src[((e >> lc) << kLogTile) + c0 + (e & (CB - 1))];
    __syncthreads();
    for (int s = kLogTile + 1; s <= p; ++s) {
        const int sr = s - 1 - kLogTile;                  // the pair's rows differ in bit sr
        const uint32_t hr = 1u << sr;
        for (uint32_t t = threadIdx.x; t < kTile / 2; t += blockDim.x) {
            const uint32_t cc = t & (CB - 1), rp = t >> lc;
            const uint32_t r0 = ((rp >> sr) << (sr + 1)) | (rp & (hr - 1)), r1 = r0 + hr;
            const uint32_t k = c0 + cc + ((r0 & (hr - 1)) << kLogTile);      // position mod 2^(s-1)
            const float2 w = twiddle(tw, (1u << (s - 1)) - 1 + k, kInverse);
            const uint32_t i0 = (r0 << lc) | cc, i1 = (r1 << lc) | cc;
            const float2 u = a[i0], v = cmul(w, a[i1]);
            a[i1] = csub(u, v);
            a[i0] = cadd(u, v);
        }
        __syncthreads();
    }
    if (kInverse) {
        float* row = x + r * stride;
        for (uint32_t e = threadIdx.x; e < kTile; e += blockDim.x) {
            const uint32_t g = c0 + (e & (CB - 1)) + ((e >> lc) << kLogTile);
            if (g < n) row[g] = inv_epilogue(a[e], scale, rot[g]);
        }
    } else {
        // bitrev(g) = bitrev13(c) * R + bitrev_lr(rr): each column lands on R consecutive positions
        float2* dst = s2 + r * P;
        for (uint32_t e = threadIdx.x; e < kTile; e += blockDim.x) {
            const uint32_t cc = e >> lr, rq = e & ((1u << lr) - 1), rr = bitrev(rq, lr), c = c0 + cc;
            dst[(bitrev(c, kLogTile) << lr) | rq] = fwd_epilogue(a[(rr << lc) | cc], c + (rr << kLogTile), P);
        }
    }
}

}  // namespace
}  // namespace pu

struct pu_tools_cfo {
    pu_ctx* ctx = nullptr;
    uint32_t n = 0;
    int p = 0;                    // log2 of the transform size; 0: the call leaves rows untouched
    float scale = 0.0f;           // 1.0f / P, as the host evaluates it
    size_t chunk = 0;             // rows per pass of the two-pass schedule (scratch bound)
    pu::Buffer tw, rot, s1, s2;
    ~pu_tools_cfo() { tw.release(); rot.release(); s1.release(); s2.release(); }
};

namespace pu {
namespace {

// rows x[b * stride ...] for b < B, device memory, on st
pu_status tools_cfo_rows(pu_tools_cfo* h, float* x, size_t B, size_t stride, cudaStream_t st) {
    const int p = h->p;
    const float2* tw = static_cast<const float2*>(h->tw.ptr);
    const float2* rot = static_cast<const float2*>(h->rot.ptr);
    (void)cudaGetLastError();
    if (p <= kLogTile) {
        const unsigned threads = std::min(kThreads, 1 << (p - 1));
        for (size_t b0 = 0; b0 < B; b0 += 65535u * 1024u) {
            const size_t nb = std::min<size_t>(B - b0, 65535u * 1024u);
            cfo_row_kernel<<<static_cast<unsigned>(nb), threads, sizeof(float2) << p, st>>>(x + b0 * stride, stride, h->n, p, tw, rot, h->scale);
            h->ctx->launches.fetch_add(1);
            PU_CUDA_TRY(cudaGetLastError());
        }
        return PU_OK;
    }
    float2* s1 = static_cast<float2*>(h->s1.ptr);
    float2* s2 = static_cast<float2*>(h->s2.ptr);
    const unsigned tiles = 1u << (p - kLogTile);
    const size_t smem = sizeof(float2) * kTile;
    for (size_t b0 = 0; b0 < B; b0 += h->chunk) {
        const dim3 grid(tiles, static_cast<unsigned>(std::min(h->chunk, B - b0)));
        float* xr = x + b0 * stride;
        cfo_pass_a_kernel<false><<<grid, kThreads, smem, st>>>(xr, stride, h->n, nullptr, s1, p, tw);
        cfo_pass_b_kernel<false><<<grid, kThreads, smem, st>>>(s1, s2, nullptr, 0, h->n, p, tw, nullptr, 0.0f);
        cfo_pass_a_kernel<true><<<grid, kThreads, smem, st>>>(nullptr, 0, h->n, s2, s1, p, tw);
        cfo_pass_b_kernel<true><<<grid, kThreads, smem, st>>>(s1, nullptr, xr, stride, h->n, p, tw, rot, h->scale);
        h->ctx->launches.fetch_add(4);
        PU_CUDA_TRY(cudaGetLastError());
    }
    return PU_OK;
}

}  // namespace
}  // namespace pu

extern "C" {

pu_status pu_tools_cfo_create(pu_ctx* ctx, size_t n, float cfo_hz, float sample_rate, pu_tools_cfo** out) {
    PU_REQUIRE(ctx && out, "pu_tools_cfo_create: NULL argument");
    *out = nullptr;
    PU_REQUIRE(sample_rate > 0 && std::isfinite(cfo_hz), "pu_tools_cfo_create: bad sample rate or offset");
    if (n > (size_t(1) << pu::kMaxLog2)) {
        pu::set_error("pu_tools_cfo_create: %zu samples; the device injector takes up to 2^20 (pu_tools_apply_cfo has no limit)", n);
        return PU_ERR_UNSUPPORTED;
    }
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu_tools_cfo* h = new pu_tools_cfo();
    h->ctx = ctx;
    h->n = static_cast<uint32_t>(n);
    if (n < 128 || std::abs(cfo_hz) < 0.001f) { *out = h; return PU_OK; }        // the host function's no-op cases (tools_cfo.cpp)
    int p = 0;
    while ((size_t(1) << p) < n) ++p;
    const size_t P = size_t(1) << p;
    h->p = p;
    h->scale = 1.0f / P;
    std::vector<std::complex<float>> tw0(P / 2), tw(P - 1), rot(n);
    pu::tools_cfo_twiddles(P, tw0.data());
    for (int s = 1; s <= p; ++s)                        // stage s: tw0[k << (p - s)] for k < 2^(s-1), at 2^(s-1) - 1 + k
        for (size_t k = 0; k < (size_t(1) << (s - 1)); ++k) tw[(size_t(1) << (s - 1)) - 1 + k] = tw0[k << (p - s)];
    pu::tools_cfo_rotator(n, cfo_hz, sample_rate, rot.data());
    pu_status s = PU_OK;
    auto fail = [&](pu_status e) { pu_tools_cfo_destroy(h); return e; };
    if ((s = h->tw.reserve(tw.size() * sizeof(float2))) != PU_OK || (s = h->rot.reserve(rot.size() * sizeof(float2))) != PU_OK) return fail(s);
    if (p > pu::kLogTile) {
        h->chunk = std::max<size_t>(1, pu::kScratchBytes / (2 * P * sizeof(float2)));
        if ((s = h->s1.reserve(h->chunk * P * sizeof(float2))) != PU_OK || (s = h->s2.reserve(h->chunk * P * sizeof(float2))) != PU_OK) return fail(s);
    }
    cudaError_t e = cudaMemcpy(h->tw.ptr, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->rot.ptr, rot.data(), rot.size() * sizeof(float2), cudaMemcpyHostToDevice);
    const int smem = static_cast<int>(sizeof(float2) * pu::kTile);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pu::cfo_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pu::cfo_pass_a_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pu::cfo_pass_a_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pu::cfo_pass_b_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pu::cfo_pass_b_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) {
        pu::set_error("pu_tools_cfo_create: %s", cudaGetErrorString(e));
        return fail(PU_ERR_CUDA);
    }
    *out = h;
    return PU_OK;
}

void pu_tools_cfo_destroy(pu_tools_cfo* h) {
    if (!h) return;
    cudaSetDevice(h->ctx->device);
    delete h;
}

pu_status pu_tools_cfo_apply_batch(pu_tools_cfo* h, float* samples, size_t B, size_t stride, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_tools_cfo_apply_batch: NULL handle");
    PU_REQUIRE(space == PU_MEM_HOST || space == PU_MEM_DEVICE, "pu_tools_cfo_apply_batch: bad memory space");
    PU_REQUIRE(stride >= h->n, "pu_tools_cfo_apply_batch: stride shorter than a row");
    PU_REQUIRE(samples || B == 0, "pu_tools_cfo_apply_batch: NULL samples");
    if (B == 0 || h->p == 0) return PU_OK;
    PU_CUDA_TRY(cudaSetDevice(h->ctx->device));
    cudaStream_t st = pu::pick_stream(h->ctx, stream, space);
    if (space == PU_MEM_DEVICE) return pu::tools_cfo_rows(h, samples, B, stride, st);
    // host rows: only the n samples of each row travel
    pu::HostStage hs(h->ctx, st, B);
    float* d;
    hs.inout(&d, samples, h->n, stride);
    return hs.run([&](size_t nb) { return pu::tools_cfo_rows(h, d, nb, h->n, st); });
}

}  // extern "C"
