// projectultra_b200/csrc/interleave.cu — ChannelInterleaver::deinterleave (ldpc_decoder.cpp:612-620) of soft bits on the GPU for any
// receiver (pu_llr_deinterleave_batch): the step RxPipeline takes between getSoftBits and decodeSoft (SURVEY §3.2), 648 soft bits at a
// time, so every codeword of a frame is deinterleaved on its own.
//
// ChannelInterleaver(bps, 648): perm[i] = i * step mod 648 with step coprime to 648; deinterleave out[inv[i]] = in[i], i.e. out[k] =
// in[k * step mod 648].  One integer per call, no table.  The kernel moves each codeword through shared memory: coalesced reads of the
// received order, coalesced writes of the decoder order, in place.  It is bound by HBM: 4 bytes read and 4 written per soft bit.
#include "pu_internal.h"

namespace pu {
namespace {

constexpr int kCwPerCta = 4;                 // 4 x 648 floats = 10.1 KB of shared memory, 10 loads in flight per thread
constexpr int kThreads = 256;
constexpr int kPerThread = (kCwPerCta * PU_LDPC_N + kThreads - 1) / kThreads;

__global__ void __launch_bounds__(kThreads) llr_deinterleave_kernel(float* __restrict__ llr, size_t llr_stride, unsigned n_blocks,
                                                                    size_t n_cw, int step) {
    __shared__ float s[kCwPerCta * PU_LDPC_N];
    __shared__ float* row[kCwPerCta];        // codeword w of the CTA: one 64-bit division each, not one per soft bit
    const size_t q0 = static_cast<size_t>(blockIdx.x) * kCwPerCta;
    if (threadIdx.x < kCwPerCta) {
        const size_t q = q0 + threadIdx.x;
        row[threadIdx.x] = llr + (q / n_blocks) * llr_stride + (q % n_blocks) * PU_LDPC_N;
    }
    __syncthreads();
    auto at = [&](int w) { return row[w]; };
    float v[kPerThread];
#pragma unroll
    for (int r = 0; r < kPerThread; ++r) {
        const int i = threadIdx.x + r * kThreads, w = i / PU_LDPC_N;
        if (i < kCwPerCta * PU_LDPC_N && q0 + w < n_cw) v[r] = at(w)[i - w * PU_LDPC_N];
    }
#pragma unroll
    for (int r = 0; r < kPerThread; ++r) {
        const int i = threadIdx.x + r * kThreads;
        if (i < kCwPerCta * PU_LDPC_N && q0 + i / PU_LDPC_N < n_cw) s[i] = v[r];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kPerThread; ++r) {
        const int i = threadIdx.x + r * kThreads, w = i / PU_LDPC_N, k = i - w * PU_LDPC_N;
        if (i < kCwPerCta * PU_LDPC_N && q0 + w < n_cw) at(w)[k] = s[w * PU_LDPC_N + k * step % PU_LDPC_N];
    }
}

}  // namespace

pu_status llr_deinterleave_enqueue(pu_ctx* ctx, float* llr, size_t B, size_t llr_stride, size_t n_blocks, size_t bits_per_symbol, cudaStream_t st) {
    const size_t n_cw = B * n_blocks;
    if (n_cw == 0) return PU_OK;
    size_t step = 0;
    pu_status s = pu_channel_interleaver_perm(bits_per_symbol, PU_LDPC_N, nullptr, nullptr, &step);
    if (s != PU_OK) return s;
    (void)cudaGetLastError();
    llr_deinterleave_kernel<<<static_cast<unsigned>((n_cw + kCwPerCta - 1) / kCwPerCta), kThreads, 0, st>>>(
        llr, llr_stride, static_cast<unsigned>(n_blocks), n_cw, static_cast<int>(step));
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

}  // namespace pu

extern "C" {

pu_status pu_llr_deinterleave_batch(pu_ctx* ctx, float* llr, size_t B, size_t llr_stride, size_t n_blocks, size_t bits_per_symbol,
                                    pu_memspace space, void* stream) {
    PU_REQUIRE(ctx, "pu_llr_deinterleave_batch: NULL context");
    PU_REQUIRE(space == PU_MEM_HOST || space == PU_MEM_DEVICE, "pu_llr_deinterleave_batch: bad memory space");
    PU_REQUIRE(bits_per_symbol > 0, "pu_llr_deinterleave_batch: bits_per_symbol is zero");
    PU_REQUIRE(n_blocks * PU_LDPC_N <= llr_stride, "pu_llr_deinterleave_batch: n_blocks * 648 exceeds llr_stride");
    PU_REQUIRE(llr || B == 0 || n_blocks == 0, "pu_llr_deinterleave_batch: NULL llr");
    PU_REQUIRE(B * n_blocks < (size_t(1) << 33), "pu_llr_deinterleave_batch: batch too large");
    if (B == 0 || n_blocks == 0) return PU_OK;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_DEVICE) return pu::llr_deinterleave_enqueue(ctx, llr, B, llr_stride, n_blocks, bits_per_symbol, st);
    // host memory: the first n_blocks * 648 soft bits of every row go down and come back; the rest of the row is not staged
    const size_t row = n_blocks * PU_LDPC_N;
    pu::HostStage hs(ctx, st, B);
    float* d;
    hs.inout(&d, llr, row, llr_stride);
    return hs.run([&](size_t nb) { return pu::llr_deinterleave_enqueue(ctx, d, nb, row, n_blocks, bits_per_symbol, st); });
}

}  // extern "C"
