// projectultra_b200/csrc/ldpc_encode.cu — batched LDPC / protocol-v2 frame encoder on the GPU: pu_ldpc_encode_batch (one codeword per
// row, LDPCEncoder::encode) and pu_frame_encode_batch (v2::encodeFrameWithLDPC per row), one CTA per row, both through the encoder the
// batched OFDM transmitter runs (ldpc_encode.cuh).  The sweep driver uses them to keep the coded bits of fresh trials, which its
// transmitters encode inside their own kernels and do not hand out.
#include "frame_v2.cuh"
#include "ldpc_encode.cuh"
#include "pu_internal.h"

void pu_ldpc_encoder_view(const pu_ldpc* h, int* k, int* m, const uint8_t** cn_ninfo, const uint16_t** cn_check, const uint16_t** cn_var);   // ldpc_decode.cu
pu_ctx* pu_ldpc_context(const pu_ldpc* h);                                                                                                  // ldpc_decode.cu
extern "C" int pu_ldpc_rate(const pu_ldpc*);

namespace pu {
namespace {

__global__ void __launch_bounds__(128) ldpc_encode_kernel(LdpcEncDev e, const uint8_t* __restrict__ frames, size_t frame_stride, int frame_bytes,
                                                          int n_cw, int bpc, uint8_t* __restrict__ coded, size_t coded_stride) {
    extern __shared__ __align__(16) uint8_t enc_smem[];
    ldpc_encode_frame_cta(e, frames + static_cast<size_t>(blockIdx.x) * frame_stride, frame_bytes, n_cw, bpc, enc_smem,
                          ldpc_encode_parity_of(enc_smem, n_cw));
    uint8_t* out = coded + static_cast<size_t>(blockIdx.x) * coded_stride;
    for (int i = threadIdx.x; i < n_cw * (PU_LDPC_N / 8); i += blockDim.x) out[i] = enc_smem[i];
}

// B frames of frame_bytes bytes -> n_cw codewords each (bpc frame bytes in CW0) -> coded[b * coded_stride .. + n_cw * 81)
pu_status encode_frames(const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes, int n_cw, int bpc, size_t B,
                        uint8_t* coded, size_t coded_stride, pu_memspace space, void* stream) {
    if (B == 0) return PU_OK;
    PU_REQUIRE(frames || frame_bytes == 0, "pu_frame_encode_batch: NULL frames");
    const size_t row = static_cast<size_t>(n_cw) * (PU_LDPC_N / 8);
    PU_REQUIRE(coded_stride >= row, "pu_frame_encode_batch: coded rows shorter than the codewords of a frame");
    pu_ctx* ctx = pu_ldpc_context(code);
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    LdpcEncDev e{};
    pu_ldpc_encoder_view(code, &e.k, &e.m, &e.cn_ninfo, &e.cn_check, &e.cn_var);
    cudaStream_t st = pick_stream(ctx, stream, space);
    const size_t smem = ldpc_encode_smem(n_cw, e.m);
    auto launch = [&](const uint8_t* d_frames, size_t d_frame_stride, size_t nb, uint8_t* d_coded, size_t d_coded_stride) -> pu_status {
        (void)cudaGetLastError();
        ldpc_encode_kernel<<<static_cast<unsigned>(nb), 128, smem, st>>>(e, d_frames, d_frame_stride, static_cast<int>(frame_bytes), n_cw, bpc,
                                                                        d_coded, d_coded_stride);
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        return PU_OK;
    };
    if (space == PU_MEM_DEVICE) return launch(frames, frame_stride, B, coded, coded_stride);
    // host memory: the bytes of every coded row beyond its codewords are not staged and stay as they were
    HostStage hs(ctx, st, B);
    const uint8_t* d_frames;
    uint8_t* d_coded;
    hs.in(&d_frames, frames, frame_bytes, frame_stride);
    hs.out(&d_coded, coded, row, coded_stride);
    return hs.run([&](size_t nb) { return launch(d_frames, frame_bytes, nb, d_coded, row); });
}

}  // namespace
}  // namespace pu

extern "C" {

pu_status pu_ldpc_encode_batch(const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes, size_t B,
                               uint8_t* coded, size_t coded_stride, pu_memspace space, void* stream) {
    PU_REQUIRE(code, "pu_ldpc_encode_batch: NULL handle");
    const int k = pu_ldpc_info_bits(code);
    PU_REQUIRE(payload_bytes * 8 <= static_cast<size_t>(k) && (B == 0 || payload_bytes <= payload_stride),
               "pu_ldpc_encode_batch: payload longer than one codeword's information bits or than its row");
    PU_REQUIRE(B == 0 || coded, "pu_ldpc_encode_batch: NULL coded");
    // the one-codeword frame: CW0 carries k / 8 bytes, the payload zero padded to them (pu_ofdm_tx_batch's case)
    return pu::encode_frames(code, payload, payload_stride, payload_bytes, 1, k / 8, B, coded, coded_stride, space, stream);
}

pu_status pu_frame_encode_batch(const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes, size_t B, uint8_t* coded,
                                size_t coded_stride, size_t* n_codewords, pu_memspace space, void* stream) {
    PU_REQUIRE(code && n_codewords, "pu_frame_encode_batch: NULL argument");
    const int rate = pu_ldpc_rate(code);
    const uint64_t ncw = pu::frame_codewords(rate, frame_bytes);
    *n_codewords = static_cast<size_t>(ncw);
    if (B == 0 || !coded) return PU_OK;            // codeword count query
    PU_REQUIRE(ncw <= 255, "pu_frame_encode_batch: frame needs more than 255 codewords");
    PU_REQUIRE(frame_bytes <= frame_stride, "pu_frame_encode_batch: frame longer than its row");
    return pu::encode_frames(code, frames, frame_stride, frame_bytes, static_cast<int>(ncw), pu::frame_bytes_per_codeword(rate), B, coded,
                             coded_stride, space, stream);
}

}  // extern "C"
