// projectultra_b200/csrc/ofdm_tx_gpu.cu — batched transmitter on the GPU (SURVEY §8f next-3/next-4): codeword chunking + LDPC
// encode + OFDM modulate, one frame per CTA, so that every Monte-Carlo frame can carry a fresh random payload like the reference's
// tools do instead of drawing from a host-built pool of waveforms.  One kernel serves both entry points: pu_ofdm_tx_batch is the
// one-codeword frame (a payload of at most k / 8 bytes is CW0 of its own zero-padded frame), pu_frame_tx_batch any frame of 1..255
// codewords modulated back to back.
//
// Reference behaviour (bit-identical waveforms; the host twin is csrc/ofdm_tx.cpp + ldpc_code.cpp: ldpc_encode + frame_v2.cu):
//   v2::encodeFrameWithLDPC (chunking)                    src/protocol/frame_v2.cpp:1079-1127
//   LDPCEncoder::encode                                   src/fec/ldpc_encoder.cpp:193-257  (parity_i = XOR of H_data row i)
//   OFDMModulator::modulate / mapBits                     src/ofdm/modulator.cpp:348-477, :76-106
//   differential encoding, pilots, IFFT + CP, passband    :393-470 (state carried per carrier over the symbols of a frame, across
//                                                         codeword boundaries; the last symbol carries the carriers that still
//                                                         have a first bit, the rest of its carriers stay empty)
//   generatePreamble / generateTrainingSymbols            :479-580  (payload independent: built once on the host, copied)
//   peak normalisation of the tools                       tools/test_mode_snr.cpp:52-56
// The inverse FFT is the reference's radix-2 DIT with conjugated twiddles and 1/N scaling on a shared-memory buffer
// (fft_smem.cuh); constellation points / differential steps come from host-built tables, so no libm call is involved.
#include "fft_smem.cuh"
#include "ldpc_encode.cuh"
#include "ofdm_dev.cuh"
#include "pu_internal.h"

namespace pu {

struct TxDev {
    int nfft, cp, sym_len, guard, n_data, n_pilot, bps, differential;
    int pre_len, n_sym, frame_len;     // preamble samples, data symbols, total samples
    int osc_start;                     // mixer position of the first data symbol (the Schmidl-Cox preamble repeats one STS and one
                                       // LTS waveform, so the mixer has only advanced by two symbols there: modulator.cpp:479-532)
    float scale;                       // ModemConfig::output_scale
    int il_inv;                        // pu_ofdm_set_tx_interleave: step^-1 mod 648 of ChannelInterleaver (bit j of a codeword is coded
                                       // bit j * il_inv mod 648), 0 = no interleaving
    LdpcEncDev enc;                    // LDPC dimensions and tables (ldpc_encode.cuh)
    const int* data_bin;
    const int* pilot_bin;
    const float* pilot_sign;
    const float2* twiddle;
    const float2* osc;                 // [frame_len] TX mixer NCO::next() samples (center_freq + tx_cfo)
    const float* preamble;             // [pre_len]
    const float2* points;              // [1 << bps] constellation points (coherent) or differential steps
};

// Shared memory of one CTA: the encoder's coded frame and parity table (ldpc_encode_smem; 255 codewords take 20.7 KB of coded bytes)
template <int NFFT>
__global__ void __launch_bounds__(128) ofdm_tx_kernel(TxDev t, const uint8_t* __restrict__ frames, size_t frame_stride, int frame_bytes, int n_cw,
                                                      int bpc, float peak, float* __restrict__ out, size_t out_stride) {
    __shared__ float2 buf[NFFT];
    __shared__ float red[4];
    extern __shared__ __align__(16) uint8_t tx_smem[];
    uint8_t* coded = tx_smem;
    const int tid = threadIdx.x, T = blockDim.x;
    const uint8_t* fr = frames + static_cast<size_t>(blockIdx.x) * frame_stride;
    float* w = out + static_cast<size_t>(blockIdx.x) * out_stride;

    for (int i = tid; i < t.pre_len; i += T) w[i] = __ldg(&t.preamble[i]);
    ldpc_encode_frame_cta(t.enc, fr, frame_bytes, n_cw, bpc, coded, ldpc_encode_parity_of(tx_smem, n_cw));

    const int total_bits = n_cw * PU_LDPC_N;
    const int per_sym = t.n_data * t.bps;
    float2 diff = make_float2(1.0f, 0.0f);                // this thread's carrier (tid < n_data), carried over the symbols of the frame
    float mx = 0.0f;
    if (peak > 0.0f)
        for (int i = tid; i < t.pre_len; i += T) mx = fmaxf(mx, fabsf(__ldg(&t.preamble[i])));
    for (int s = 0; s < t.n_sym; ++s) {
        for (int i = tid; i < NFFT; i += T) buf[i] = make_float2(0.0f, 0.0f);
        __syncthreads();
        if (tid < t.n_data) {
            const int b0 = s * per_sym + tid * t.bps;
            if (b0 < total_bits) {                        // a carrier exists while data remains at its first bit (:418-436)
                unsigned v = 0;
                for (int b = 0; b < t.bps; ++b) {
                    int bit = b0 + b;
                    if (t.il_inv && bit < total_bits) {   // the codeword's own ChannelInterleaver: the coded bytes stay as encoded
                        const int c = bit / PU_LDPC_N;
                        bit = c * PU_LDPC_N + (bit - c * PU_LDPC_N) * t.il_inv % PU_LDPC_N;
                    }
                    v = (v << 1) | ((bit < total_bits) ? ((coded[bit >> 3] >> (7 - (bit & 7))) & 1u) : 0u);
                }
                float2 sym = __ldg(&t.points[v]);
                if (t.differential) {
                    sym = cmul(diff, sym);                // diff_state * step
                    diff = sym;
                }
                buf[t.data_bin[tid]] = sym;
            }
        }
        if (tid < t.n_pilot) buf[t.pilot_bin[tid]] = make_float2(t.pilot_sign[tid], 0.0f);
        __syncthreads();
        fft_smem<NFFT>(buf, t.twiddle, true);
        const int base = t.pre_len + s * t.sym_len;
        for (int i = tid; i < t.cp + NFFT; i += T) {
            const float2 v = buf[i < t.cp ? NFFT - t.cp + i : i - t.cp];
            const float x = __fmul_rn(cmul(v, __ldg(&t.osc[t.osc_start + s * t.sym_len + i])).x, t.scale);   // (v * osc).real() * scale
            w[base + i] = x;
            mx = fmaxf(mx, fabsf(x));
        }
        for (int i = tid; i < t.guard; i += T) w[base + t.cp + NFFT + i] = 0.0f;
        __syncthreads();
    }
    if (peak > 0.0f) {                                    // w * (peak / max|w|), tools/test_mode_snr.cpp:52-56
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((tid & 31) == 0) red[tid >> 5] = mx;
        __syncthreads();
        mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
        if (mx > 0.0f) {
            const float f = __fdiv_rn(peak, mx);
            for (int i = tid; i < t.frame_len; i += T) w[i] = __fmul_rn(w[i], f);
        }
    }
}

cudaError_t ofdm_tx_launch(const TxDev& t, const uint8_t* frames, size_t frame_stride, int frame_bytes, int n_cw, int bpc, size_t B, float peak,
                           float* out, size_t out_stride, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    const size_t smem = ldpc_encode_smem(n_cw, t.enc.m);
    if (t.nfft == 512)
        ofdm_tx_kernel<512><<<static_cast<unsigned>(B), 128, smem, st>>>(t, frames, frame_stride, frame_bytes, n_cw, bpc, peak, out, out_stride);
    else
        ofdm_tx_kernel<1024><<<static_cast<unsigned>(B), 128, smem, st>>>(t, frames, frame_stride, frame_bytes, n_cw, bpc, peak, out, out_stride);
    return cudaGetLastError();
}

}  // namespace pu
