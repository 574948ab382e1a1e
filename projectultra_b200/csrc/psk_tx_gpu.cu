// projectultra_b200/csrc/psk_tx_gpu.cu — batched single-carrier and multi-carrier DPSK transmitters on the GPU (SURVEY §8f next-3, PSK
// half): LDPC encode + modulate, one frame per CTA, so that every Monte-Carlo trial of a PSK sweep carries its own payload like the
// reference's tools do (tools/test_dpsk_snr.cpp:40-60, tools/test_mc_dpsk.cpp:180-196) instead of indexing a host-built pool.
//
// Reference behaviour (bit-identical waveforms; the host twins are csrc/psk_tx.cpp: pu_dpsk_tx / pu_mcdpsk_tx):
//   LDPCEncoder::encode                                      src/fec/ldpc_encoder.cpp:193-257
//   DPSKModulator::generatePreamble / modulate / modulateSymbol   src/psk/dpsk.hpp:118-153, 212-279 (raised-cosine pulse :289-300)
//   MultiCarrierDPSKModulator::generateTrainingSequence / generateReferenceSymbol / modulate   src/psk/multi_carrier_dpsk.hpp:118-243
// What depends on the payload is little: the per-symbol phase (a serial float recurrence over <= 648 symbols) and the per-carrier
// differential state.  Everything else is a function of the sample index alone and is tabulated ON THE HOST with the host libm, as
// the reference evaluates it: the Barker preamble / training + reference symbols (copied), the carrier phase of every data sample
// (the reference's `carrier_phase += inc` recurrence with its once-per-symbol wrap), the pulse shape, polar(1, i * inc_c) per
// (carrier, sample).  The device evaluates cos(carrier_phase + symbol_phase) with the glibc restatement of ref_math.cuh.
#include <cmath>
#include <complex>
#include <vector>

#include "ldpc_encode.cuh"
#include "ofdm_dev.cuh"
#include "psk_handles.h"
#include "ref_math.cuh"

void pu_ldpc_encoder_view(const pu_ldpc* h, int* k, int* m, const uint8_t** cn_ninfo, const uint16_t** cn_check, const uint16_t** cn_var);   // ldpc_decode.cu
namespace pu { std::vector<float> mcdpsk_carrier_freqs(const pu_mcdpsk_config& c); }   // psk_tx.cpp

namespace pu {

constexpr double kTxPi = 3.14159265358979323846;   // M_PI

// LDPCEncoder::encode of one block into bits[648]: k information bits (payload, zero padded), then the m parity bits
__device__ __forceinline__ void encode_block(const LdpcEncDev& e, const uint8_t* __restrict__ pl, int payload_bytes, uint8_t* bits) {
    const int tid = threadIdx.x, T = blockDim.x;
    for (int j = tid; j < e.k; j += T) bits[j] = (j < payload_bytes * 8) ? ((pl[j >> 3] >> (7 - (j & 7))) & 1) : 0;
    __syncthreads();
    for (int p = tid; p < e.m; p += T) {
        unsigned acc = 0;
        const int ninfo = e.cn_ninfo[p];
        for (int q = 0; q < ninfo; ++q) acc ^= bits[e.cn_var[q * e.m + p]];
        bits[e.k + e.cn_check[p]] = static_cast<uint8_t>(acc);
    }
    __syncthreads();
}

// w *= peak / max|w| over the frame (tools/test_mode_snr.cpp:52-56); mx = this thread's running maximum
__device__ __forceinline__ void peak_normalise(float* w, int frame_len, float peak, float mx, float* red) {
    const int tid = threadIdx.x, T = blockDim.x;
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = 0.0f;
    for (int i = 0; i < (T >> 5); ++i) mx = fmaxf(mx, red[i]);
    if (mx > 0.0f) {
        const float f = __fdiv_rn(peak, mx);
        for (int i = tid; i < frame_len; i += T) w[i] = __fmul_rn(w[i], f);
    }
}

struct DpskTxDev {
    LdpcEncDev enc;
    int sps, bps, nsym, pre_len, frame_len;
    float inc_tab[8];            // DPSKConfig::phase_increment(v), dpsk.hpp:72-86
    float symbol_phase0;         // symbol_phase_ behind the preamble
    const float* preamble;       // [pre_len]
    const float* phase;          // [nsym * sps] carrier_phase_ at every data sample
    const float* pulse;          // [sps]
};

__global__ void __launch_bounds__(256) dpsk_tx_kernel(DpskTxDev t, const uint8_t* __restrict__ payload, size_t payload_stride, int payload_bytes,
                                                      float peak, float* __restrict__ out, size_t out_stride) {
    __shared__ uint8_t bits[PU_LDPC_N];
    __shared__ float symphase[PU_LDPC_N];
    __shared__ float red[8];
    const int tid = threadIdx.x, T = blockDim.x;
    float* w = out + static_cast<size_t>(blockIdx.x) * out_stride;
    encode_block(t.enc, payload + static_cast<size_t>(blockIdx.x) * payload_stride, payload_bytes, bits);
    float mx = 0.0f;
    for (int i = tid; i < t.pre_len; i += T) {
        const float v = __ldg(&t.preamble[i]);
        w[i] = v;
        mx = fmaxf(mx, fabsf(v));
    }
    if (tid == 0) {      // modulateSymbol's symbol_phase_ recurrence (:252-254): serial, float, wrapped against the DOUBLE 2 pi
        float sp = t.symbol_phase0;
        for (int s = 0; s < t.nsym; ++s) {
            int v = 0;
            for (int b = 0; b < t.bps; ++b)
                if (bits[s * t.bps + b]) v |= 1 << (t.bps - 1 - b);
            sp = __fadd_rn(sp, t.inc_tab[v]);
            while (static_cast<double>(sp) >= 2.0f * kTxPi) sp = static_cast<float>(static_cast<double>(sp) - 2.0f * kTxPi);
            symphase[s] = sp;
        }
    }
    __syncthreads();
    const int n_data = t.nsym * t.sps;
    for (int n = tid; n < n_data; n += T) {
        const int s = n / t.sps, i = n - s * t.sps;
        const float x = __fmul_rn(__ldg(&t.pulse[i]), refmath::cosf_ref(__fadd_rn(__ldg(&t.phase[n]), symphase[s])));   // :262-266
        w[t.pre_len + n] = x;
        mx = fmaxf(mx, fabsf(x));
    }
    if (peak > 0.0f) {
        __syncthreads();
        peak_normalise(w, t.frame_len, peak, mx, red);
    }
}

struct McTxDev {
    LdpcEncDev enc;
    int nc, sps, bits_c, nsym, pre_len, frame_len;
    int il_inv;                  // pu_mcdpsk_set_tx_interleave: coded bit j * il_inv mod 648 goes out as bit j; 0 = no interleaving
    float2 change[4];            // std::polar(1.0f, phase change of symbol value v), multi_carrier_dpsk.hpp:198-214
    const float* preamble;       // [pre_len] training sequence + reference symbol
    const float2* polar;         // [nc][sps] std::polar(1.0f, i * inc_c)
};

constexpr int kMcMaxCarriers = 64;

__global__ void __launch_bounds__(256) mcdpsk_tx_kernel(McTxDev t, const uint8_t* __restrict__ payload, size_t payload_stride, int payload_bytes,
                                                        float peak, float* __restrict__ out, size_t out_stride) {
    extern __shared__ float2 cur[];          // [nsym][nc] differential state of every (symbol, carrier)
    __shared__ uint8_t bits[PU_LDPC_N];
    __shared__ float red[8];
    const int tid = threadIdx.x, T = blockDim.x;
    float* w = out + static_cast<size_t>(blockIdx.x) * out_stride;
    encode_block(t.enc, payload + static_cast<size_t>(blockIdx.x) * payload_stride, payload_bytes, bits);
    float mx = 0.0f;
    for (int i = tid; i < t.pre_len; i += T) {
        const float v = __ldg(&t.preamble[i]);
        w[i] = v;
        mx = fmaxf(mx, fabsf(v));
    }
    if (tid < t.nc) {    // per carrier: current = prev * polar(1, change); current /= |current| (:216-221), serial over the symbols
        float2 prev = make_float2(1.0f, 0.0f);                       // the reference symbol (:161-163)
        for (int s = 0; s < t.nsym; ++s) {
            int v = 0;
            for (int b = 0; b < t.bits_c; ++b) {
                const int pos = (s * t.nc + tid) * t.bits_c + b;
                v = (v << 1) | (pos < PU_LDPC_N ? bits[t.il_inv ? pos * t.il_inv % PU_LDPC_N : pos] : 0);   // zero padding of the last symbol (:186-188)
            }
            float2 c = cmul(prev, t.change[v]);
            c = cdivs(c, cabs_ref(c));
            prev = c;
            cur[s * t.nc + tid] = c;
        }
    }
    __syncthreads();
    const int n_data = t.nsym * t.sps;
    const float ncf = static_cast<float>(t.nc);
    for (int n = tid; n < n_data; n += T) {
        const int s = n / t.sps, i = n - s * t.sps;
        float acc = 0.0f;
        for (int c = 0; c < t.nc; ++c) {                             // output[i] += (current * polar(1, t)).real() / nc, carriers in order
            const float2 p = __ldg(&t.polar[c * t.sps + i]);
            const float2 z = cur[s * t.nc + c];
            acc = __fadd_rn(acc, __fdiv_rn(__fsub_rn(__fmul_rn(z.x, p.x), __fmul_rn(z.y, p.y)), ncf));
        }
        w[t.pre_len + n] = acc;
        mx = fmaxf(mx, fabsf(acc));
    }
    if (peak > 0.0f) {
        __syncthreads();
        peak_normalise(w, t.frame_len, peak, mx, red);
    }
}

}  // namespace pu

extern "C" {
pu_status pu_dpsk_tx(const pu_dpsk_config* cfg, int layout, const uint8_t* data, size_t n_bytes, float* out, size_t out_cap, size_t* out_len);
pu_status pu_mcdpsk_tx(const pu_mcdpsk_config* cfg, const uint8_t* data, size_t n_bytes, float* out, size_t out_cap, size_t* out_len);

pu_status pu_dpsk_tx_batch(pu_dpsk* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes, size_t B,
                           float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream) {
    PU_REQUIRE(h && code && frame_len, "pu_dpsk_tx_batch: NULL argument");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu::DpskTxDev t{};
    pu_ldpc_encoder_view(code, &t.enc.k, &t.enc.m, &t.enc.cn_ninfo, &t.enc.cn_check, &t.enc.cn_var);
    PU_REQUIRE(payload_bytes * 8 <= static_cast<size_t>(t.enc.k) && payload_bytes <= payload_stride, "pu_dpsk_tx_batch: payload longer than one codeword's information bits");
    const pu_dpsk_config& c = h->cfg;
    t.sps = static_cast<int>(c.samples_per_symbol);
    t.bps = c.modulation == 0 ? 1 : c.modulation == 1 ? 2 : 3;
    t.nsym = (PU_LDPC_N + t.bps - 1) / t.bps;
    pu_status s;
    if (h->tx_pre_len == 0) {
        // generatePreamble (dpsk.hpp:118-153) through the host transmitter, then the state it leaves behind: the carrier phase of
        // every later sample (`carrier_phase_ += inc` per sample, wrapped once per symbol, :268-276) and symbol_phase_
        size_t n = 0;
        pu_dpsk_tx(&c, 0, nullptr, 0, nullptr, 0, &n);
        std::vector<float> pre(n);
        if ((s = pu_dpsk_tx(&c, 0, nullptr, 0, pre.data(), n, &n)) != PU_OK) return s;
        static const int barker[13] = {1, 1, 1, 1, 1, -1, -1, 1, 1, -1, 1, -1, 1};
        const float inc = static_cast<float>(2.0f * pu::kTxPi * c.carrier_freq / c.sample_rate);
        float phase = 0.0f, sym_phase = 0.0f;
        for (int rep = 0; rep < 3; ++rep)
            for (int b = 0; b < 13; ++b) {
                if (barker[b] < 0) sym_phase = static_cast<float>(sym_phase + pu::kTxPi);
                for (uint32_t i = 0; i < c.samples_per_symbol; ++i) {
                    phase += inc;
                    if (phase > 2.0f * pu::kTxPi) phase = static_cast<float>(phase - 2.0f * pu::kTxPi);
                }
            }
        const int max_sym = PU_LDPC_N;      // DBPSK: one symbol per coded bit
        std::vector<float> tab(static_cast<size_t>(max_sym) * t.sps);
        float cp = phase;
        for (int sy = 0; sy < max_sym; ++sy) {
            for (int i = 0; i < t.sps; ++i) {
                tab[static_cast<size_t>(sy) * t.sps + i] = cp;
                cp += inc;
            }
            while (cp >= 2.0f * pu::kTxPi) cp = static_cast<float>(cp - 2.0f * pu::kTxPi);
        }
        std::vector<float> pulse(t.sps);
        for (int i = 0; i < t.sps; ++i) {                              // buildPulseShape, :289-300
            const float tt = static_cast<float>(i) / t.sps;
            pulse[i] = static_cast<float>(0.5f * (1.0f - std::cos(2.0f * pu::kTxPi * tt)));
        }
        if ((s = h->d_tx_pre.upload(pre.data(), pre.size())) != PU_OK || (s = h->d_tx_phase.upload(tab.data(), tab.size())) != PU_OK ||
            (s = h->d_tx_pulse.upload(pulse.data(), pulse.size())) != PU_OK)
            return s;
        h->tx_pre_len = pre.size();
        h->tx_phase_syms = static_cast<size_t>(max_sym);
        h->tx_symbol_phase0 = sym_phase;
    }
    t.pre_len = static_cast<int>(h->tx_pre_len);
    t.frame_len = t.pre_len + t.nsym * t.sps;
    *frame_len = static_cast<size_t>(t.frame_len);
    if (B == 0 || !out) return PU_OK;                // length query
    PU_REQUIRE(payload && out_stride >= static_cast<size_t>(t.frame_len), "pu_dpsk_tx_batch: output rows shorter than a frame");
    for (int v = 0; v < 8; ++v)                      // DPSKConfig::phase_increment, :72-86
        t.inc_tab[v] = c.modulation == 0 ? ((v & 1) ? static_cast<float>(pu::kTxPi) : 0.0f)
                       : c.modulation == 1 ? static_cast<float>(((v & 3) * 2 + 1) * pu::kTxPi / 4.0f)
                                           : static_cast<float>((v & 7) * pu::kTxPi / 4.0f + pu::kTxPi / 8.0f);
    t.symbol_phase0 = h->tx_symbol_phase0;
    t.preamble = static_cast<const float*>(h->d_tx_pre.p);
    t.phase = static_cast<const float*>(h->d_tx_phase.p);
    t.pulse = static_cast<const float*>(h->d_tx_pulse.p);
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    (void)cudaGetLastError();
    if (space == PU_MEM_HOST) {
        // host memory: every output row comes back whole, zeros beyond *frame_len
        pu::HostStage hs(ctx, st, B);
        const uint8_t* d_payload;
        float* d_tx;
        hs.in(&d_payload, payload, payload_stride);
        hs.out(&d_tx, out, out_stride);
        return hs.run([&](size_t nb) {
            return pu_dpsk_tx_batch(h, code, d_payload, payload_stride, payload_bytes, nb, peak, d_tx, out_stride, frame_len, PU_MEM_DEVICE, st);
        });
    }
    pu::dpsk_tx_kernel<<<static_cast<unsigned>(B), 256, 0, st>>>(t, payload, payload_stride, static_cast<int>(payload_bytes), peak, out, out_stride);
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_mcdpsk_tx_batch(pu_mcdpsk* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes, size_t B,
                             float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream) {
    PU_REQUIRE(h && code && frame_len, "pu_mcdpsk_tx_batch: NULL argument");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu::McTxDev t{};
    pu_ldpc_encoder_view(code, &t.enc.k, &t.enc.m, &t.enc.cn_ninfo, &t.enc.cn_check, &t.enc.cn_var);
    PU_REQUIRE(payload_bytes * 8 <= static_cast<size_t>(t.enc.k) && payload_bytes <= payload_stride, "pu_mcdpsk_tx_batch: payload longer than one codeword's information bits");
    const pu_mcdpsk_config& c = h->cfg;
    PU_REQUIRE(c.num_carriers <= pu::kMcMaxCarriers && (c.bits_per_symbol == 1 || c.bits_per_symbol == 2), "pu_mcdpsk_tx_batch: bad configuration");
    t.nc = static_cast<int>(c.num_carriers); t.sps = static_cast<int>(c.samples_per_symbol); t.bits_c = static_cast<int>(c.bits_per_symbol);
    const int per_sym = t.nc * t.bits_c;
    t.nsym = (PU_LDPC_N + per_sym - 1) / per_sym;
    pu_status s;
    if (h->tx_pre_len == 0) {
        size_t n = 0;
        pu_mcdpsk_tx(&c, nullptr, 0, nullptr, 0, &n);              // training sequence + reference symbol (:118-173)
        std::vector<float> pre(n);
        if ((s = pu_mcdpsk_tx(&c, nullptr, 0, pre.data(), n, &n)) != PU_OK) return s;
        const std::vector<float> freqs = pu::mcdpsk_carrier_freqs(c);
        std::vector<std::complex<float>> pol(static_cast<size_t>(t.nc) * t.sps);
        for (int k = 0; k < t.nc; ++k) {
            const float inc = static_cast<float>(2.0f * pu::kTxPi * freqs[k] / c.sample_rate);
            for (int i = 0; i < t.sps; ++i) pol[static_cast<size_t>(k) * t.sps + i] = std::polar(1.0f, i * inc);   // :226-229
        }
        if ((s = h->d_tx_pre.upload(pre.data(), pre.size())) != PU_OK || (s = h->d_tx_polar.upload(pol.data(), pol.size())) != PU_OK) return s;
        h->tx_pre_len = pre.size();
    }
    t.pre_len = static_cast<int>(h->tx_pre_len);
    t.frame_len = t.pre_len + t.nsym * t.sps;
    *frame_len = static_cast<size_t>(t.frame_len);
    if (B == 0 || !out) return PU_OK;
    PU_REQUIRE(payload && out_stride >= static_cast<size_t>(t.frame_len), "pu_mcdpsk_tx_batch: output rows shorter than a frame");
    static const float dqpsk_phases[] = {static_cast<float>(pu::kTxPi / 4), static_cast<float>(3 * pu::kTxPi / 4),
                                         static_cast<float>(-3 * pu::kTxPi / 4), static_cast<float>(-pu::kTxPi / 4)};
    for (int v = 0; v < 4; ++v) {
        const float change = t.bits_c == 2 ? dqpsk_phases[v] : ((v & 1) ? static_cast<float>(pu::kTxPi) : 0.0f);
        const std::complex<float> p = std::polar(1.0f, change);
        t.change[v] = make_float2(p.real(), p.imag());
    }
    t.preamble = static_cast<const float*>(h->d_tx_pre.p);
    t.polar = static_cast<const float2*>(h->d_tx_polar.p);
    t.il_inv = h->tx_il_inv;
    const size_t smem = static_cast<size_t>(t.nsym) * t.nc * sizeof(float2);
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    (void)cudaGetLastError();
    if (space == PU_MEM_HOST) {
        // host memory: every output row comes back whole, zeros beyond *frame_len
        pu::HostStage hs(ctx, st, B);
        const uint8_t* d_payload;
        float* d_tx;
        hs.in(&d_payload, payload, payload_stride);
        hs.out(&d_tx, out, out_stride);
        return hs.run([&](size_t nb) {
            return pu_mcdpsk_tx_batch(h, code, d_payload, payload_stride, payload_bytes, nb, peak, d_tx, out_stride, frame_len, PU_MEM_DEVICE, st);
        });
    }
    pu::mcdpsk_tx_kernel<<<static_cast<unsigned>(B), 256, smem, st>>>(t, payload, payload_stride, static_cast<int>(payload_bytes), peak, out, out_stride);
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_mcdpsk_set_tx_interleave(pu_mcdpsk* h, size_t bits_per_symbol) {
    PU_REQUIRE(h, "pu_mcdpsk_set_tx_interleave: NULL handle");
    h->tx_il_inv = bits_per_symbol ? static_cast<int>(pu::channel_interleaver_inverse_step(bits_per_symbol)) : 0;
    return PU_OK;
}

}  // extern "C"
