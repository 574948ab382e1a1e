// projectultra_b200/csrc/channel.cu — batched Watterson two-tap Rayleigh fading + AWGN channel for sm_100a and
// the pu_channel_* entry points of the C ABI.
//
// Reference behaviour: sim::WattersonChannel (src/sim/hf_channel.hpp:67-168,258-275) -- per sample
//   fading_k <- (1-a) fading_k + a * sqrt(1/a) * (N(0,1) + j N(0,1)),  k = 1, 2, both starting from (1, 0)  (:91-92, :258-275)
//   out = x[n] g1 |fading_1| + x[n-d-1] g2 |fading_2| + sigma N(0,1)                                    (:125-153)
// with d = floor(delay_ms * fs / 1000) (:72-78; the d+1-entry zero-initialised deque gives an effective delay of d+1
// samples, SURVEY Q11), a = 1 - exp(-2 pi f_d / fs) (:87-88) and sigma = rms(input) * 10^(-snr/20) (:110-119).
// What is NOT reproduced is the reference's random stream (mt19937 + libstdc++ normal_distribution, implementation
// defined): it is replaced by the counter-based generator of pu_rng.cuh, and the one-pole recurrence is evaluated as
// a 32-wide inclusive scan with fused multiply-adds instead of sample by sample.  Both are a SPECIFICATION of this
// simulator, restated independently by the CPU twin oracle/pu_oracle_channel.c (bit-identical output); against the
// reference the channel is checked statistically (tests/test_channel_gpu.py).  The optional CFO injector of the
// reference (applyCFO, :173-232) is out of scope: the Monte-Carlo configs are CFO-free (SURVEY §8d).
//
// Kernel shape: one warp per frame; lane l owns samples 128 g + 4 l .. + 3 (16-byte coalesced loads/stores); the recurrence is
// serial over a lane's four samples and a Kogge-Stone scan over the lanes (see channel_kernel).
#include <cmath>
#include <memory>
#include <new>
#include <vector>

#include "pu_internal.h"
#include "pu_rng.cuh"
#include "ref_math.cuh"

namespace pu {

struct ChannelParams {
    int fading, multipath, noise;
    int delay;               // d: second path reads x[n - d - 1]
    float g1, g2;
    float alpha, noise_scale;       // a, sqrt(1/a)
    float qj[4];             // (1-a)^(j+1): carry-in weight of a lane's j-th sample
    float qs[5];             // (1-a)^(4 * 2^s): Kogge-Stone multipliers over lanes (a lane spans 4 samples)
    float ql[32];            // (1-a)^(4 l): weight of the group's carry-in at lane l
};

// One warp per frame, 128 samples per step: lane l owns samples base + 4 l .. 4 l + 3 (one 16-byte load / store, one Philox call
// for its four noise normals, two for its 16 fading innovations).  The one-pole recurrence f[n] = q f[n-1] + e[n] is evaluated as
//   in-lane:  s_0 = e_0, s_j = fma(q, s_{j-1}, e_j)                     (the lane's own innovations, zero state before the lane)
//   lanes:    inclusive Kogge-Stone scan of A_l = s_3 with multipliers q^(4 2^s); E_l = A_{l-1} (0 for lane 0)
//   carry:    P_l = fma(q^(4 l), C, E_l),  f_j = fma(q^(j+1), P_l, s_j),  C' = f_3 of lane 31
// -- the evaluation order is part of the simulator's specification (restated by the CPU twin oracle/pu_oracle_channel.c).
__global__ void __launch_bounds__(256) channel_kernel(ChannelParams p, const float* __restrict__ tx_pool, size_t pool_stride,
                                                      const uint32_t* __restrict__ tx_index, const float* __restrict__ noise_std,
                                                      const uint64_t* __restrict__ seed, size_t B, int L,
                                                      float* __restrict__ rx) {
    const int lane = threadIdx.x & 31;
    const size_t frame = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
    if (frame >= B) return;
    const float* x = tx_pool + static_cast<size_t>(tx_index ? tx_index[frame] : 0) * pool_stride;
    float* y = rx + frame * static_cast<size_t>(L);
    const uint64_t sd = seed[frame];
    const uint32_t k0 = static_cast<uint32_t>(sd), k1 = static_cast<uint32_t>(sd >> 32);
    const float sigma = noise_std[frame];
    const float ql = p.ql[lane];
    const float q = p.qj[0];
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
    const bool two_path = p.multipath && p.delay > 0;
    float carry[4] = {1.0f, 0.0f, 1.0f, 0.0f};   // fading1_, fading2_ start at (1, 0)
    for (int base = 0; base < L; base += 128) {
        const int n0 = base + 4 * lane;
        float xv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (vec && n0 + 3 < L) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(x + n0));
            xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (n0 + j < L) xv[j] = __ldg(&x[n0 + j]);
        }
        float m1[4] = {1.0f, 1.0f, 1.0f, 1.0f}, m2[4] = {1.0f, 1.0f, 1.0f, 1.0f};
        if (p.fading) {
            float z[4][4];      // [sample j][component]
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float zz[2][4];
                rng::fading_innovations2(k0, k1, static_cast<uint32_t>((n0 >> 1) + h), zz);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    z[2 * h][c] = (n0 + 2 * h < L) ? zz[0][c] : 0.0f;
                    z[2 * h + 1][c] = (n0 + 2 * h + 1 < L) ? zz[1][c] : 0.0f;
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float s[4];
                s[0] = rng::r_mul(p.alpha, rng::r_mul(p.noise_scale, z[0][c]));
#pragma unroll
                for (int j = 1; j < 4; ++j) s[j] = rng::r_fma(q, s[j - 1], rng::r_mul(p.alpha, rng::r_mul(p.noise_scale, z[j][c])));
                float v = s[3];
#pragma unroll
                for (int t = 0; t < 5; ++t) {
                    const float up = __shfl_up_sync(0xffffffffu, v, 1 << t);
                    if (lane >= (1 << t)) v = rng::r_fma(p.qs[t], up, v);
                }
                float e = __shfl_up_sync(0xffffffffu, v, 1);
                if (lane == 0) e = 0.0f;
                const float pl = rng::r_fma(ql, carry[c], e);
                float f[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) f[j] = rng::r_fma(p.qj[j], pl, s[j]);
                carry[c] = __shfl_sync(0xffffffffu, f[3], 31);
#pragma unroll
                for (int j = 0; j < 4; ++j) z[j][c] = f[j];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                m1[j] = rng::r_sqrt(rng::r_fma(z[j][0], z[j][0], rng::r_mul(z[j][1], z[j][1])));
                m2[j] = rng::r_sqrt(rng::r_fma(z[j][2], z[j][2], rng::r_mul(z[j][3], z[j][3])));
            }
        }
        if (n0 >= L) continue;
        float zn[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (p.noise) {
            const rng::U4 w = rng::philox4x32_10(static_cast<uint32_t>(n0 >> 2), 0u, rng::kStreamNoise, 0u, k0, k1);
            rng::box_muller(w.x, w.y, &zn[0], &zn[1]);
            rng::box_muller(w.z, w.w, &zn[2], &zn[3]);
        }
        float out[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (two_path) {
                const int nd = n0 + j - p.delay - 1;
                const float xd = (nd >= 0 && n0 + j < L) ? __ldg(&x[nd]) : 0.0f;
                out[j] = rng::r_fma(rng::r_mul(xd, p.g2), m2[j], rng::r_mul(rng::r_mul(xv[j], p.g1), m1[j]));
            } else {
                out[j] = rng::r_mul(xv[j], m1[j]);
            }
            if (p.noise) out[j] = rng::r_fma(sigma, zn[j], out[j]);
        }
        if (vec && n0 + 3 < L) {
            *reinterpret_cast<float4*>(y + n0) = make_float4(out[0], out[1], out[2], out[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (n0 + j < L) y[n0 + j] = out[j];
        }
    }
}

// AWGN-only fast path: no recurrence, each lane produces 4 consecutive samples from one Philox call.
__global__ void __launch_bounds__(256) awgn_kernel(const float* __restrict__ tx_pool, size_t pool_stride,
                                                   const uint32_t* __restrict__ tx_index, const float* __restrict__ noise_std,
                                                   const uint64_t* __restrict__ seed, size_t B, int L, float* __restrict__ rx) {
    const int lane = threadIdx.x & 31;
    const size_t frame = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
    if (frame >= B) return;
    const float* x = tx_pool + static_cast<size_t>(tx_index ? tx_index[frame] : 0) * pool_stride;
    float* y = rx + frame * static_cast<size_t>(L);
    const uint64_t sd = seed[frame];
    const uint32_t k0 = static_cast<uint32_t>(sd), k1 = static_cast<uint32_t>(sd >> 32);
    const float sigma = noise_std[frame];
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
    for (int q = lane; 4 * q < L; q += 32) {
        const rng::U4 w = rng::philox4x32_10(static_cast<uint32_t>(q), 0u, rng::kStreamNoise, 0u, k0, k1);
        float z[4];
        rng::box_muller(w.x, w.y, &z[0], &z[1]);
        rng::box_muller(w.z, w.w, &z[2], &z[3]);
        const int n = 4 * q;
        if (vec && n + 3 < L) {
            const float4 xv = __ldg(reinterpret_cast<const float4*>(x + n));
            float4 o;
            o.x = rng::r_fma(sigma, z[0], xv.x);
            o.y = rng::r_fma(sigma, z[1], xv.y);
            o.z = rng::r_fma(sigma, z[2], xv.z);
            o.w = rng::r_fma(sigma, z[3], xv.w);
            *reinterpret_cast<float4*>(y + n) = o;
        } else {
            for (int j = 0; j < 4 && n + j < L; ++j) y[n + j] = rng::r_fma(sigma, z[j], __ldg(&x[n + j]));
        }
    }
}

// WattersonChannel::applyCFO (src/sim/hf_channel.hpp:173-232), the channel's optional CFO injector, in place on one frame per warp:
// mix to baseband around 1500 Hz, 48-tap running-sum lowpass, rotate by the CFO phase, mix back up.  The running sums and the phase
// are serial float recurrences (`sum += x[i]; sum -= x[i-48]`, `phase += inc` with its one-sided wrap): three lanes walk them 32
// samples at a time out of shared memory while the mixing before and after them runs on all lanes.  Deterministic (no random draw),
// so this kernel IS pinned bit for bit to the reference (tests/test_channel.py) -- the mixer table comes from the host libm as the
// reference evaluates it, the rotator's cos/sin are the glibc restatements of ref_math.cuh (|phase| stays far below 120).
constexpr int kCfoWin = 48;
__global__ void __launch_bounds__(128) channel_cfo_kernel(float* __restrict__ samples, size_t stride, size_t B, int L, const float* __restrict__ cfo_hz,
                                                          double fs_d, const float2* __restrict__ mix) {
    __shared__ float ring[4][2][96];       // I_bb / Q_bb of the last 96 samples (index i % 96)
    __shared__ float stage[4][3][32];      // I_filt, Q_filt, phase of the chunk
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t frame = static_cast<size_t>(blockIdx.x) * 4 + warp;
    if (frame >= B) return;
    const float cfo = cfo_hz[frame];
    if (L < 256 || !(fabsf(cfo) > 0.001f)) return;        // :163, :174
    float* x = samples + frame * stride;
    const float phase_inc = static_cast<float>(__ddiv_rn(__dmul_rn(2.0f * 3.14159265358979323846, static_cast<double>(cfo)), fs_d));   // :101
    float acc = 0.0f;          // lane 0: I_sum, lane 1: Q_sum, lane 2: phase
    for (int base = 0; base < L; base += 32) {
        const int i = base + lane;
        float2 m = make_float2(0.0f, 0.0f);
        if (i < L) {
            m = __ldg(&mix[i]);
            const float xv = x[i];
            ring[warp][0][i % 96] = __fmul_rn(xv, m.x);
            ring[warp][1][i % 96] = __fmul_rn(xv, m.y);
        }
        __syncwarp();
        const int cnt = min(32, L - base);
        if (lane < 2) {
            const float* r = ring[warp][lane];
            for (int k = 0; k < cnt; ++k) {
                const int j = base + k;
                acc = __fadd_rn(acc, r[j % 96]);
                if (j >= kCfoWin) acc = __fsub_rn(acc, r[(j - kCfoWin) % 96]);
                stage[warp][lane][k] = __fdiv_rn(acc, static_cast<float>(min(j + 1, kCfoWin)));
            }
        } else if (lane == 2) {
            for (int k = 0; k < cnt; ++k) {
                stage[warp][2][k] = acc;
                acc = __fadd_rn(acc, phase_inc);
                if (static_cast<double>(acc) > 2.0f * 3.14159265358979323846) acc = static_cast<float>(static_cast<double>(acc) - 2.0f * 3.14159265358979323846);
            }
        }
        __syncwarp();
        if (i < L) {
            const float fi = stage[warp][0][lane], fq = stage[warp][1][lane], ph = stage[warp][2][lane];
            const float cc = refmath::cosf_ref(ph), cs = refmath::sinf_ref(ph);
            const float ic = __fsub_rn(__fmul_rn(fi, cc), __fmul_rn(fq, cs)), qc = __fadd_rn(__fmul_rn(fi, cs), __fmul_rn(fq, cc));
            x[i] = __fmul_rn(2.0f, __fsub_rn(__fmul_rn(ic, m.x), __fmul_rn(qc, m.y)));
        }
        __syncwarp();
    }
}

static ChannelParams make_params(const pu_channel_config& c) {
    ChannelParams p{};
    p.fading = c.fading_enabled != 0;
    p.multipath = c.multipath_enabled != 0;
    p.noise = c.noise_enabled != 0;
    p.delay = static_cast<int>(static_cast<size_t>(c.delay_spread_ms * static_cast<float>(c.sample_rate) / 1000.0f));   // hf_channel.hpp:72-75
    p.g1 = c.path1_gain;
    p.g2 = c.path2_gain;
    const float norm_doppler = c.doppler_spread_hz / static_cast<float>(c.sample_rate);
    p.alpha = static_cast<float>(1.0f - std::exp(-2.0f * 3.14159265358979323846 * norm_doppler));                      // :87-88
    p.noise_scale = p.alpha > 0.0f ? std::sqrt(1.0f / p.alpha) : 0.0f;                                                  // :264
    const float a = 1.0f - p.alpha;
    float v = a;
    for (int j = 0; j < 4; ++j) { p.qj[j] = v; v = v * a; }          // q, q^2, q^3, q^4 by repeated multiplication (fp32)
    v = p.qj[3];
    for (int s = 0; s < 5; ++s) { p.qs[s] = v; v = v * v; }          // q^4, q^8, ... by repeated squaring
    v = 1.0f;
    for (int l = 0; l < 32; ++l) { p.ql[l] = v; v = v * p.qj[3]; }   // 1, q^4, q^8, ... by repeated multiplication
    return p;
}

}  // namespace pu

namespace pu {
// pu_channel_noise_std for every row of tx[B][stride] (device): the ordered fp32 power sum of the reference's tools
// (tools/test_mode_snr.cpp:58-61) / of WattersonChannel::process (hf_channel.hpp:110-119), one thread per frame.  The
// SNR-dependent factor -- powf(10, snr/10) (convention 1) or powf(10, -snr/20) (convention 0) -- is evaluated on the host
// per SNR point and gathered per frame, so no device pow enters the noise level.
__global__ void noise_std_kernel(const float* __restrict__ tx, size_t stride, int L, size_t B, const float* __restrict__ factor, int convention,
                                 float* __restrict__ out) {
    const size_t b = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (b >= B) return;
    const float* w = tx + b * stride;
    float acc = 0.0f;
    for (int i = 0; i < L; ++i) acc = __fadd_rn(acc, __fmul_rn(w[i], w[i]));
    const float mean = __fdiv_rn(acc, static_cast<float>(L));
    out[b] = convention == 0 ? __fmul_rn(__fsqrt_rn(mean), factor[b]) : __fsqrt_rn(__fdiv_rn(mean, factor[b]));
}
}  // namespace pu

extern "C" {

pu_status pu_channel_params(const pu_channel_config* cfg, int32_t* delay_samples, float* alpha, float* noise_scale,
                            float* apow2_5, float* apl_32) {
    PU_REQUIRE(cfg, "pu_channel_params: NULL config");
    const pu::ChannelParams p = pu::make_params(*cfg);
    if (delay_samples) *delay_samples = p.delay;
    if (alpha) *alpha = p.alpha;
    if (noise_scale) *noise_scale = p.noise_scale;
    if (apow2_5) std::memcpy(apow2_5, p.qs, sizeof(p.qs));
    if (apl_32) std::memcpy(apl_32, p.ql, sizeof(p.ql));
    return PU_OK;
}

pu_status pu_channel_noise_std_batch(pu_ctx* ctx, const float* tx, size_t tx_stride, size_t L, size_t B, const float* snr_factor,
                                     int convention, float* noise_std, void* stream) {
    PU_REQUIRE(ctx, "pu_channel_noise_std_batch: NULL context");
    if (B == 0) return PU_OK;
    PU_REQUIRE(tx && snr_factor && noise_std && tx_stride >= L && L > 0, "pu_channel_noise_std_batch: bad argument");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    (void)cudaGetLastError();
    pu::noise_std_kernel<<<static_cast<unsigned>((B + 63) / 64), 64, 0, st>>>(tx, tx_stride, static_cast<int>(L), B, snr_factor, convention, noise_std);
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

}  // extern "C"

namespace pu {
// the ordered fp32 power sum of pu_channel_noise_std, separately: a sweep needs it once per waveform, not once per SNR point
float channel_power_sum(const float* tx, size_t L) {
    float acc = 0.0f;
    for (size_t i = 0; i < L; ++i) acc += tx[i] * tx[i];
    return acc;
}
float channel_noise_std_from_sum(float acc, size_t L, float snr_db, int convention) {
    if (convention == 0) {          // WattersonChannel::process, hf_channel.hpp:110-119
        const float rms = std::sqrt(acc / L);
        return rms * std::pow(10.0f, -snr_db / 20.0f);
    }
    const float sp = acc / L;       // tools/test_mode_snr.cpp:58-61 (mean frame power, AWGN tools)
    return std::sqrt(sp / std::pow(10.0f, snr_db / 10.0f));
}
}  // namespace pu

extern "C" {

float pu_channel_noise_std(const float* tx, size_t L, float snr_db, int convention) {
    if (!tx || L == 0) return 0.0f;
    return pu::channel_noise_std_from_sum(pu::channel_power_sum(tx, L), L, snr_db, convention);
}

pu_status pu_channel_apply_cfo_batch(pu_ctx* ctx, float* samples, size_t B, size_t L, size_t stride, const float* cfo_hz, uint32_t sample_rate,
                                     pu_memspace space, void* stream) {
    PU_REQUIRE(ctx, "pu_channel_apply_cfo_batch: NULL context");
    if (B == 0 || L == 0) return PU_OK;
    PU_REQUIRE(samples && cfo_hz && stride >= L && sample_rate > 0 && L < (1u << 30), "pu_channel_apply_cfo_batch: bad argument");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (ctx->cfo_mix_len < L || ctx->cfo_mix_fs != sample_rate) {
        // mix_phase = 2 pi fc t with t = float(i) / fs, evaluated as the reference does (double product stored to float, host cosf / sinf)
        std::vector<float2> tab(L);
        const float fc = 1500.0f, fs = static_cast<float>(sample_rate);
        for (size_t i = 0; i < L; ++i) {
            const float t = static_cast<float>(i) / fs;
            const float mix_phase = static_cast<float>(2.0f * 3.14159265358979323846 * fc * t);
            tab[i] = make_float2(std::cos(mix_phase), std::sin(mix_phase));
        }
        pu_status s = ctx->cfo_mix.reserve(L * sizeof(float2));
        if (s != PU_OK) return s;
        PU_CUDA_TRY(cudaMemcpyAsync(ctx->cfo_mix.ptr, tab.data(), L * sizeof(float2), cudaMemcpyHostToDevice, st));
        PU_CUDA_TRY(cudaStreamSynchronize(st));       // `tab` is pageable and goes out of scope
        ctx->cfo_mix_len = L;
        ctx->cfo_mix_fs = sample_rate;
    }
    auto launch = [&](float* d_x, size_t d_stride, size_t nb, const float* d_cfo) -> pu_status {
        (void)cudaGetLastError();
        pu::channel_cfo_kernel<<<static_cast<unsigned>((nb + 3) / 4), 128, 0, st>>>(d_x, d_stride, nb, static_cast<int>(L), d_cfo,
                                                                                   static_cast<double>(sample_rate), static_cast<const float2*>(ctx->cfo_mix.ptr));
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        return PU_OK;
    };
    if (space == PU_MEM_DEVICE) return launch(samples, stride, B, cfo_hz);
    pu::HostStage hs(ctx, st, B);
    float* d_x;
    const float* d_cfo;
    hs.inout(&d_x, samples, L, stride);
    hs.in(&d_cfo, cfo_hz, 1);
    return hs.run([&](size_t nb) { return launch(d_x, L, nb, d_cfo); });
}

pu_status pu_channel_apply_batch(pu_ctx* ctx, const pu_channel_config* cfg, const float* tx_pool, size_t pool_stride,
                                 size_t pool_count, const uint32_t* tx_index, const float* noise_std,
                                 const uint64_t* seed, size_t B, size_t L, float* rx, pu_memspace space, void* stream) {
    PU_REQUIRE(ctx && cfg, "pu_channel_apply_batch: NULL argument");
    if (B == 0 || L == 0) return PU_OK;
    PU_REQUIRE(tx_pool && noise_std && seed && rx, "pu_channel_apply_batch: NULL data pointer");
    PU_REQUIRE(pool_stride >= L && pool_count >= 1, "pu_channel_apply_batch: pool_stride < L or empty pool");
    PU_REQUIRE(L < (1u << 30), "pu_channel_apply_batch: frame too long");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const pu::ChannelParams p = pu::make_params(*cfg);
    const bool awgn_only = !p.fading && !(p.multipath && p.delay > 0) && p.noise;
    auto launch = [&](const float* d_pool, const uint32_t* d_idx, const float* d_std, const uint64_t* d_seed, size_t nb,
                      float* d_rx) -> pu_status {
        const unsigned blocks = static_cast<unsigned>((nb * 32 + 255) / 256);
        (void)cudaGetLastError();
        if (awgn_only) pu::awgn_kernel<<<blocks, 256, 0, st>>>(d_pool, pool_stride, d_idx, d_std, d_seed, nb, static_cast<int>(L), d_rx);
        else pu::channel_kernel<<<blocks, 256, 0, st>>>(p, d_pool, pool_stride, d_idx, d_std, d_seed, nb, static_cast<int>(L), d_rx);
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        return PU_OK;
    };
    if (space == PU_MEM_DEVICE) return launch(tx_pool, tx_index, noise_std, seed, B, rx);

    // host buffers: the indices come from outside the program, check them before any kernel reads the pool with them
    if (tx_index) for (size_t b = 0; b < B; ++b) PU_REQUIRE(tx_index[b] < pool_count, "pu_channel_apply_batch: tx_index out of range");
    pu::HostStage hs(ctx, st, B);
    const float *d_pool, *d_std;
    const uint32_t* d_idx;
    const uint64_t* d_seed;
    float* d_rx;
    hs.whole(&d_pool, tx_pool, pool_count * pool_stride);
    hs.in(&d_idx, tx_index, 1);
    hs.in(&d_std, noise_std, 1);
    hs.in(&d_seed, seed, 1);
    hs.out(&d_rx, rx, L);
    return hs.run([&](size_t nb) { return launch(d_pool, d_idx, d_std, d_seed, nb, d_rx); });
}

}  // extern "C"
