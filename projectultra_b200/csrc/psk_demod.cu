// projectultra_b200/csrc/psk_demod.cu — batched single-carrier and multi-carrier DPSK soft demodulators for sm_100a and
// the pu_dpsk_* / pu_mcdpsk_* entry points of the C ABI (externally timed frames: the Monte-Carlo sim knows where the
// data starts; Barker / chirp acquisition is SURVEY §8f next-2).
//
// Reference behaviour
//   DPSKDemodulator (src/psk/dpsk.hpp): carrier tables :311-323, correlateSymbol :777-787 (I += x cos, Q -= x sin,
//   sequential fp32 sums, / N), demodulateSoft :827-879 (diff = cur conj(prev), |diff|, atan2, optional CFO / initial
//   phase compensation :857-865, confidence = min(10 |diff|, 5)), phaseToBits :1002-1052, setReferenceSymbol :889-892.
//   MultiCarrierDPSKDemodulator (src/psk/multi_carrier_dpsk.hpp): demodulateOneSymbol :663-678 (per-carrier DFT bin
//   with std::polar(1, -phase), phase accumulated in fp32), processTraining :390-422, setReference :424-435,
//   demodulateSoft :437-472 (normalised differential, confidence = |cur| N_c 4, clamp +-10).
//
// Numerics: the correlations are SEQUENTIAL fp32 sums in the reference, so each (symbol[, carrier]) sum is one thread
// walking its samples in order with unfused multiply/add -- bit-identical; parallelism comes from the thousands of
// symbols in a batch.  Carrier / mixer tables are computed on the host with the host libm exactly as the reference
// computes them (MC-DPSK mixer phases reach 167 rad).  atan2f / sinf / cosf / hypotf are the restatements of
// ref_math.cuh.  Compiled with -fmad=false.
//
// Kernel shape: correlation = a warp owns 32 (symbol[, carrier]) sums; samples are staged through a padded shared
// tile with coalesced 128-byte row loads, 32 samples per row per round, so HBM sees each sample once (bound: HBM,
// 4 bytes and 4 flops per sample).  A second, tiny kernel turns neighbouring correlations into LLRs.
#include <cmath>
#include <complex>
#include <memory>
#include <new>
#include <vector>

#include "ofdm_dev.cuh"
#include "pu_async.cuh"
#include "pu_internal.h"

namespace pu {

std::vector<float> mcdpsk_carrier_freqs(const pu_mcdpsk_config& c);   // psk_tx.cpp

constexpr int kPskThreads = 128;
constexpr int kPskChunk = 32;

// ---------------------------------------------------------------------------------------------- single carrier
// corr[frame][s] for s in [0, n_corr): symbol s starts at sample first_start + s * sps.
__global__ void __launch_bounds__(kPskThreads) dpsk_correlate_kernel(const float* __restrict__ samples, size_t frame_stride,
                                                                     long first_start, int sps, int n_corr,
                                                                     const float* __restrict__ ccos, const float* __restrict__ csin,
                                                                     float2* __restrict__ corr, const int* __restrict__ frame_start,
                                                                     int has_ref, int L) {
    extern __shared__ float sm[];
    float* tcos = sm;                       // [sps]
    float* tsin = sm + sps;                 // [sps]
    float* tile = sm + 2 * sps;             // [warps][32][33]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < sps; i += blockDim.x) {
        tcos[i] = __ldg(&ccos[i]);
        tsin[i] = __ldg(&csin[i]);
    }
    __syncthreads();
    const size_t frame = blockIdx.y;
    // per-frame data start (acquired frames): symbols from frame_start[frame] (minus the reference symbol) to the end of the row
    const int n_all = n_corr;
    if (frame_start) {
        const int st = frame_start[frame];
        if (!(st > 0 && st < L)) return;                            // no preamble found: no symbols (tools/test_dpsk_snr.cpp:69)
        first_start = static_cast<long>(st) - has_ref * sps;
        n_corr = min(n_corr, (L - st) / sps + has_ref);
    }
    const float* x = samples + frame * frame_stride + first_start;
    const int s0 = (blockIdx.x * (kPskThreads / 32) + warp) * 32;   // first symbol of this warp
    if (s0 >= n_corr) return;
    float* wt = tile + warp * 32 * 33;
    const int s = s0 + lane;
    float I = 0.0f, Q = 0.0f;
    for (int c0 = 0; c0 < sps; c0 += kPskChunk) {
        const int cn = min(kPskChunk, sps - c0);
        __syncwarp();
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {                              // coalesced: row r = symbol s0 + r, 32 consecutive samples
            float v = 0.0f;
            if (s0 + r < n_corr && lane < cn) v = __ldg(&x[static_cast<size_t>(s0 + r) * sps + c0 + lane]);
            wt[r * 33 + lane] = v;
        }
        __syncwarp();
        for (int i = 0; i < cn; ++i) {                              // dpsk.hpp:781-784, in order, unfused
            const float xv = wt[lane * 33 + i];
            I = __fadd_rn(I, __fmul_rn(xv, tcos[c0 + i]));
            Q = __fsub_rn(Q, __fmul_rn(xv, tsin[c0 + i]));
        }
    }
    if (s < n_corr) corr[frame * n_all + s] = make_float2(__fdiv_rn(I, static_cast<float>(sps)), __fdiv_rn(Q, static_cast<float>(sps)));
}

__device__ __forceinline__ float wrap_0_2pi(float phase) {   // while (phase < 0) phase += 2 pi; while (phase >= 2 pi) phase -= 2 pi
    const double two_pi = 2.0f * 3.14159265358979323846;
    while (phase < 0.0f) phase = static_cast<float>(__dadd_rn(static_cast<double>(phase), two_pi));
    while (static_cast<double>(phase) >= two_pi) phase = static_cast<float>(__dsub_rn(static_cast<double>(phase), two_pi));
    return phase;
}

__global__ void dpsk_llr_kernel(const float2* __restrict__ corr, int n_corr, int has_ref, int n_sym, int mod, int sps, float sample_rate,
                                const float* __restrict__ est_cfo, const float* __restrict__ phase_off, size_t B,
                                float* __restrict__ llr, size_t llr_stride, const int* __restrict__ frame_start, int L,
                                int* __restrict__ n_llr) {
    const size_t g = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (g >= B * static_cast<size_t>(n_sym)) return;
    const size_t frame = g / n_sym;
    const int s = static_cast<int>(g - frame * n_sym);
    if (frame_start) {
        const int st = frame_start[frame];
        const int mine = (st > 0 && st < L) ? (L - st) / sps : 0;
        if (s == 0 && n_llr) n_llr[frame] = static_cast<int>(min(static_cast<size_t>(mine) * (mod + 1), llr_stride));
        if (s >= mine) return;
    }
    const float2* c = corr + frame * n_corr + has_ref;
    const float2 cur = c[s];
    const float2 prev = (s > 0 || has_ref) ? c[s - 1] : make_float2(1.0f, 0.0f);   // prev_symbol_ (:840, :889-892)
    const float2 df = cmul(cur, cconj(prev));                                       // :848
    const float magnitude = cabs_ref(df);                                           // :851
    float phase = refmath::atan2f_ref(df.y, df.x);                                  // :854
    const float cfo = est_cfo ? est_cfo[frame] : 0.0f, poff = phase_off ? phase_off[frame] : 0.0f;
    if (fabsf(cfo) > 0.5f || fabsf(poff) > 0.01f) {                                 // :857-865
        const double two_pi = 2.0f * 3.14159265358979323846, pi = 3.14159265358979323846;
        const float cfo_phase = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(two_pi, static_cast<double>(cfo)), static_cast<double>(sps)),
                                                             static_cast<double>(sample_rate)));
        phase = __fsub_rn(phase, cfo_phase);
        phase = __fsub_rn(phase, poff);
        while (static_cast<double>(phase) > pi) phase = static_cast<float>(__dsub_rn(static_cast<double>(phase), two_pi));
        while (static_cast<double>(phase) < -pi) phase = static_cast<float>(__dadd_rn(static_cast<double>(phase), two_pi));
    }
    const float confidence = fminf(__fmul_rn(magnitude, 10.0f), 5.0f);              // :868
    phase = wrap_0_2pi(phase);                                                      // phaseToBits :1006-1007
    const int bps = mod + 1;
    float l[3];
    if (mod == 0) {
        l[0] = __fmul_rn(confidence, refmath::cosf_ref(phase));
    } else {
        l[0] = __fmul_rn(confidence, refmath::sinf_ref(phase));
        l[1] = __fmul_rn(confidence, refmath::sinf_ref(__fmul_rn(2.0f, phase)));
        if (mod == 2) l[2] = __fmul_rn(confidence, refmath::sinf_ref(__fmul_rn(4.0f, phase)));
    }
    float* out = llr + frame * llr_stride;
    for (int b = 0; b < bps; ++b) {
        const size_t pos = static_cast<size_t>(s) * bps + b;
        if (pos < llr_stride) out[pos] = l[b];
    }
}

// ---------------------------------------------------------------------------------------------- Barker-13 acquisition
// DPSKDemodulator::findPreamble (src/psk/dpsk.hpp:338-481) for B frames, one frame per CTA (SURVEY §8f next-2, DPSK half):
// energy gate, coarse search at one-symbol steps, fine search at one-sample steps around the best coarse position
// (computeDifferentialScore :489-546), threshold + global-outlier tests, estimateCFOTolerant (:550-593),
// refineTimingWithMatchedFilter (:708-771, only when |cfo| < 0.5 Hz), estimateInitialPhaseOffset (:659-704).
// Every ordered sum of the reference is an ordered sum here (one thread per sum); what is parallel is what the reference
// computes independently: the symbol correlations at different offsets, the scores of different start positions, the
// matched-filter candidates.  The symbol correlation at sample offset o is shared by every start r = o - s * sps, so the fine
// search evaluates 40 * sps correlations once (shared memory) instead of 2 * sps * 39.
constexpr int kBkSyms = 39, kBkDiffs = 38, kBkThreads = 512;
__constant__ int kBarker13[13] = {1, 1, 1, 1, 1, -1, -1, 1, 1, -1, 1, -1, 1};
__device__ __forceinline__ int bk_pattern(int i) { return kBarker13[(i + 1) % 13]; }   // expected_pattern[i] = BARKER13[(i + 1) % 13]

// correlateSymbol (:777-787) of the sps samples at x
__device__ __forceinline__ float2 bk_correlate(const float* __restrict__ x, int sps, const float* tcos, const float* tsin) {
    float I = 0.0f, Q = 0.0f;
    for (int i = 0; i < sps; ++i) {
        const float v = x[i];
        I = __fadd_rn(I, __fmul_rn(v, tcos[i]));
        Q = __fsub_rn(Q, __fmul_rn(v, tsin[i]));
    }
    return make_float2(__fdiv_rn(I, static_cast<float>(sps)), __fdiv_rn(Q, static_cast<float>(sps)));
}

// computeDifferentialScore from the symbol correlations c[0], c[stride], ... (:496-545)
__device__ float bk_score(const float2* c, int stride) {
    float total_energy = 0.0f;
    for (int s = 0; s < kBkSyms; ++s) total_energy = __fadd_rn(total_energy, cnorm(c[s * stride]));
    if (total_energy < __fmul_rn(0.001f, static_cast<float>(kBkSyms))) return 0.0f;
    float2 sum = make_float2(0.0f, 0.0f);
    float magnitude_sum = 0.0f;
    for (int i = 0; i < kBkDiffs; ++i) {
        const float2 diff = cmul(c[(i + 1) * stride], cconj(c[i * stride]));
        const float magnitude = cabs_ref(diff);
        if (magnitude < 1e-10f) continue;
        const float2 dn = make_float2(__fdiv_rn(diff.x, magnitude), __fdiv_rn(diff.y, magnitude));
        sum = cadd(sum, cmul(dn, make_float2(static_cast<float>(bk_pattern(i)), -0.0f)));   // diff_norm * conj(Complex(expected, 0))
        magnitude_sum = __fadd_rn(magnitude_sum, magnitude);
    }
    if (magnitude_sum < 1e-10f) return 0.0f;
    return __fdiv_rn(cabs_ref(sum), static_cast<float>(kBkDiffs));
}

struct BkShared {
    float scores[kBkThreads * 2];   // coarse (<= 4 * 39) then fine (<= 2 * sps) scores
    float2 c0[4 * kBkSyms + kBkSyms + 4];
    float best_score, global_avg, cfo, rms;
    int best_offset, fine_start, fine_end, result;
    float red_c[kBkThreads / 32];
    int red_i[kBkThreads / 32];
    float2 ph[12];
};

__global__ void __launch_bounds__(kBkThreads) dpsk_find_preamble_kernel(const float* __restrict__ samples, size_t frame_stride, int L, int sps,
                                                                        float fs, const float* __restrict__ ccos, const float* __restrict__ csin,
                                                                        const float* __restrict__ mf_template, float mf_energy,
                                                                        int* __restrict__ out_start, float* __restrict__ out_cfo,
                                                                        float* __restrict__ out_phase) {
    extern __shared__ __align__(16) unsigned char bk_smem[];
    float* tcos = reinterpret_cast<float*>(bk_smem);                 // [sps]
    float* tsin = tcos + sps;                                        // [sps]
    float2* C = reinterpret_cast<float2*>(tsin + sps);               // [40 * sps] fine correlations; later the matched-filter template
    __shared__ BkShared S;
    const int tid = threadIdx.x, T = blockDim.x;
    const float* x = samples + static_cast<size_t>(blockIdx.x) * frame_stride;
    const int preamble = kBkSyms * sps;
    for (int i = tid; i < sps; i += T) { tcos[i] = __ldg(&ccos[i]); tsin[i] = __ldg(&csin[i]); }
    if (tid == 0) { S.result = -1; S.cfo = 0.0f; S.best_offset = -1; S.best_score = 0.0f; }
    __syncthreads();
    bool alive = L >= preamble + preamble / 2;                        // :354-355
    const int max_search = min(L - preamble, preamble * 4);           // :393
    const int n_starts = alive ? (max_search + sps - 1) / sps : 0;    // coarse positions 0, sps, ... < max_search
    // ---- coarse symbol correlations (all threads), then the energy gate (:359-368): ONE ordered sum over up to 2 preambles of samples.
    // Read by its thread straight from global memory it was the kernel: ~30 000 dependent load-multiply-adds with a handful of loads
    // in flight (the v34 capture: issue-active 32 %, every other warp at the barrier).  Now all threads stage 2 048-sample chunks into
    // shared memory with cp.async, one chunk ahead, and thread 0 sums from there at the add latency.
    if (alive) {
        for (int m = tid; m < n_starts + kBkDiffs; m += T) S.c0[m] = bk_correlate(x + m * sps, sps, tcos, tsin);
        constexpr int CH = 2048;
        float* stg = reinterpret_cast<float*>(C);                     // [2][CH]: the fine correlations' storage is idle until later
        const int check = min(L, preamble * 2), nch = (check + CH - 1) / CH;
        auto fetch = [&](int k, int buf) {
            for (int j = tid; j < CH; j += T)
                if (k * CH + j < check) cp_async4(smem_u32(stg + buf * CH + j), x + k * CH + j);
            cp_async_commit();
        };
        float energy = 0.0f;
        fetch(0, 0);
        for (int k = 0; k < nch; ++k) {
            if (k + 1 < nch) fetch(k + 1, (k + 1) & 1); else cp_async_commit();
            cp_async_wait_but_one();
            __syncthreads();
            if (tid == 0) {
                const float* pch = stg + (k & 1) * CH;
                const int cnt = min(CH, check - k * CH);
#pragma unroll 8
                for (int i = 0; i < cnt; ++i) energy = __fadd_rn(energy, __fmul_rn(pch[i], pch[i]));
            }
            __syncthreads();                                          // the chunk is fetched again two steps on
        }
        if (tid == 0) S.rms = __fsqrt_rn(__fdiv_rn(energy, static_cast<float>(check)));
    }
    __syncthreads();
    alive = alive && !(S.rms < 0.01f);
    if (alive) {
        for (int m = tid; m < n_starts; m += T) S.scores[m] = bk_score(S.c0 + m, 1);
        __syncthreads();
        if (tid == 0) {                                               // :403-414, in order
            float best = 0.0f, sum = 0.0f;
            int bo = -1;
            for (int m = 0; m < n_starts; ++m) {
                const float sc = S.scores[m];
                sum = __fadd_rn(sum, sc);
                if (sc > best) { best = sc; bo = m * sps; }
            }
            S.best_score = best;
            S.best_offset = bo;
            S.global_avg = n_starts > 0 ? __fdiv_rn(sum, static_cast<float>(n_starts)) : 0.0f;
            S.fine_start = max(0, bo - sps);
            S.fine_end = min(max_search, bo + sps);
        }
        __syncthreads();
        const bool fine = S.best_offset >= 0 && S.best_score > __fmul_rn(0.80f, 0.7f);   // :417
        if (fine) {
            const int f0 = S.fine_start, n_fine = S.fine_end - S.fine_start;
            const int n_off = n_fine + kBkDiffs * sps;
            for (int o = tid; o < n_off; o += T) C[o] = bk_correlate(x + f0 + o, sps, tcos, tsin);
            __syncthreads();
            for (int r = tid; r < n_fine; r += T) S.scores[r] = bk_score(C + r, sps);
            __syncthreads();
            if (tid == 0) {                                           // :421-428, in order
                float best = S.best_score;
                int bo = S.best_offset;
                for (int r = 0; r < n_fine; ++r)
                    if (S.scores[r] > best) { best = S.scores[r]; bo = f0 + r; }
                S.best_score = best;
                S.best_offset = bo;
            }
            __syncthreads();
        }
        alive = fine && !(S.best_score < 0.80f) && !(S.global_avg > 0.0f && S.best_score < __fmul_rn(S.global_avg, 1.3f));   // :434-448
    }
    if (alive) {
        // ---- estimateCFOTolerant(best_offset) from the correlations the fine search left in C (:550-593)
        if (tid == 0) {
            const float2* c = C + (S.best_offset - S.fine_start);
            float2 corr = make_float2(0.0f, 0.0f);
            int nd = 0;
            float2 prev = make_float2(0.0f, 0.0f);
            for (int s = 0; s <= kBkDiffs; ++s) {
                const float2 cur = c[s * sps];
                if (s > 0 && cabs_ref(prev) > 0.01f && cabs_ref(cur) > 0.01f) {
                    float2 d = cmul(cur, cconj(prev));
                    const float m = cabs_ref(d);
                    d = make_float2(__fdiv_rn(d.x, m), __fdiv_rn(d.y, m));
                    // diffs are compacted and paired with expected_pattern[position in the list] (:575-579)
                    corr = cadd(corr, cmul(d, make_float2(static_cast<float>(bk_pattern(nd)), -0.0f)));
                    ++nd;
                }
                prev = cur;
            }
            float cfo = 0.0f;
            if (nd >= 10) {
                const float phase_offset = refmath::atan2f_ref(corr.y, corr.x);
                const float symbol_duration = __fdiv_rn(static_cast<float>(sps), fs);
                cfo = -static_cast<float>(__ddiv_rn(static_cast<double>(phase_offset),
                                                    __dmul_rn(2.0f * 3.14159265358979323846, static_cast<double>(symbol_duration))));
            }
            S.cfo = cfo;
        }
        __syncthreads();
        // ---- refineTimingWithMatchedFilter(best_offset, cfo_hz = 0) when |cfo| < 0.5 (:457-461, :708-771)
        if (fabsf(S.cfo) < 0.5f) {
            const int n = 6 * sps;
            float* tm = reinterpret_cast<float*>(C);
            for (int j = tid; j < n; j += T) tm[j] = __ldg(&mf_template[j]);
            __syncthreads();
            const int coarse = S.best_offset;
            const int fs2 = max(0, coarse - sps), fe2 = min(L - n, coarse + sps);
            float bc = -1.0f;
            int bi = coarse;
            for (int i = fs2 + tid; i <= fe2; i += T) {
                const float* r = x + i;
                float corr = 0.0f, sig = 0.0f;
                for (int j = 0; j < n; ++j) {
                    const float v = r[j];
                    corr = __fadd_rn(corr, __fmul_rn(v, tm[j]));
                    sig = __fadd_rn(sig, __fmul_rn(v, v));
                }
                const float norm = __fsqrt_rn(__fmul_rn(sig, mf_energy));
                if (norm < 1e-10f) continue;
                const float nc = __fdiv_rn(fabsf(corr), norm);
                if (nc > bc) { bc = nc; bi = i; }
            }
            // first maximum in ascending i: larger value wins, equal value -> smaller index; threads without a candidate hold -1
            for (int o = 16; o > 0; o >>= 1) {
                const float oc = __shfl_xor_sync(0xffffffffu, bc, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (oc > bc || (oc == bc && oc >= 0.0f && oi < bi)) { bc = oc; bi = oi; }
            }
            if ((tid & 31) == 0) { S.red_c[tid >> 5] = bc; S.red_i[tid >> 5] = bi; }
            __syncthreads();
            if (tid == 0) {
                for (int w = 1; w < T / 32; ++w)
                    if (S.red_c[w] > bc || (S.red_c[w] == bc && bc >= 0.0f && S.red_i[w] < bi)) { bc = S.red_c[w]; bi = S.red_i[w]; }
                S.best_offset = bc >= 0.0f ? bi : coarse;
            }
            __syncthreads();
        }
        // ---- estimateInitialPhaseOffset(best_offset) (:659-704): 11 symbol correlations at the final position
        const int bo = S.best_offset;
        if (tid < 11 && bo + tid * sps + sps <= L) S.ph[tid] = bk_correlate(x + bo + tid * sps, sps, tcos, tsin);
        __syncthreads();
        if (tid == 0) {
            const double two_pi = 2.0f * 3.14159265358979323846, pi = 3.14159265358979323846;
            float sum = 0.0f;
            int ne = 0;
            float2 prev = make_float2(0.0f, 0.0f);
            for (int s = 0; s <= 10 && s < kBkDiffs; ++s) {
                if (bo + s * sps + sps > L) break;
                const float2 cur = S.ph[s];
                if (s > 0 && cabs_ref(prev) > 0.01f && cabs_ref(cur) > 0.01f) {
                    const float2 d = cmul(cur, cconj(prev));
                    float measured = refmath::atan2f_ref(d.y, d.x);
                    const float expected = bk_pattern(s - 1) > 0 ? 0.0f : static_cast<float>(pi);
                    const float cfo_phase = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(two_pi, static_cast<double>(S.cfo)), static_cast<double>(sps)),
                                                                         static_cast<double>(fs)));
                    measured = __fsub_rn(measured, cfo_phase);
                    float error = __fsub_rn(measured, expected);
                    while (static_cast<double>(error) > pi) error = static_cast<float>(__dsub_rn(static_cast<double>(error), two_pi));
                    while (static_cast<double>(error) < -pi) error = static_cast<float>(__dadd_rn(static_cast<double>(error), two_pi));
                    sum = __fadd_rn(sum, error);   // the reference sums the list afterwards, in the same order
                    ++ne;
                }
                prev = cur;
            }
            out_phase[blockIdx.x] = ne ? __fdiv_rn(sum, static_cast<float>(ne)) : 0.0f;
            out_cfo[blockIdx.x] = S.cfo;
            out_start[blockIdx.x] = bo + preamble;
        }
    } else if (tid == 0) {
        out_start[blockIdx.x] = -1;
        out_cfo[blockIdx.x] = 0.0f;
        out_phase[blockIdx.x] = 0.0f;
    }
}

// ---------------------------------------------------------------------------------------------- multi carrier
// corr[frame][sym][c]: pair index t = sym * nc + c; a CTA owns kPskThreads consecutive pairs of one frame.
__global__ void __launch_bounds__(kPskThreads) mcdpsk_correlate_kernel(const float* __restrict__ samples, size_t frame_stride, int sps,
                                                                       int nc, int n_sym, const float2* __restrict__ mixer,
                                                                       float2* __restrict__ corr) {
    extern __shared__ float sm[];            // tile [rows][33]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t frame = blockIdx.y;
    const float* x = samples + frame * frame_stride;
    const int n_pairs = n_sym * nc;
    const int t0 = blockIdx.x * kPskThreads;
    const int t = t0 + tid;
    const bool live = t < n_pairs;
    const int sym_lo = t0 / nc;
    const int sym_hi = min(n_sym - 1, (min(t0 + kPskThreads, n_pairs) - 1) / nc);
    const int rows = sym_hi - sym_lo + 1;
    const int sym = live ? t / nc : sym_lo, c = live ? t - sym * nc : 0;
    const float2* mx = mixer + static_cast<size_t>(c) * sps;
    const int row = sym - sym_lo;
    float sr = 0.0f, si = 0.0f;
    for (int c0 = 0; c0 < sps; c0 += kPskChunk) {
        const int cn = min(kPskChunk, sps - c0);
        __syncthreads();
        for (int r = warp; r < rows; r += kPskThreads / 32)
            sm[r * 33 + lane] = (lane < cn) ? __ldg(&x[static_cast<size_t>(sym_lo + r) * sps + c0 + lane]) : 0.0f;
        __syncthreads();
        for (int i = 0; i < cn; ++i) {                               // multi_carrier_dpsk.hpp:671-675, in order, unfused
            const float xv = sm[row * 33 + i];
            const float2 m = __ldg(&mx[c0 + i]);
            sr = __fadd_rn(sr, __fmul_rn(m.x, xv));
            si = __fadd_rn(si, __fmul_rn(m.y, xv));
        }
    }
    if (live) corr[frame * n_pairs + t] = make_float2(__fdiv_rn(sr, static_cast<float>(sps)), __fdiv_rn(si, static_cast<float>(sps)));
}

__global__ void mcdpsk_llr_kernel(const float2* __restrict__ corr, int nc, int n_sym, int training, int bits, int sps, float sample_rate,
                                  const float2* __restrict__ expected_diff, size_t B, float* __restrict__ llr, size_t llr_stride,
                                  float* __restrict__ residual_cfo) {
    const int n_data = n_sym - training - 1;
    const size_t per_frame = static_cast<size_t>(n_data > 0 ? n_data : 0) * nc;
    const size_t g = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (residual_cfo && g < B) {                                     // processTraining (:390-422), one thread per frame
        const float2* c0 = corr + g * static_cast<size_t>(n_sym) * nc;
        float cfo = 0.0f;
        if (training >= 2) {
            float sum = 0.0f;
            for (int c = 0; c < nc; ++c) {
                const float2 actual = cmul(c0[nc + c], cconj(c0[c]));
                const float2 err = cmul(actual, cconj(expected_diff[c]));
                sum = __fadd_rn(sum, refmath::atan2f_ref(err.y, err.x));
            }
            const float avg = __fdiv_rn(sum, static_cast<float>(nc));
            const float symbol_duration = __fdiv_rn(static_cast<float>(sps), sample_rate);
            cfo = static_cast<float>(__ddiv_rn(static_cast<double>(avg), __dmul_rn(2.0f * 3.14159265358979323846, static_cast<double>(symbol_duration))));
            cfo = fmaxf(-50.0f, fminf(50.0f, __fadd_rn(0.0f, cfo)));   // cfo_hz_ += residual, clamped (:420-421)
        }
        residual_cfo[g] = cfo;
    }
    if (g >= B * per_frame) return;
    const size_t frame = g / per_frame;
    const int t = static_cast<int>(g - frame * per_frame);
    const int sd = t / nc, c = t - sd * nc;
    const float2* cf = corr + frame * static_cast<size_t>(n_sym) * nc;
    const float2 cur = cf[(training + 1 + sd) * nc + c];
    const float2 pv = cf[(training + sd) * nc + c];                  // previous data symbol, or the reference symbol for sd == 0
    const float pmag = cabs_ref(pv);
    const float pthr = sd == 0 ? 0.001f : 0.0001f;                   // setReference (:430) vs demodulateSoft (:448)
    const float2 prev = pmag > pthr ? cdivs(pv, pmag) : make_float2(1.0f, 0.0f);
    const float mag = cabs_ref(cur);
    const float2 nrm = mag > 0.0001f ? cdivs(cur, mag) : make_float2(1.0f, 0.0f);
    const float2 df = cmul(nrm, cconj(prev));
    float phase = refmath::atan2f_ref(df.y, df.x);
    const float confidence = __fmul_rn(__fmul_rn(mag, static_cast<float>(nc)), 4.0f);
    phase = wrap_0_2pi(phase);
    float* out = llr + frame * llr_stride;
    const size_t base = static_cast<size_t>(t) * bits;
    if (bits == 2) {
        const float sb0 = __fmul_rn(confidence, refmath::sinf_ref(phase));
        const float sb1 = __fmul_rn(confidence, refmath::sinf_ref(__fmul_rn(2.0f, phase)));
        if (base < llr_stride) out[base] = fmaxf(-10.0f, fminf(10.0f, sb0));
        if (base + 1 < llr_stride) out[base + 1] = fmaxf(-10.0f, fminf(10.0f, sb1));
    } else {
        const float sb = __fmul_rn(confidence, refmath::cosf_ref(phase));
        if (base < llr_stride) out[base] = fmaxf(-10.0f, fminf(10.0f, sb));
    }
}

// ---------------------------------------------------------------------------------------------- MC-DPSK CFO correction
// MultiCarrierDPSKDemodulator::applyCFOCorrection (multi_carrier_dpsk.hpp:633-658) on whole frames, as processGotChirp applies it
// when |cfo| > 0.1 Hz (:565-569): analytic signal by the 127-tap Blackman-windowed Hilbert FIR (HilbertTransform::process,
// src/dsp/filters.cpp:293-317: Q = ordered 127-tap sum over the delay line, I = the input delayed by 63 samples, delay line
// zero-filled before the frame), multiplied by e^{j phase} with the per-sample phase recurrence phase += inc (one wrap test
// per sample), real part kept.  One frame per CTA; the phase recurrence is walked T samples at a time with the bit-for-bit link
// check of ofdm_demod.cu (every accepted value is the reference's by induction); everything else is independent per sample.
constexpr int kHilbertTaps = 127, kCfoThreads = 256;
struct HilbertTaps { float c[kHilbertTaps]; };

__global__ void __launch_bounds__(kCfoThreads) mcdpsk_cfo_correct_kernel(HilbertTaps taps, const float* __restrict__ in, size_t stride, int L,
                                                                          float fs, const float* __restrict__ cfo_hz,
                                                                          float* __restrict__ out, const int* __restrict__ frame_start) {
    __shared__ int fail[kCfoThreads / 32];
    __shared__ float next_phase;
    const int tid = threadIdx.x, T = blockDim.x;
    // optional per-frame window (frames located by the chirp): the span [start, row end) is moved to the front of the output row
    // and the rest of the row is cleared; start < 0 or beyond the row = no frame
    const int Lrow = L;
    int start = frame_start ? frame_start[blockIdx.x] : 0;
    if (start < 0 || start > Lrow) start = Lrow;
    const float* x = in + static_cast<size_t>(blockIdx.x) * stride + start;
    float* y = out + static_cast<size_t>(blockIdx.x) * stride;
    L = Lrow - start;
    for (int i = L + tid; i < Lrow; i += T) y[i] = 0.0f;
    const float cfo = cfo_hz[blockIdx.x];
    if (!(fabsf(cfo) > 0.1f) || fabsf(cfo) < 0.01f || L < 128) {         // processGotChirp :565, applyCFOCorrection :634
        for (int i = tid; i < L; i += T) y[i] = x[i];
        return;
    }
    const double pi = 3.14159265358979323846;
    const float inc = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(-2.0f, pi), static_cast<double>(cfo)), static_cast<double>(fs)));
    auto step = [&](float ph) {
        ph = __fadd_rn(ph, inc);
        if (static_cast<double>(ph) > pi) ph = static_cast<float>(__dsub_rn(static_cast<double>(ph), __dmul_rn(2.0f, pi)));
        if (static_cast<double>(ph) < -pi) ph = static_cast<float>(__dadd_rn(static_cast<double>(ph), __dmul_rn(2.0f, pi)));
        return ph;
    };
    float ph = 0.0f;                                                       // cfo_initial_phase_ of a fresh demodulator
    for (int i0 = 0; i0 < L;) {
        const unsigned b0 = __float_as_uint(ph);
        const unsigned delta = __float_as_uint(step(ph)) - b0;
        const float cand = __uint_as_float(b0 + static_cast<unsigned>(tid) * delta);
        const float nxt = step(cand);
        const bool broken = __float_as_uint(nxt) != b0 + static_cast<unsigned>(tid + 1) * delta;
        const unsigned bal = __ballot_sync(0xffffffffu, broken);
        if ((tid & 31) == 0) fail[tid >> 5] = bal ? (tid + __ffs(bal) - 1) : T;
        __syncthreads();
        int f = T;
        for (int w = 0; w < T / 32; ++w) f = min(f, fail[w]);
        const int nvalid = min(f < T ? f + 1 : T, L - i0);
        if (tid == nvalid - 1) next_phase = nxt;
        if (tid < nvalid) {
            const int i = i0 + tid;
            float q = 0.0f;                                                // ordered: coeffs[0] * x[i], coeffs[1] * x[i-1], ...
#pragma unroll 1
            for (int k = 0; k < kHilbertTaps; ++k) q = __fadd_rn(q, __fmul_rn(taps.c[k], i - k >= 0 ? x[i - k] : 0.0f));
            const float re = i >= 63 ? x[i - 63] : 0.0f;                   // delay_samples_ = 63
            float sn, cs;
            sn = refmath::sinf_ref(cand);
            cs = refmath::cosf_ref(cand);
            y[i] = __fsub_rn(__fmul_rn(re, cs), __fmul_rn(q, sn));         // (analytic[i] * rotation).real()
        }
        __syncthreads();
        ph = next_phase;
        i0 += nvalid;
    }
}

}  // namespace pu

#include "psk_handles.h"

extern "C" {

pu_status pu_dpsk_create(pu_ctx* ctx, const pu_dpsk_config* cfg, pu_dpsk** out) {
    PU_REQUIRE(ctx && cfg && out, "pu_dpsk_create: NULL argument");
    *out = nullptr;
    if (cfg->samples_per_symbol == 0 || cfg->samples_per_symbol > 8192 || cfg->modulation > 2 || !(cfg->sample_rate > 0)) {
        pu::set_error("pu_dpsk_create: samples_per_symbol must be in [1, 8192], modulation 0..2 (DBPSK/DQPSK/D8PSK)");
        return PU_ERR_UNSUPPORTED;
    }
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    std::unique_ptr<pu_dpsk> h(new (std::nothrow) pu_dpsk());
    if (!h) return PU_ERR_NOMEM;
    h->ctx = ctx;
    h->device = ctx->device;
    h->cfg = *cfg;
    const int n = static_cast<int>(cfg->samples_per_symbol);
    std::vector<float> cs(n), sn(n);
    const float inc = static_cast<float>(2.0f * 3.14159265358979323846 * cfg->carrier_freq / cfg->sample_rate);   // dpsk.hpp:315
    for (int i = 0; i < n; ++i) {
        const float phase = inc * i;
        sn[i] = std::sin(phase);
        cs[i] = std::cos(phase);
    }
    pu_status s;
    if ((s = h->d_cos.upload(cs.data(), cs.size())) != PU_OK) return s;
    if ((s = h->d_sin.upload(sn.data(), sn.size())) != PU_OK) return s;
    {   // refineTimingWithMatchedFilter's template for cfo_hz = 0 (dpsk.hpp:712-735)
        static const int barker[6] = {1, 1, 1, 1, 1, -1};
        std::vector<float> tm;
        tm.reserve(static_cast<size_t>(6) * n);
        const float adjusted = cfg->carrier_freq + 0.0f;
        const float carrier_inc = static_cast<float>(2.0f * 3.14159265358979323846 * adjusted / cfg->sample_rate);
        float phase = 0.0f, symbol_phase = 0.0f;
        for (int sy = 0; sy < 6; ++sy) {
            if (barker[sy] < 0) symbol_phase = static_cast<float>(symbol_phase + 3.14159265358979323846);
            for (int i = 0; i < n; ++i) {
                tm.push_back(std::cos(phase + symbol_phase));
                phase += carrier_inc;
                if (phase > 2.0f * 3.14159265358979323846) phase = static_cast<float>(phase - 2.0f * 3.14159265358979323846);
            }
        }
        float e = 0.0f;
        for (float t : tm) e += t * t;
        h->mf_energy = e;
        if ((s = h->d_mf.upload(tm.data(), tm.size())) != PU_OK) return s;
    }
    *out = h.release();
    return PU_OK;
}

static pu_status dpsk_launch(pu_dpsk* h, const float* d_samples, size_t B, size_t L, size_t data_start, int ref_mode,
                             const float* d_cfo, const float* d_poff, float* d_llr, size_t llr_stride, cudaStream_t st,
                             const int* d_fstart, int* d_nllr);

static pu_status dpsk_find_launch(pu_dpsk* h, const float* d_samples, size_t B, size_t L, int* d_start, float* d_cfo, float* d_phase,
                                  cudaStream_t st) {
    const int sps = static_cast<int>(h->cfg.samples_per_symbol);
    if (sps > 512) {
        pu::set_error("pu_dpsk_find_preamble_batch: samples_per_symbol > 512 is not supported (shared-memory budget of the fine search)");
        return PU_ERR_UNSUPPORTED;
    }
    const size_t smem = sizeof(float) * (2 * static_cast<size_t>(sps) + std::max<size_t>(2 * 40 * static_cast<size_t>(sps), 4096));   // (4096: the energy gate's staging chunks)
    (void)cudaGetLastError();
    cudaFuncSetAttribute(pu::dpsk_find_preamble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    pu::dpsk_find_preamble_kernel<<<static_cast<unsigned>(B), pu::kBkThreads, smem, st>>>(
        d_samples, L, static_cast<int>(L), sps, h->cfg.sample_rate, static_cast<const float*>(h->d_cos.p), static_cast<const float*>(h->d_sin.p),
        static_cast<const float*>(h->d_mf.p), h->mf_energy, d_start, d_cfo, d_phase);
    h->ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_dpsk_receive_batch(pu_dpsk* h, const float* samples, size_t B, size_t L, float* llr_out, size_t llr_stride, int32_t* n_llr,
                                int32_t* data_start, float* est_cfo_hz, float* phase_offset, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_dpsk_receive_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && data_start && est_cfo_hz && phase_offset, "pu_dpsk_receive_batch: NULL data pointer");
    PU_REQUIRE(L < (1u << 30), "pu_dpsk_receive_batch: frame too long");
    PU_REQUIRE(!llr_out || (llr_stride > 0 && n_llr), "pu_dpsk_receive_batch: llr_out needs llr_stride and n_llr");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const int sps = static_cast<int>(h->cfg.samples_per_symbol);
    pu_status s;
    if (space == PU_MEM_DEVICE) {
        if ((s = dpsk_find_launch(h, samples, B, L, data_start, est_cfo_hz, phase_offset, st)) != PU_OK) return s;
        if (!llr_out || L <= static_cast<size_t>(39) * sps) return PU_OK;
        return dpsk_launch(h, samples, B, L, static_cast<size_t>(39) * sps, 1, est_cfo_hz, phase_offset, llr_out, llr_stride, st, data_start, n_llr);
    }
    pu::HostStage hs(ctx, st, B);
    const float* d_x;
    float *d_llr, *d_cfo, *d_phase;
    int32_t *d_n, *d_start;
    hs.in(&d_x, samples, L);
    hs.out(&d_llr, llr_out, llr_stride);
    hs.out(&d_n, llr_out ? n_llr : nullptr, 1);
    hs.out(&d_start, data_start, 1);
    hs.out(&d_cfo, est_cfo_hz, 1);
    hs.out(&d_phase, phase_offset, 1);
    return hs.run([&](size_t nb) {
        return pu_dpsk_receive_batch(h, d_x, nb, L, d_llr, llr_stride, d_n, d_start, d_cfo, d_phase, PU_MEM_DEVICE, st);
    });
}

void pu_dpsk_destroy(pu_dpsk* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    h->corr.release();
    delete h;
}

int pu_dpsk_bits_per_symbol(const pu_dpsk* h) { return h ? static_cast<int>(h->cfg.modulation) + 1 : -1; }

static pu_status dpsk_launch(pu_dpsk* h, const float* d_samples, size_t B, size_t L, size_t data_start, int ref_mode,
                             const float* d_cfo, const float* d_poff, float* d_llr, size_t llr_stride, cudaStream_t st,
                             const int* d_fstart, int* d_nllr) {
    const int sps = static_cast<int>(h->cfg.samples_per_symbol);
    // with per-frame starts data_start is the smallest possible start (one preamble), which bounds the symbol count
    const int has_ref = (ref_mode == 1 && data_start >= static_cast<size_t>(sps)) ? 1 : 0;
    const int n_sym = static_cast<int>((L - data_start) / sps);
    if (n_sym == 0) return PU_OK;
    const int n_corr = n_sym + has_ref;
    pu_status s;
    if ((s = h->corr.reserve(B * static_cast<size_t>(n_corr) * sizeof(float2))) != PU_OK) return s;
    float2* corr = static_cast<float2*>(h->corr.ptr);
    const size_t smem = sizeof(float) * (2 * static_cast<size_t>(sps) + (pu::kPskThreads / 32) * 32 * 33);
    (void)cudaGetLastError();
    if (smem > 48 * 1024) cudaFuncSetAttribute(pu::dpsk_correlate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    const size_t kMaxY = 65535;
    for (size_t off = 0; off < B; off += kMaxY) {
        const size_t nb = std::min(kMaxY, B - off);
        const dim3 grid(static_cast<unsigned>((n_corr + pu::kPskThreads - 1) / pu::kPskThreads), static_cast<unsigned>(nb));
        pu::dpsk_correlate_kernel<<<grid, pu::kPskThreads, smem, st>>>(d_samples + off * L, L, static_cast<long>(data_start) - has_ref * sps, sps,
                                                                     n_corr, static_cast<const float*>(h->d_cos.p),
                                                                     static_cast<const float*>(h->d_sin.p), corr + off * n_corr,
                                                                     d_fstart ? d_fstart + off : nullptr, has_ref, static_cast<int>(L));
        h->ctx->launches.fetch_add(1);
    }
    const size_t total = B * static_cast<size_t>(n_sym);
    pu::dpsk_llr_kernel<<<static_cast<unsigned>((total + 127) / 128), 128, 0, st>>>(corr, n_corr, has_ref, n_sym, static_cast<int>(h->cfg.modulation),
                                                                                  sps, h->cfg.sample_rate, d_cfo, d_poff, B, d_llr, llr_stride, d_fstart,
                                                                                  static_cast<int>(L), d_nllr);
    h->ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_dpsk_demod_soft_batch(pu_dpsk* h, const float* samples, size_t B, size_t L, size_t data_start, int ref_mode,
                                   const float* est_cfo_hz, const float* phase_offset, float* llr_out, size_t llr_stride,
                                   pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_dpsk_demod_soft_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && llr_out, "pu_dpsk_demod_soft_batch: NULL data pointer");
    PU_REQUIRE(data_start <= L, "pu_dpsk_demod_soft_batch: data_start beyond the frame");
    PU_REQUIRE(ref_mode == 0 || ref_mode == 1, "pu_dpsk_demod_soft_batch: ref_mode must be 0 or 1");
    PU_REQUIRE(llr_stride > 0, "pu_dpsk_demod_soft_batch: llr_stride is zero");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_DEVICE) return dpsk_launch(h, samples, B, L, data_start, ref_mode, est_cfo_hz, phase_offset, llr_out, llr_stride, st, nullptr, nullptr);
    pu::HostStage hs(ctx, st, B);
    const float *d_x, *d_cfo, *d_phase;
    float* d_llr;
    hs.in(&d_x, samples, L);
    hs.in(&d_cfo, est_cfo_hz, 1);
    hs.in(&d_phase, phase_offset, 1);
    hs.out(&d_llr, llr_out, llr_stride);
    return hs.run([&](size_t nb) { return dpsk_launch(h, d_x, nb, L, data_start, ref_mode, d_cfo, d_phase, d_llr, llr_stride, st, nullptr, nullptr); });
}

pu_status pu_mcdpsk_create(pu_ctx* ctx, const pu_mcdpsk_config* cfg, pu_mcdpsk** out) {
    PU_REQUIRE(ctx && cfg && out, "pu_mcdpsk_create: NULL argument");
    *out = nullptr;
    if (cfg->num_carriers < 1 || cfg->num_carriers > 64 || cfg->samples_per_symbol == 0 || cfg->samples_per_symbol > 8192 ||
        (cfg->bits_per_symbol != 1 && cfg->bits_per_symbol != 2) || !(cfg->sample_rate > 0)) {
        pu::set_error("pu_mcdpsk_create: num_carriers in [1, 64], samples_per_symbol in [1, 8192], bits_per_symbol 1 or 2");
        return PU_ERR_UNSUPPORTED;
    }
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    std::unique_ptr<pu_mcdpsk> h(new (std::nothrow) pu_mcdpsk());
    if (!h) return PU_ERR_NOMEM;
    h->ctx = ctx;
    h->device = ctx->device;
    h->cfg = *cfg;
    const int nc = static_cast<int>(cfg->num_carriers), sps = static_cast<int>(cfg->samples_per_symbol);
    const std::vector<float> freqs = pu::mcdpsk_carrier_freqs(*cfg);
    std::vector<std::complex<float>> mixer(static_cast<size_t>(nc) * sps), expected(nc);
    for (int c = 0; c < nc; ++c) {
        const float inc = static_cast<float>(2.0f * 3.14159265358979323846 * freqs[c] / cfg->sample_rate);   // :667
        float phase = 0.0f;
        for (int i = 0; i < sps; ++i) {
            mixer[static_cast<size_t>(c) * sps + i] = std::polar(1.0f, -phase);                              // :672
            phase += inc;
        }
        const float expected_phase = static_cast<float>((c * 1 - c * 0) * 3.14159265358979323846 / 2.0f);    // :404
        expected[c] = std::polar(1.0f, expected_phase);
    }
    pu_status s;
    if ((s = h->d_mixer.upload(mixer.data(), mixer.size())) != PU_OK) return s;
    if ((s = h->d_expected.upload(expected.data(), expected.size())) != PU_OK) return s;
    *out = h.release();
    return PU_OK;
}

void pu_mcdpsk_destroy(pu_mcdpsk* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    h->corr.release();
    h->corrected.release();
    delete h;
}

static pu_status mcdpsk_launch(pu_mcdpsk* h, const float* d_samples, size_t B, size_t L, float* d_llr, size_t llr_stride, float* d_cfo,
                               cudaStream_t st) {
    const int sps = static_cast<int>(h->cfg.samples_per_symbol), nc = static_cast<int>(h->cfg.num_carriers);
    const int training = static_cast<int>(h->cfg.training_symbols);
    const int n_sym = static_cast<int>(L / sps);
    const int n_pairs = n_sym * nc;
    pu_status s;
    if ((s = h->corr.reserve(B * static_cast<size_t>(n_pairs) * sizeof(float2))) != PU_OK) return s;
    float2* corr = static_cast<float2*>(h->corr.ptr);
    const int rows_max = pu::kPskThreads / nc + 2;
    const size_t smem = sizeof(float) * static_cast<size_t>(rows_max) * 33;
    (void)cudaGetLastError();
    const size_t kMaxY = 65535;
    for (size_t off = 0; off < B; off += kMaxY) {
        const size_t nb = std::min(kMaxY, B - off);
        const dim3 grid(static_cast<unsigned>((n_pairs + pu::kPskThreads - 1) / pu::kPskThreads), static_cast<unsigned>(nb));
        pu::mcdpsk_correlate_kernel<<<grid, pu::kPskThreads, smem, st>>>(d_samples + off * L, L, sps, nc, n_sym,
                                                                       static_cast<const float2*>(h->d_mixer.p), corr + off * n_pairs);
        h->ctx->launches.fetch_add(1);
    }
    const int n_data = n_sym - training - 1;
    const size_t total = std::max(B * static_cast<size_t>(std::max(n_data, 0)) * nc, B);
    pu::mcdpsk_llr_kernel<<<static_cast<unsigned>((total + 127) / 128), 128, 0, st>>>(
        corr, nc, n_sym, training, static_cast<int>(h->cfg.bits_per_symbol), sps, h->cfg.sample_rate,
        static_cast<const float2*>(h->d_expected.p), B, d_llr, llr_stride, d_cfo);
    h->ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_mcdpsk_demod_soft_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, float* llr_out, size_t llr_stride,
                                     float* residual_cfo_hz, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_mcdpsk_demod_soft_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && llr_out, "pu_mcdpsk_demod_soft_batch: NULL data pointer");
    PU_REQUIRE(llr_stride > 0, "pu_mcdpsk_demod_soft_batch: llr_stride is zero");
    PU_REQUIRE(L >= static_cast<size_t>(h->cfg.training_symbols + 1) * h->cfg.samples_per_symbol,
               "pu_mcdpsk_demod_soft_batch: frame shorter than training + reference symbols");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_DEVICE) return mcdpsk_launch(h, samples, B, L, llr_out, llr_stride, residual_cfo_hz, st);
    pu::HostStage hs(ctx, st, B);
    const float* d_x;
    float *d_llr, *d_res;
    hs.in(&d_x, samples, L);
    hs.out(&d_llr, llr_out, llr_stride);
    hs.out(&d_res, residual_cfo_hz, 1);
    return hs.run([&](size_t nb) { return mcdpsk_launch(h, d_x, nb, L, d_llr, llr_stride, d_res, st); });
}

// MultiCarrierDPSKDemodulator behind an externally detected chirp (MCDPSKWaveform::process, src/waveform/mc_dpsk_waveform.cpp:144-170:
// setChirpDetected(cfo) -> process(training + ref + data) -> getSoftBits), i.e. processGotChirp (multi_carrier_dpsk.hpp:533-627).
static pu_status mcdpsk_got_chirp(pu_mcdpsk* h, const float* d_x, size_t B, size_t L, const float* d_cfo, const int* d_start,
                                  const std::vector<int>* h_start, float* d_llr, size_t llr_stride, std::vector<int32_t>& n_h,
                                  std::vector<float>& after_h, cudaStream_t st) {
    pu_ctx* ctx = h->ctx;
    const size_t pre = static_cast<size_t>(h->cfg.training_symbols + 1) * h->cfg.samples_per_symbol;
    pu::DevMem dres;
    pu_status s;
    std::vector<float> res(B, 0.0f), cfo_h(B);
    size_t Lmax = 0;                                     // longest per-frame span
    std::vector<size_t> Lb(B, L);
    for (size_t b = 0; b < B; ++b) {
        if (h_start) { const int st0 = (*h_start)[b]; Lb[b] = (st0 >= 0 && static_cast<size_t>(st0) <= L) ? L - static_cast<size_t>(st0) : 0; }
        Lmax = std::max(Lmax, Lb[b]);
    }
    if (Lmax > pre) {   // processGotChirp needs data behind the preamble; otherwise it keeps waiting (no soft bits)
        if ((s = h->corrected.reserve(B * L * sizeof(float))) != PU_OK) return s;   // 0.7 GB at 2 048 x 84 200: not per call
        float* dy = static_cast<float*>(h->corrected.ptr);
        if ((s = dres.upload(res.data(), B)) != PU_OK) return s;
        pu::HilbertTaps taps;
        const int M = (pu::kHilbertTaps - 1) / 2;
        for (int n = 0; n < pu::kHilbertTaps; ++n) {                       // HilbertTransform ctor, src/dsp/filters.cpp:266-291
            const int k = n - M;
            float c = 0;
            if (k != 0 && k % 2 != 0) c = static_cast<float>(2.0f / (3.14159265358979323846 * k));
            const float w = static_cast<float>(2.0f * 3.14159265358979323846 * n / (pu::kHilbertTaps - 1));
            c *= 0.42f - 0.5f * std::cos(w) + 0.08f * std::cos(2.0f * w);
            taps.c[n] = c;
        }
        (void)cudaGetLastError();
        pu::mcdpsk_cfo_correct_kernel<<<static_cast<unsigned>(B), pu::kCfoThreads, 0, st>>>(taps, d_x, L, static_cast<int>(L), h->cfg.sample_rate,
                                                                                            d_cfo, dy, d_start);
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        if ((s = mcdpsk_launch(h, dy, B, L, d_llr, llr_stride, static_cast<float*>(dres.p), st)) != PU_OK) return s;
        PU_CUDA_TRY(cudaMemcpyAsync(res.data(), dres.p, B * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    PU_CUDA_TRY(cudaMemcpyAsync(cfo_h.data(), d_cfo, B * sizeof(float), cudaMemcpyDeviceToHost, st));
    PU_CUDA_TRY(cudaStreamSynchronize(st));
    // processTraining's cfo update and the false-positive rule (:572-607), per frame on the host: a handful of scalar operations
    const int nc = static_cast<int>(h->cfg.num_carriers), bits = static_cast<int>(h->cfg.bits_per_symbol), sps = static_cast<int>(h->cfg.samples_per_symbol);
    n_h.assign(B, 0);
    after_h.assign(B, 0.0f);
    for (size_t b = 0; b < B; ++b) {
        const bool live = Lb[b] > pre;
        float cfo = cfo_h[b];
        if (live && std::fabs(cfo) > 0.1f) cfo = 0.0f;                     // applyCFOCorrection resets cfo_hz_
        const float dual = cfo;
        float after = cfo;
        if (live && h->cfg.training_symbols >= 2) after = std::max(-50.0f, std::min(50.0f, cfo + res[b]));
        if (std::fabs(dual) > 0.1f) after = cfo;
        after_h[b] = live ? after : cfo_h[b];
        const bool rejected = std::fabs(dual) < 0.1f && std::fabs(after) > 5.0f;
        const size_t nsym = live ? (Lb[b] - pre) / sps : 0;
        n_h[b] = (live && !rejected) ? static_cast<int32_t>(std::min(nsym * nc * bits, llr_stride)) : 0;
    }
    return PU_OK;
}

pu_status pu_mcdpsk_got_chirp_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, const float* chirp_cfo_hz, float* llr_out,
                                    size_t llr_stride, int32_t* n_llr, float* cfo_after_hz, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_mcdpsk_got_chirp_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && chirp_cfo_hz && llr_out && n_llr && cfo_after_hz, "pu_mcdpsk_got_chirp_batch: NULL data pointer");
    PU_REQUIRE(llr_stride > 0 && L < (1u << 30), "pu_mcdpsk_got_chirp_batch: bad size");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float *d_x, *d_cfo;
        float *d_llr, *d_after;
        int32_t* d_n;
        hs.in(&d_x, samples, L);
        hs.in(&d_cfo, chirp_cfo_hz, 1);
        hs.out(&d_llr, llr_out, llr_stride);
        hs.out(&d_n, n_llr, 1);
        hs.out(&d_after, cfo_after_hz, 1);
        return hs.run([&](size_t nb) {
            return pu_mcdpsk_got_chirp_batch(h, d_x, nb, L, d_cfo, d_llr, llr_stride, d_n, d_after, PU_MEM_DEVICE, st);
        });
    }
    std::vector<int32_t> n_h;
    std::vector<float> after_h;
    const pu_status s = mcdpsk_got_chirp(h, samples, B, L, chirp_cfo_hz, nullptr, nullptr, llr_out, llr_stride, n_h, after_h, st);
    if (s != PU_OK) return s;
    PU_CUDA_TRY(cudaMemcpyAsync(n_llr, n_h.data(), B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    PU_CUDA_TRY(cudaMemcpyAsync(cfo_after_hz, after_h.data(), B * sizeof(float), cudaMemcpyHostToDevice, st));
    return PU_OK;
}

// The IWaveform receive sequence (tools/test_iwaveform.cpp:127-160) on MC-DPSK frames [chirp pair][training][ref][data]:
// MCDPSKWaveform::detectSync (src/waveform/mc_dpsk_waveform.cpp:100-142) -> setFrequencyOffset(cfo) (:71-76) -> process (:144-170).
pu_status pu_mcdpsk_chirp_receive_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, float threshold, float* llr_out,
                                        size_t llr_stride, int32_t* n_llr, int32_t* sync_info, float* sync_values, float* cfo_after_hz,
                                        pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_mcdpsk_chirp_receive_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && sync_info && sync_values, "pu_mcdpsk_chirp_receive_batch: NULL data pointer");
    PU_REQUIRE(!llr_out || (n_llr && cfo_after_hz && llr_stride > 0), "pu_mcdpsk_chirp_receive_batch: llr_out needs n_llr, cfo_after_hz and llr_stride");
    PU_REQUIRE(L < (1u << 30), "pu_mcdpsk_chirp_receive_batch: frame too long");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu_status s;
    if (!h->chirp_ready) {
        std::vector<float> t;
        pu::chirp_templates_host(h->cfg.sample_rate, t, h->chirp);
        if ((s = h->d_chirp.upload(t.data(), t.size())) != PU_OK) return s;
        pu::chirp_dev_bind(h->chirp, static_cast<const float*>(h->d_chirp.p));
        h->chirp_ready = true;
    }
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (threshold <= 0.0f) threshold = 0.15f;        // the callers' value, tools/test_iwaveform.cpp:133
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float* d_x;
        float *d_val, *d_llr, *d_after;
        int32_t *d_info, *d_n;
        hs.in(&d_x, samples, L);
        hs.out(&d_info, sync_info, 4);
        hs.out(&d_val, sync_values, 4);
        hs.out(&d_llr, llr_out, llr_stride);
        hs.out(&d_n, llr_out ? n_llr : nullptr, 1);
        hs.out(&d_after, llr_out ? cfo_after_hz : nullptr, 1);
        return hs.run([&](size_t nb) {
            return pu_mcdpsk_chirp_receive_batch(h, d_x, nb, L, threshold, d_llr, llr_stride, d_n, d_info, d_val, d_after, PU_MEM_DEVICE, st);
        });
    }
    pu::DevMem dinfo, dval, dcfo, dstart;
    std::vector<int32_t> info_h(B * 4, 0);
    std::vector<float> val_h(B * 4, 0.0f);
    if ((s = dinfo.upload(info_h.data(), info_h.size())) != PU_OK) return s;
    if ((s = dval.upload(val_h.data(), val_h.size())) != PU_OK) return s;
    if ((s = dcfo.upload(val_h.data(), B)) != PU_OK) return s;
    (void)cudaGetLastError();
    PU_CUDA_TRY(pu::chirp_detect_launch(h->chirp, samples, B, L, static_cast<int>(L), threshold, static_cast<int>(h->cfg.samples_per_symbol),
                                        static_cast<int4*>(dinfo.p), static_cast<float4*>(dval.p), nullptr, nullptr, static_cast<float*>(dcfo.p),
                                        nullptr, nullptr, 0, 0, st));
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaStreamSynchronize(st));
    PU_CUDA_TRY(cudaMemcpy(info_h.data(), dinfo.p, info_h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    PU_CUDA_TRY(cudaMemcpy(val_h.data(), dval.p, val_h.size() * sizeof(float), cudaMemcpyDeviceToHost));
    // MCDPSKWaveform::detectSync (:117-134): the training sequence starts two chirps and two gaps behind the up chirp (the kernel's own
    // start_sample is the OFDM_CHIRP rule); tools/test_iwaveform.cpp:143 drops frames whose start lies at or beyond the end
    std::vector<int> start_h(B, -1);
    for (size_t b = 0; b < B; ++b) {
        int start = -1;
        if (info_h[4 * b]) start = static_cast<int>(static_cast<size_t>(info_h[4 * b + 1]) + 2 * static_cast<size_t>(h->chirp.n) + 2 * static_cast<size_t>(h->chirp.gap));
        info_h[4 * b + 3] = start;
        val_h[4 * b + 3] = 0.0f;                       // no rotator phase on this path (the CFO is removed by the Hilbert-FIR shift)
        start_h[b] = (start >= 0 && static_cast<size_t>(start) < L) ? start : -1;
    }
    PU_CUDA_TRY(cudaMemcpyAsync(sync_info, info_h.data(), info_h.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    PU_CUDA_TRY(cudaMemcpyAsync(sync_values, val_h.data(), val_h.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    if (!llr_out) return PU_OK;                        // detection only (IWaveform::detectSync)
    if ((s = dstart.upload(start_h.data(), B)) != PU_OK) return s;
    std::vector<int32_t> n_h;
    std::vector<float> after_h;
    if ((s = mcdpsk_got_chirp(h, samples, B, L, static_cast<const float*>(dcfo.p), static_cast<const int*>(dstart.p), &start_h, llr_out, llr_stride,
                              n_h, after_h, st)) != PU_OK) return s;
    PU_CUDA_TRY(cudaMemcpyAsync(n_llr, n_h.data(), B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    PU_CUDA_TRY(cudaMemcpyAsync(cfo_after_hz, after_h.data(), B * sizeof(float), cudaMemcpyHostToDevice, st));
    return PU_OK;
}

}  // extern "C"
