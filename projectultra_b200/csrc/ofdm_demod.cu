// projectultra_b200/csrc/ofdm_demod.cu — batched presynced OFDM receive path for sm_100a and the pu_ofdm_*
// entry points of the C ABI: baseband mix -> FFT -> LTS channel estimate -> pilot tracking -> interpolation ->
// equaliser -> soft demapper, one launch, LLRs written once.
//
// Reference behaviour: OFDMDemodulator::processPresynced (src/ofdm/demodulator.cpp:854-985) after
// reset() + setFrequencyOffset[WithPhase]() on a fresh object, i.e. the per-frame algorithm of SURVEY App. E:
//   toBaseband            src/ofdm/channel_equalizer.cpp:19-57   (NCO mix over ALL samples, optional CFO rotator)
//   extractSymbol + FFT   :59-71, src/dsp/fft.cpp:89-121         (drop CP, in-order radix-2 DIT)
//   estimateChannelFromLTS :77-328                               (data H = last LTS symbol, pilot H = mean)
//   updateChannelEstimate :330-595                               (pilot LS, phase lock, EMA, CFO / timing / noise trackers)
//   interpolateChannel    :601-631
//   equalize              :728-840                               (ZF for differential, MMSE + fade erasure for coherent)
//   demodulateSymbol      src/ofdm/demodulator.cpp:199-356, soft_demap.hpp
// The decision-directed tracker block (demodulator.cpp:362-434) is numerically dead (SURVEY §0.3/Q14: it reads
// the reference symbol after it was overwritten, so every correction is exactly (1,+-0)); it is not executed here.
//
// Numerics: the FFT performs the reference's radix-2 butterflies in the reference's order (fused in registers
// three stages at a time) with unfused fp32 multiplies/adds, so FFT bins, H and equalised symbols are bit-identical
// to the reference; the libm calls on the path (atan2f, sinf, cosf, hypotf) are restated in ref_math.cuh so that
// LLRs match to the last bit as well (up to the host libm's FMA/non-FMA variant).  Compiled with -fmad=false.
//
// Kernel shape: one frame per CTA of NFFT/8 threads; the frame's symbols are walked in order because in pilot
// modes symbol s+1's mixer depends on the CFO tracked in symbol s.  Shared memory holds one padded FFT buffer,
// the per-carrier state and the trackers.
#include <cfloat>
#include <cstdlib>
#include <memory>
#include <new>

#include "ofdm_plan.h"
#include "pu_async.cuh"
#include "frame_v2.cuh"
#include "ldpc_encode.cuh"
#include "pu_internal.h"
#include "ref_math.cuh"
#include "ofdm_dev.cuh"

namespace pu {

// Out-of-line copies of the libm restatements: the kernel calls them from 16 places, and inlining every copy made the
// warp-granular kernel 14 000 instructions long -- with each warp in a different phase of its frame the instruction
// cache thrashed (r11: 4.4 "no instruction" stall cycles per issued instruction).
namespace nl {
static __device__ __noinline__ float atan2f_ref(float y, float x) { return refmath::atan2f_ref(y, x); }
static __device__ __noinline__ float sinf_ref(float x) { return refmath::sinf_ref(x); }
static __device__ __noinline__ float cosf_ref(float x) { return refmath::cosf_ref(x); }
static __device__ __noinline__ void sincosf_ref(float x, float* s, float* c) { *s = refmath::sinf_ref(x); *c = refmath::cosf_ref(x); }
}  // namespace nl

#define PADIDX(p) ((p) + ((p) >> 3))   // one float2 of padding per 8 keeps the strided passes off the same banks

__device__ __forceinline__ void butterfly(float2& a, float2& b, float2 w) {
    const float2 t = cmul(w, b);     // Complex t = w * data[i + k + half]      (fft.cpp:108)
    b = csub(a, t);                  // data[i + k + half] = data[i + k] - t
    a = cadd(a, t);                  // data[i + k]        = data[i + k] + t
}

// R consecutive radix-2 stages (global stages S0+1 .. S0+R) on the 2^R elements base + q*2^S0 held in registers.
template <int R, int S0, int LOG2N>
__device__ __forceinline__ void stages_in_regs(float2 (&v)[1 << R], int lo, const float2* __restrict__ tw) {
#pragma unroll
    for (int t = 1; t <= R; ++t) {
        constexpr int dummy = 0;
        (void)dummy;
        const int half = 1 << (t - 1);
#pragma unroll
        for (int pr = 0; pr < (1 << (R - 1)); ++pr) {
            const int kq = pr & (half - 1);
            const int a = ((pr >> (t - 1)) << t) | kq;
            const int k = lo + (kq << S0);
            const float2 w = __ldg(&tw[k << (LOG2N - S0 - t)]);
            butterfly(v[a], v[a + half], w);
        }
    }
}

template <int R, int S0, int LOG2N>
__device__ __forceinline__ void fft_pass_smem(float2* buf, int gid, const float2* __restrict__ tw) {
    const int lo = gid & ((1 << S0) - 1);
    const int base = ((gid >> S0) << (S0 + R)) | lo;
    float2 v[1 << R];
#pragma unroll
    for (int q = 0; q < (1 << R); ++q) v[q] = buf[PADIDX(base + (q << S0))];
    stages_in_regs<R, S0, LOG2N>(v, lo, tw);
#pragma unroll
    for (int q = 0; q < (1 << R); ++q) buf[PADIDX(base + (q << S0))] = v[q];
}

// ---- warp-granular variant (WARPG): one warp walks one frame; the FFT is the two-pass register FFT of ofdm_diff.cu
//      (pass A: N/32 elements per lane, log2(N/32) stages; one padded shared-memory transpose; pass B pruned to the
//      bins within +-CW of DC), every butterfly still the reference's unfused (t = w*b, a+t, a-t) in stage order.
template <int NFFT>
struct WgGeom {
    static constexpr int LOG2N = (NFFT == 512) ? 9 : 10;
    static constexpr int EPL = NFFT / 32;                    // elements per lane
    static constexpr int LA = (NFFT == 512) ? 4 : 5;         // stages of pass A = in-lane stages of pass B
    static constexpr int CW = (NFFT == 512) ? 16 : 32;       // pass B: p = c + CW*j (+256*b8 for N = 512)
    static constexpr int PADSH = (NFFT == 512) ? 4 : 5;      // one float2 of padding per 2^PADSH
    static constexpr int BUF = NFFT + (NFFT >> PADSH);       // float2 per warp
};
struct WgTw { float2 a[16]; };                               // pass-A twiddles tw[32 m] (N = 512) / tw[32 m] (N = 1024: tw[(N/32) m])
__device__ __forceinline__ float2 wg_lo(float2 a, float2 b, float2 w) { return cadd(a, cmul(w, b)); }
__device__ __forceinline__ float2 wg_hi(float2 a, float2 b, float2 w) { return csub(a, cmul(w, b)); }

// PU_PRECISION_FAST forms of the same butterflies (BASELINE.json's 1e-4 LLR contract instead of bit-identical bins): fused
// multiply-adds, a - w b as 2a - (a + w b), and no multiplication at all for the twiddles 1 and -j.
__device__ __forceinline__ float2 fwg_lo(float2 a, float2 b, float2 w) {
    return make_float2(__fmaf_rn(w.x, b.x, __fmaf_rn(-w.y, b.y, a.x)), __fmaf_rn(w.x, b.y, __fmaf_rn(w.y, b.x, a.y)));
}
__device__ __forceinline__ float2 fwg_hi(float2 a, float2 b, float2 w) {
    return make_float2(__fmaf_rn(-w.x, b.x, __fmaf_rn(w.y, b.y, a.x)), __fmaf_rn(-w.x, b.y, __fmaf_rn(-w.y, b.x, a.y)));
}
__device__ __forceinline__ void fbutterfly(float2& a, float2& b, float2 w) {
    const float2 s = fwg_lo(a, b, w);
    b = make_float2(__fmaf_rn(2.0f, a.x, -s.x), __fmaf_rn(2.0f, a.y, -s.y));
    a = s;
}
// m = twiddle index out of QUARTER * 4 (compile-time after unrolling): 0 -> w = 1, QUARTER -> w = -j
template <int QUARTER>
__device__ __forceinline__ void fbutterfly_m(float2& a, float2& b, int m, float2 w) {
    if (m == 0) {
        const float2 t = b;
        b = make_float2(__fsub_rn(a.x, t.x), __fsub_rn(a.y, t.y));
        a = make_float2(__fadd_rn(a.x, t.x), __fadd_rn(a.y, t.y));
    } else if (m == QUARTER) {          // t = -j b = (b.y, -b.x)
        const float2 t = make_float2(b.y, -b.x);
        b = make_float2(__fsub_rn(a.x, t.x), __fsub_rn(a.y, t.y));
        a = make_float2(__fadd_rn(a.x, t.x), __fadd_rn(a.y, t.y));
    } else {
        fbutterfly(a, b, w);
    }
}

struct RxShared {
    float2 Hd[kMaxCarr];      // channel_estimate at data carriers
    float2 Hp[kMaxCarr];      // channel_estimate at pilot carriers
    float2 Fd[kMaxCarr];      // FFT bins at data carriers
    float2 Fp[kMaxCarr];      // FFT bins at pilot carriers
    float2 hls[kMaxCarr];     // h_ls_all
    float2 prevp[kMaxCarr];   // prev_pilot_phases
    float2 preveq[kMaxCarr];  // dbpsk_prev_equalized
    float2 eq[kMaxCarr];
    float2 tmpc[kMaxCarr];
    float tmpa[kMaxCarr], tmpb[kMaxCarr], tmpd[kMaxCarr];
    float cnv[kMaxCarr];      // carrier_noise_var
    int valid[kMaxCarr];
    // trackers (demodulator_impl.hpp)
    float cfo_hz, cfo_filt, rot_phase, noise_var, snr_lin, timing;
    int snr_cnt, since_sync, have_prev, cpc_init, have_preveq;
    float2 ppc, cpc;
    float cfo_used;
    int rot_fail[4];          // first broken link of each warp in the rotator-phase chain
    float rot_next;
};

// WARPG = false: one frame per CTA of NFFT/8 threads (debug dumps, carrier layouts the warp FFT does not cover).
// WARPG = true:  one frame per WARP, blockDim.x / 32 frames per CTA, no CTA-wide barrier anywhere: the serial tracker
//                sections and the HBM latency of a frame's next symbol only stall that frame's warp.
#define PU_GSYNC() do { if constexpr (WARPG) __syncwarp(); else __syncthreads(); } while (0)
// FAM: 0 = modulation family decided at run time, 1 = differential (DBPSK/DQPSK/D8PSK), 2 = coherent: the warp form is
// compiled once per family so that each instance carries only its own equaliser and demappers (instruction-cache footprint).
// FAST (warp form only): PU_PRECISION_FAST arithmetic -- FMA butterflies (above) and MUFU sin/cos (2^-21 absolute) + FMA mixing in the
// CFO rotator instead of the exact libm restatements.  The rotator PHASES stay the reference's (the per-sample float recurrence walked
// with bit-for-bit link checks): a closed form ph0 + i * inc was measured (v20) to drift from the recurrence by its systematic rounding
// bias -- up to 1e-3 rad over a frame when |phase| ~ pi -- which moves coherent-QAM LLRs by 1e-2 and more.
template <int NFFT, bool WARPG, int FAM, bool FAST = false>
__global__ void __launch_bounds__(WARPG ? 512 : NFFT / 8, 1) ofdm_presynced_kernel(
    OfdmDev d, WgTw twa, const float* __restrict__ samples, size_t frame_stride, size_t B, int n_symbols, int training,
    const float* __restrict__ cfo_hz, const float* __restrict__ cfo_phase,
    float* __restrict__ llr_out, size_t llr_stride, int llr_limit,
    float* __restrict__ snr_db_out, float* __restrict__ final_cfo_out, float* __restrict__ dbg, unsigned group_bytes,
    const int* __restrict__ frame_start, const int* __restrict__ frame_nsym) {
    constexpr int LOG2N = (NFFT == 512) ? 9 : 10;
    constexpr int T = WARPG ? 32 : NFFT / 8;
    using G = WgGeom<NFFT>;
    extern __shared__ __align__(16) unsigned char smem_all[];
    const int tid = WARPG ? static_cast<int>(threadIdx.x & 31) : static_cast<int>(threadIdx.x);
    const int wig = WARPG ? static_cast<int>(threadIdx.x >> 5) : 0;
    const size_t frame = WARPG ? static_cast<size_t>(blockIdx.x) * (blockDim.x >> 5) + wig : blockIdx.x;
    // warp form: all warps of the CTA meet at a barrier at the top of every symbol, so that they walk the same part of this long
    // kernel at the same time and share its instruction-cache lines; frames past the batch idle instead of leaving
    const bool no_frame = WARPG && frame >= B;
    const int n_symbols_cta = n_symbols;
    unsigned char* smem_raw = smem_all + static_cast<size_t>(wig) * group_bytes;
    // CTA mode: [NFFT + NFFT/8] FFT buffer, then [sym_len] rotator phases.  Warp mode: [BUF] transpose buffer (its first
    // NFFT entries double as the buffer of rotated samples), then the [2 CW] bins around DC; phases stay in registers.
    float2* buf = reinterpret_cast<float2*>(smem_raw);
    float* theta = reinterpret_cast<float*>(buf + NFFT + NFFT / 8);
    float2* binbuf = buf + G::BUF;
    RxShared& S = WARPG ? *reinterpret_cast<RxShared*>(binbuf + 2 * G::CW)
                        : *reinterpret_cast<RxShared*>(theta + ((d.sym_len + 3) & ~3));
    // optional per-frame window (acquired frames, pu_ofdm_process_batch): the symbols start frame_start[frame] samples into the
    // row and there are frame_nsym[frame] of them; the NCO restarts there (mixer.reset(), demodulator.cpp:583)
    const float* x = samples + (no_frame ? 0 : frame * frame_stride + (frame_start ? frame_start[frame] : 0));
    if (frame_nsym && !no_frame) n_symbols = min(n_symbols, max(frame_nsym[frame], 0));
    if (no_frame) n_symbols = 0;
    const int nd = d.n_data, np = d.n_pilot, nu = nd + np;
    const bool differential = FAM == 1 ? true : FAM == 2 ? false : (d.mod == PU_MOD_DBPSK || d.mod == PU_MOD_DQPSK || d.mod == PU_MOD_D8PSK);

    // warp FFT: per-lane twiddles of pass B (loop invariant)
    const int lane = tid;
    const int wc = lane & (G::CW - 1);
    const int wb8 = (NFFT == 512) ? (lane >> 4) : 0;
    const int rlane = static_cast<int>(__brev(static_cast<unsigned>(lane)) >> 27);
    float2 wl[G::LA], wh[G::LA], wlast = make_float2(0.0f, 0.0f);
    if constexpr (WARPG) {
#pragma unroll
        for (int q = 0; q < G::LA; ++q) {
            const int sh = LOG2N - (G::LA + 1 + q);
            wl[q] = __ldg(&d.twiddle[wc << sh]);
            wh[q] = __ldg(&d.twiddle[(wc + G::CW * ((1 << q) - 1)) << sh]);
        }
        if (NFFT == 512) wlast = __ldg(&d.twiddle[wb8 ? (wc + 240) : wc]);
    }

    if (tid == 0) {
        const float f = (cfo_hz && !no_frame) ? cfo_hz[frame] : 0.0f;
        S.cfo_hz = f;
        S.cfo_filt = f;
        S.rot_phase = (cfo_phase && !no_frame) ? cfo_phase[frame] : 0.0f;
        S.noise_var = 0.1f;
        S.snr_lin = 1.0f;
        S.timing = 0.0f;
        S.snr_cnt = 0;
        S.since_sync = 0;
        S.have_prev = 0;
        S.cpc_init = 0;
        S.have_preveq = 0;
        S.ppc = make_float2(1.0f, 0.0f);
        S.cpc = make_float2(1.0f, 0.0f);
    }
    for (int i = tid; i < kMaxCarr; i += T) {
        S.Hd[i] = make_float2(1.0f, 0.0f);
        S.Hp[i] = make_float2(1.0f, 0.0f);
        S.preveq[i] = make_float2(1.0f, 0.0f);   // differential reference (1,0): channel_equalizer.cpp:300, demodulator.cpp:251-255
        S.tmpc[i] = make_float2(0.0f, 0.0f);     // h_sum_pilot accumulator during the LTS phase
    }
    PU_GSYNC();

    // Warp form: the FFT window of the NEXT symbol is staged into shared memory with per-lane cp.async while the equaliser /
    // tracker / demapper part of the current one runs (v26 capture of the synchronous form: 2.4 long-scoreboard stall cycles per
    // issued instruction, 31 % of all stall samples on the pass-A loads -- with one CTA per SM walking the symbols in step,
    // nothing else was there to cover the DRAM latency).  The staging area is the upper half of the transpose buffer (floats
    // [NFFT, 2 NFFT) of buf), free between the pass-B reads of one symbol and pass A of the next; the rotated samples
    // zbuf[k] (bytes 8k..8k+7) are written in ascending k and overwrite only staged samples 2k - NFFT (+1) <= k, already used.
    float* xsm = reinterpret_cast<float*>(buf) + NFFT;
    auto next_fft_symbol = [&](int after) {           // first symbol > after that runs an FFT (LTS symbols but the last do not when np == 0)
        const int c = after + 1;
        return (np == 0 && c < training - 1) ? training - 1 : c;
    };
    auto stage = [&](int sn) {
        if (sn >= n_symbols) return;
        const float* src = x + static_cast<size_t>(sn) * d.sym_len + d.cp;
        const uint32_t dst = smem_u32(xsm);
        if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
            for (int m = 0; m < NFFT / 128; ++m) cp_async16(dst + 16 * (32 * m + lane), src + 4 * (32 * m + lane));
        } else {                                      // acquired frames start on any sample
#pragma unroll 8
            for (int m = 0; m < NFFT / 32; ++m) cp_async4(dst + 4 * (32 * m + lane), src + 32 * m + lane);
        }
        cp_async_commit();
    };
    if constexpr (WARPG) stage(next_fft_symbol(-1));
    int llr_pos = 0;   // LLRs emitted so far (same for all threads)
    for (int s = 0; s < (WARPG ? n_symbols_cta : n_symbols); ++s) {
        if constexpr (WARPG) {
            __syncthreads();
            if (s >= n_symbols) continue;
        }
        const bool is_train = s < training;
        const float* xs = x + static_cast<size_t>(s) * d.sym_len;
        const float2* nco = d.nco + static_cast<size_t>(s) * d.sym_len;
        if constexpr (WARPG) {
            // the warp waits on nothing but its own loads: pull the NEXT symbol's samples into L2 while this one is processed
            if (s + 1 < n_symbols) {
                const char* nx = reinterpret_cast<const char*>(xs + d.sym_len);
                for (int off = tid * 128; off < d.sym_len * 4; off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + off));
            }
        }
        // ---------------- rotator phases (channel_equalizer.cpp:23,39-51): a per-sample float recurrence
        //   theta[i] = ph;  ph = wrap(fl(ph + inc)).
        // Run T samples at a time: while ph stays in one binade every step adds the same number of ulps, so the next T
        // values are bits(ph) + t * (bits(step(ph)) - bits(ph)); thread t checks its own link step(c_t) == c_{t+1} bit for
        // bit, and the chain is accepted up to the first broken link (binade change, zero crossing, +-pi wrap), where the
        // true successor computed by that thread restarts it.  Every accepted value is thus the reference's value by
        // induction, at ~sym_len / T rounds instead of sym_len dependent additions on one thread.
        const bool rot = fabsf(S.cfo_hz) > 0.01f;
        const float rot_inc = static_cast<float>(__ddiv_rn(__dmul_rn(-2.0f * 3.14159265358979323846, (double)S.cfo_hz), (double)d.sample_rate));
        auto rot_step = [&](float ph) {
            const float pi_hi = 3.14159274101257324f;   // smallest float > M_PI: (double)ph > M_PI  <=>  ph >= pi_hi
            // 2 pi = two_hi + two_lo (float + float).  For pi <= |ph| < 4.2 the reference's float((double)ph -+ 2 pi) equals
            // fl(fl(ph -+ two_hi) -+ two_lo): the first difference is exact (Sterbenz) and lands on the 2^-22 grid of [2, 4), and
            // two_lo = -0.733 ulp of that grid, far from a rounding tie in either precision (tests/test_oracle_ofdm.py checks all
            // 4 019 851 floats of the interval).  Anything larger (|cfo| > 7 kHz) takes the double path, on a warp-uniform branch
            // so that the common case issues no FP64 conversion at all.
            const float two_hi = 6.2831854820251465f, two_lo = -1.7484555e-7f;
            ph = __fadd_rn(ph, rot_inc);
            const float a = fabsf(ph);
            if (__any_sync(0xffffffffu, !(a < 4.2f))) {
                if (ph >= pi_hi) ph = static_cast<float>((double)ph - 2.0f * 3.14159265358979323846);
                else if (ph <= -pi_hi) ph = static_cast<float>((double)ph + 2.0f * 3.14159265358979323846);
            } else if (a >= pi_hi) {
                ph = ph > 0.0f ? __fsub_rn(__fsub_rn(ph, two_hi), two_lo) : __fadd_rn(__fadd_rn(ph, two_hi), two_lo);
            }
            return ph;
        };
        if (!WARPG && rot) {
            float ph = S.rot_phase;
            for (int i = 0; i < d.sym_len;) {
                const unsigned b0 = __float_as_uint(ph);
                const unsigned delta = __float_as_uint(rot_step(ph)) - b0;
                const float cand = __uint_as_float(b0 + static_cast<unsigned>(tid) * delta);
                const float nxt = rot_step(cand);
                const bool broken = __float_as_uint(nxt) != b0 + static_cast<unsigned>(tid + 1) * delta;
                const unsigned bal = __ballot_sync(0xffffffffu, broken);
                if ((tid & 31) == 0) S.rot_fail[tid >> 5] = bal ? (tid + __ffs(bal) - 1) : T;
                PU_GSYNC();
                int f = T;
#pragma unroll
                for (int w = 0; w < T / 32; ++w) f = min(f, S.rot_fail[w]);
                const int nvalid = min(f < T ? f + 1 : T, d.sym_len - i);    // c_0 .. c_f are the reference's values
                if (tid < nvalid) theta[i + tid] = cand;
                if (tid == nvalid - 1) S.rot_next = nxt;                      // true successor of the last accepted value
                PU_GSYNC();
                ph = S.rot_next;
                i += nvalid;
            }
            if (tid == 0) S.rot_phase = ph;
        }
        if (tid == 0) S.cfo_used = S.cfo_hz;
        PU_GSYNC();
        const bool skip_fft = is_train && np == 0 && s != training - 1;   // data H uses the LAST LTS symbol only (:179-185)
        if constexpr (WARPG) {
            constexpr int EPL = G::EPL, LA = G::LA, CW = G::CW;
            float2* zbuf = buf;                                   // [NFFT] rotated samples in natural order (rot only)
            if (!skip_fft) {
                cp_async_wait_all();                              // this symbol's FFT window has landed in xsm
                __syncwarp();
            }
            if (rot) {
                // ---------------- rotator (channel_equalizer.cpp:23,39-51): the per-sample phase recurrence of the whole symbol
                //   with the bit-for-bit link check described above; the lane that holds the phase of a sample of the FFT window
                //   mixes that sample itself, so the phases never leave registers.
                // The chain (b0, delta, i0) -- sample i0 has phase bits b0 and every link adds delta ulps -- persists across the symbol.
                // Samples are taken 128 at a time: each lane forms its four candidates b0 + t delta and their float successors
                // (independent instructions, no loop-carried dependency) and ONE vote says whether all 128 links hold and none comes
                // near +-pi; that is the common case (a break needs a binade change, a zero crossing or a wrap) and costs ~8
                // instructions per 32 samples.  Otherwise the four windows are re-walked one by one with the full rot_step, the
                // chain restarting behind each broken link from the true successor computed by the lane that owns it.
                float ph = S.rot_phase;
                unsigned b0 = __float_as_uint(ph), delta = __float_as_uint(rot_step(ph)) - b0;
                int i0 = 0, wbase = 0;
                const bool keep = !skip_fft;
                // sample i of the symbol rotated by phase th -> out; false outside the FFT window.  Reads and writes of the warp are
                // separated by __syncwarp (the rotated samples overwrite staged samples other lanes have read, see above).
                auto mix = [&](int i, float th, float2& out) {
                    const int k = i - d.cp;
                    if (!(keep && k >= 0 && k < NFFT)) return false;
                    const float xv = xsm[k];
                    const float2 o = __ldg(&nco[i]);
                    float sn, cs;
                    const float2 z = make_float2(__fmul_rn(o.x, xv), __fmul_rn(-o.y, xv));       // samples[i] * conj(osc) (:36)
                    if constexpr (FAST) {            // the reference's phase, MUFU sin/cos (2^-21 absolute), FMA mix
                        __sincosf(th, &sn, &cs);
                        out = make_float2(__fmaf_rn(z.x, cs, -__fmul_rn(z.y, sn)), __fmaf_rn(z.x, sn, __fmul_rn(z.y, cs)));
                    } else {
                        nl::sincosf_ref(th, &sn, &cs);
                        out = cmul(z, make_float2(cs, sn));                                       // mixed *= correction (:42)
                    }
                    return true;
                };
                auto window = [&](int len) {                      // the next len (<= 32) samples, link by link
                    float mine = 0.0f;
                    int done = 0;
                    while (done < len) {
                        const int t = wbase + lane - i0;
                        const float cand = __uint_as_float(b0 + static_cast<unsigned>(t) * delta);
                        const float nxt = rot_step(cand);
                        const bool inside = lane >= done && lane < len;
                        const bool broken = inside && __float_as_uint(nxt) != b0 + static_cast<unsigned>(t + 1) * delta;
                        const unsigned bal = __ballot_sync(0xffffffffu, broken);
                        const int last = bal ? (__ffs(bal) - 1) : (len - 1);      // lane of the last accepted value
                        if (inside && lane <= last) mine = cand;
                        if (bal) {                                                 // its true successor restarts the chain
                            ph = __shfl_sync(0xffffffffu, nxt, last);
                            i0 = wbase + last + 1;
                            b0 = __float_as_uint(ph);
                            delta = __float_as_uint(rot_step(ph)) - b0;
                        }
                        done = last + 1;
                    }
                    float2 r;
                    const bool ok = lane < len && mix(wbase + lane, mine, r);
                    __syncwarp();
                    if (ok) zbuf[wbase + lane - d.cp] = r;
                    wbase += len;
                };
                const float pi_lo = 3.1415925f;                   // largest float below pi_hi: |nxt| <= pi_lo  <=>  rot_step does not wrap
                while (wbase < d.sym_len) {
                    float cand[4];
                    bool brk = false;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int i = wbase + 32 * k + lane;
                        const unsigned cb = b0 + static_cast<unsigned>(i - i0) * delta;
                        cand[k] = __uint_as_float(cb);
                        const float nxt = __fadd_rn(cand[k], rot_inc);
                        brk |= i < d.sym_len && (__float_as_uint(nxt) != cb + delta || !(fabsf(nxt) <= pi_lo));
                    }
                    if (!__any_sync(0xffffffffu, brk)) {
                        float2 r[4];
                        bool ok[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) ok[k] = mix(wbase + 32 * k + lane, cand[k], r[k]);
                        __syncwarp();
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (ok[k]) zbuf[wbase + 32 * k + lane - d.cp] = r[k];
                        wbase += 128;
                    } else {
                        for (int k = 0; k < 4 && wbase < d.sym_len; ++k) window(min(32, d.sym_len - wbase));
                    }
                }
                __syncwarp();                    // every lane has read S.rot_phase (the shuffles of window() order execution, not memory)
                if (lane == 0) S.rot_phase = __uint_as_float(b0 + static_cast<unsigned>(d.sym_len - i0) * delta);   // phase behind the last sample
                __syncwarp();
            }
            if (!skip_fft) {
                // ---------------- pass A: lane g owns bit-reversed positions EPL g .. EPL g + EPL-1 = samples brev5(g) + 32 brev(q)
                float2 v[EPL];
#pragma unroll
                for (int q = 0; q < EPL; ++q) {
                    const int brq = static_cast<int>(__brev(static_cast<unsigned>(q)) >> (32 - LA));
                    const int n = rlane + 32 * brq;
                    if (rot) {
                        v[q] = zbuf[n];
                    } else {
                        const float xv = xsm[n];
                        const float2 o = __ldg(&nco[d.cp + n]);
                        v[q] = make_float2(__fmul_rn(o.x, xv), __fmul_rn(-o.y, xv));               // samples[i] * conj(osc) (:36)
                    }
                }
#pragma unroll
                for (int t = 1; t <= LA; ++t) {
                    const int half = 1 << (t - 1);
#pragma unroll
                    for (int pr = 0; pr < EPL / 2; ++pr) {
                        const int kq = pr & (half - 1);
                        const int a = ((pr >> (t - 1)) << t) | kq;
                        if constexpr (FAST) fbutterfly_m<(1 << LA) / 4>(v[a], v[a + half], kq << (LA - t), twa.a[kq << (LA - t)]);
                        else butterfly(v[a], v[a + half], twa.a[kq << (LA - t)]);
                    }
                }
                __syncwarp();                                       // zbuf has been read by every lane
#pragma unroll
                for (int q = 0; q < EPL; ++q) {
                    const int p = EPL * lane + q;
                    buf[p + (p >> G::PADSH)] = v[q];
                }
                __syncwarp();
                // ---------------- pass B: lane (b8, c) owns p = c + CW j (+ 256 b8); pruned to the outputs at j = 0 and j = EPL-1
#pragma unroll
                for (int j = 0; j < EPL; ++j) {
                    const int p = wc + CW * j + 256 * wb8;
                    v[j] = buf[p + (p >> G::PADSH)];
                }
                __syncwarp();                                       // buf has been read by every lane:
                stage(next_fft_symbol(s));                          // the next FFT window travels during the rest of this symbol
#pragma unroll
                for (int j = 0; j < EPL; j += 2) {
                    if constexpr (FAST) fbutterfly(v[j], v[j + 1], wl[0]);
                    else butterfly(v[j], v[j + 1], wl[0]);
                }
#pragma unroll
                for (int q = 1; q < LA; ++q) {
                    const int step = 1 << (q + 1), hh = 1 << q;
#pragma unroll
                    for (int j = 0; j < EPL; j += step) {
                        if constexpr (FAST) {
                            v[j] = fwg_lo(v[j], v[j + hh], wl[q]);
                            v[j + step - 1] = fwg_hi(v[j + step - 1 - hh], v[j + step - 1], wh[q]);
                        } else {
                            v[j] = wg_lo(v[j], v[j + hh], wl[q]);
                            v[j + step - 1] = wg_hi(v[j + step - 1 - hh], v[j + step - 1], wh[q]);
                        }
                    }
                }
                if (NFFT == 512) {
                    // stage 9 pairs lane (0,c) with lane (1,c): bin c = A0 + w B0 on lane (0,c); bin 496 + c = A15 - w B15 on lane (1,c)
                    const float2 send = wb8 ? v[0] : v[EPL - 1];
                    float2 recv;
                    recv.x = __shfl_xor_sync(0xffffffffu, send.x, 16);
                    recv.y = __shfl_xor_sync(0xffffffffu, send.y, 16);
                    if constexpr (FAST) binbuf[lane] = wb8 ? fwg_hi(recv, v[EPL - 1], wlast) : fwg_lo(v[0], recv, wlast);
                    else binbuf[lane] = wb8 ? wg_hi(recv, v[EPL - 1], wlast) : wg_lo(v[0], recv, wlast);
                } else {
                    binbuf[wc] = v[0];                              // bin c
                    binbuf[CW + wc] = v[EPL - 1];                   // bin N - CW + c
                }
                __syncwarp();
                for (int u = tid; u < nu; u += T) {
                    const int bin = u < nd ? d.data_bin[u] : d.pilot_bin[u - nd];
                    const float2 out = binbuf[bin < NFFT / 2 ? bin : bin - NFFT + 2 * CW];
                    if (u < nd) S.Fd[u] = out;
                    else S.Fp[u - nd] = out;
                }
            }
        } else {
            if (!skip_fft) {
                // ---------------- mix + stages 1..3: group g owns bit-reversed positions 8g..8g+7 = samples brev(8g+q)
                {
                    const int g = tid;
                    const int r = __brev(static_cast<unsigned>(g)) >> (32 - (LOG2N - 3));
                    float2 v[8];
    #pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int brq = ((q & 1) << 2) | (q & 2) | ((q >> 2) & 1);
                        const int n = d.cp + (brq << (LOG2N - 3)) + r;
                        const float xv = __ldg(&xs[n]);
                        const float2 o = __ldg(&nco[n]);
                        float2 z = make_float2(__fmul_rn(o.x, xv), __fmul_rn(-o.y, xv));   // samples[i] * conj(osc) (:36)
                        if (rot) {
                            float sn, cs;
                            nl::sincosf_ref(theta[n], &sn, &cs);
                            z = cmul(z, make_float2(cs, sn));                               // mixed *= correction (:42)
                        }
                        v[q] = z;
                    }
                    stages_in_regs<3, 0, LOG2N>(v, 0, d.twiddle);
    #pragma unroll
                    for (int q = 0; q < 8; ++q) buf[PADIDX(8 * g + q)] = v[q];
                }
                PU_GSYNC();
                fft_pass_smem<3, 3, LOG2N>(buf, tid, d.twiddle);     // stages 4..6
                PU_GSYNC();
                if constexpr (NFFT == 512) {
                    fft_pass_smem<2, 6, LOG2N>(buf, tid, d.twiddle);          // stages 7..8: 128 groups of 4
                    fft_pass_smem<2, 6, LOG2N>(buf, tid + T, d.twiddle);
                } else {
                    fft_pass_smem<3, 6, LOG2N>(buf, tid, d.twiddle);          // stages 7..9
                }
                PU_GSYNC();
                // ---------------- last stage, only for the bins that are used
                for (int u = tid; u < nu; u += T) {
                    const int bin = u < nd ? d.data_bin[u] : d.pilot_bin[u - nd];
                    const int k = bin & (NFFT / 2 - 1);
                    const float2 w = __ldg(&d.twiddle[k]);
                    const float2 a = buf[PADIDX(k)];
                    const float2 t = cmul(w, buf[PADIDX(k + NFFT / 2)]);
                    const float2 out = (bin < NFFT / 2) ? cadd(a, t) : csub(a, t);
                    if (u < nd) S.Fd[u] = out;
                    else S.Fp[u - nd] = out;
                }
            }
        }
        PU_GSYNC();

        if (is_train) {
            // ---------------- estimateChannelFromLTS (channel_equalizer.cpp:137-194)
            if (!skip_fft) {
                for (int i = tid; i < nd; i += T)
                    if (s == training - 1) S.Hd[i] = cdiv(S.Fd[i], d.zc[i]);
                for (int i = tid; i < np; i += T)   // rx / (+-1, 0) accumulated over the training symbols
                    S.tmpc[i] = cadd(S.tmpc[i], make_float2(__fmul_rn(S.Fp[i].x, d.pilot_sign[i]), __fmul_rn(S.Fp[i].y, d.pilot_sign[i])));
            }
            if (s == training - 1) {
                PU_GSYNC();
                const float inv = __fdiv_rn(1.0f, static_cast<float>(training));
                for (int i = tid; i < np; i += T) S.Hp[i] = cscale(inv, S.tmpc[i]);
                for (int i = tid; i < nd; i += T) S.tmpa[i] = cabs_ref(S.Hd[i]);
                PU_GSYNC();
                if (tid == 0) {   // reporting-only SNR estimate (:208-225)
                    float sum = 0.0f;
                    for (int i = 0; i < nd; ++i) sum = __fadd_rn(sum, S.tmpa[i]);
                    const float avg = __fdiv_rn(sum, static_cast<float>(nd));
                    if (avg > 1e-6f && S.noise_var > 1e-10f)
                        S.snr_lin = clampf(0.1f, 10000.0f, __fdiv_rn(__fmul_rn(avg, avg), S.noise_var));
                    S.snr_cnt = training;   // :327
                }
            }
            PU_GSYNC();
            continue;
        }

        // ================= data symbol =================
        if (np > 0) {
            // ---------------- updateChannelEstimate (channel_equalizer.cpp:330-595)
            const float alpha = (S.snr_cnt == 0) ? 1.0f : 0.9f;
            for (int i = tid; i < np; i += T)
                S.hls[i] = make_float2(__fmul_rn(S.Fp[i].x, d.pilot_sign[i]), __fmul_rn(S.Fp[i].y, d.pilot_sign[i]));
            PU_GSYNC();
            if (tid == 0 && !S.cpc_init) {   // carrier phase lock on the first data symbol (:348-357)
                float2 sum = make_float2(0.0f, 0.0f);
                for (int i = 0; i < np; ++i) sum = cadd(sum, S.hls[i]);
                const float2 avg = cdivs(sum, static_cast<float>(np));
                const float mag = cabs_ref(avg);
                if (mag > 0.01f) {
                    S.cpc = cdivs(cconj(avg), mag);
                    S.cpc_init = 1;
                }
            }
            PU_GSYNC();
            const int have_prev = S.have_prev;
            for (int i = tid; i < np; i += T) {
                const float2 h = cmul(S.hls[i], S.cpc);   // :360-362
                S.hls[i] = h;
                const float nh = cnorm(h);
                S.tmpa[i] = nh;
                int v = 0;
                float dn = 0.0f;
                float2 unit = make_float2(0.0f, 0.0f);
                int vu = 0;
                if (have_prev) {
                    const float2 p = S.prevp[i];
                    const float npv = cnorm(p);
                    if (npv > 1e-6f && nh > 1e-6f) {
                        v = 1;
                        dn = cnorm(csub(h, p));                        // temporal noise (:402-406)
                        const float2 df = cmul(h, cconj(p));           // CFO phase step (:426-435)
                        const float mag = cabs_ref(df);
                        if (mag > 1e-6f) {
                            unit = cdivs(df, mag);
                            vu = 1;
                        }
                    }
                }
                S.tmpb[i] = dn;
                S.valid[i] = v | (vu << 1);
                S.tmpc[i] = unit;
                const float2 hold = S.Hp[i];
                S.Hp[i] = cadd(cscale(alpha, h), cscale(__fsub_rn(1.0f, alpha), hold));   // EMA (:410-411)
                if (S.snr_cnt >= 3 && nh >= 1e-6f) S.tmpd[i] = nl::atan2f_ref(h.y, h.x);          // std::arg for the timing fit (:483)
            }
            PU_GSYNC();
            if (tid == 0) {
                float sp_sum = 0.0f;
                for (int i = 0; i < np; ++i) sp_sum = __fadd_rn(sp_sum, S.tmpa[i]);
                const float signal_power = __fdiv_rn(sp_sum, static_cast<float>(np));
                float noise_sum = 0.0f;
                int noise_count = 0;
                for (int i = 0; i < np; ++i)
                    if (S.valid[i] & 1) { noise_sum = __fadd_rn(noise_sum, S.tmpb[i]); ++noise_count; }
                if (noise_count == 0) { noise_sum = __fdiv_rn(signal_power, 31.6f); noise_count = 1; }   // :415-418
                if (have_prev) {   // :421-467
                    float2 ps = make_float2(0.0f, 0.0f);
                    int vc = 0;
                    for (int i = 0; i < np; ++i)
                        if (S.valid[i] & 2) { ps = cadd(ps, S.tmpc[i]); ++vc; }
                    if (vc > 0) {
                        const float2 avg = cdivs(ps, static_cast<float>(vc));
                        const float apd = nl::atan2f_ref(avg.y, avg.x);
                        float sn, cs;
                        nl::sincosf_ref(-apd, &sn, &cs);
                        S.ppc = make_float2(cs, sn);
                        const float sym_dur = __fdiv_rn(static_cast<float>(d.sym_len), d.sample_rate);
                        const float residual = static_cast<float>(__ddiv_rn((double)apd, __dmul_rn(2.0f * 3.14159265358979323846, (double)sym_dur)));
                        const float total = __fadd_rn(S.cfo_hz, residual);
                        float a = 0.3f;
                        if (S.since_sync < 10) {
                            const float progress = __fdiv_rn(static_cast<float>(S.since_sync), 10.0f);
                            a = __fadd_rn(__fmul_rn(0.9f, __fsub_rn(1.0f, progress)), __fmul_rn(0.3f, progress));
                        }
                        if (fabsf(residual) > 10.0f) a = fmaxf(a, 0.9f);
                        S.since_sync++;
                        S.cfo_filt = __fadd_rn(__fmul_rn(a, total), __fmul_rn(__fsub_rn(1.0f, a), S.cfo_filt));
                        S.cfo_hz = clampf(-90.0f, 90.0f, S.cfo_filt);
                    }
                } else {
                    S.ppc = make_float2(1.0f, 0.0f);   // :468-470
                }
                if (S.snr_cnt >= 3) {   // timing slope by least squares over the pilots (:473-509)
                    float sk = 0.0f, sk2 = 0.0f, sph = 0.0f, skp = 0.0f;
                    int cnt = 0;
                    for (int i = 0; i < np; ++i) {
                        if (S.tmpa[i] < 1e-6f) continue;
                        int k = d.pilot_bin[i];
                        if (k > NFFT / 2) k -= NFFT;
                        const float ph = S.tmpd[i];
                        sk = __fadd_rn(sk, static_cast<float>(k));
                        sk2 = __fadd_rn(sk2, static_cast<float>(k * k));
                        sph = __fadd_rn(sph, ph);
                        skp = __fadd_rn(skp, __fmul_rn(static_cast<float>(k), ph));
                        ++cnt;
                    }
                    if (cnt >= 3) {
                        const float n = static_cast<float>(cnt);
                        const float den = __fsub_rn(__fmul_rn(n, sk2), __fmul_rn(sk, sk));
                        if (fabsf(den) > 1e-6f) {
                            const float slope = __fdiv_rn(__fsub_rn(__fmul_rn(n, skp), __fmul_rn(sk, sph)), den);
                            const float inst = static_cast<float>(__ddiv_rn((double)__fmul_rn(slope, static_cast<float>(NFFT)), 2.0f * 3.14159265358979323846));
                            float tm = __fadd_rn(__fmul_rn(0.3f, inst), __fmul_rn(__fsub_rn(1.0f, 0.3f), S.timing));
                            const float maxt = __fmul_rn(50.0f, __fdiv_rn(static_cast<float>(NFFT), 512.0f));
                            S.timing = clampf(-maxt, maxt, tm);
                        }
                    }
                }
                S.have_prev = 1;
                if (noise_count > 1 && noise_sum > 0.0f) {   // :584-592
                    float nv = __fdiv_rn(noise_sum, static_cast<float>(noise_count - 1));
                    if (nv < 1e-6f) nv = 1e-6f;
                    S.noise_var = nv;
                    const float inst = clampf(0.1f, 10000.0f, __fdiv_rn(signal_power, nv));
                    S.snr_lin = __fadd_rn(__fmul_rn(0.3f, inst), __fmul_rn(__fsub_rn(1.0f, 0.3f), S.snr_lin));
                }
                S.snr_cnt++;
            }
            for (int i = tid; i < np; i += T) S.prevp[i] = S.hls[i];   // :512
            PU_GSYNC();
            // coherent timing fix, interpolation, timing restore (:514-567, :601-631)
            const float timing = S.timing;
            const bool fix = !differential && fabsf(timing) > 0.1f;
            if (fix) {
                for (int i = tid; i < np; i += T) {
                    int k = d.pilot_bin[i];
                    if (k > NFFT / 2) k -= NFFT;
                    const float tp = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(2.0f * 3.14159265358979323846, (double)k), (double)timing), (double)static_cast<float>(NFFT)));
                    float sn, cs;
                    nl::sincosf_ref(-tp, &sn, &cs);                 // std::exp(Complex(0, -timing_phase))
                    S.Hp[i] = cmul(S.Hp[i], make_float2(cs, sn));
                }
                PU_GSYNC();
            }
            for (int i = tid; i < nd; i += T) {
                const int lo = d.interp_lo[i], hi = d.interp_hi[i];
                if (lo >= 0 && hi >= 0) {
                    const float2 H1 = S.Hp[lo], H2 = S.Hp[hi];
                    const float2 pd = cmul(H2, cconj(H1));
                    const float ph = fabsf(nl::atan2f_ref(pd.y, pd.x));
                    const float a = d.interp_alpha[i];
                    if (ph > 1.5708f) S.Hd[i] = (a < 0.5f) ? H1 : H2;
                    else S.Hd[i] = cadd(cscale(__fsub_rn(1.0f, a), H1), cscale(a, H2));
                } else if (lo >= 0) {
                    S.Hd[i] = S.Hp[lo];
                } else if (hi >= 0) {
                    S.Hd[i] = S.Hp[hi];
                }
            }
            if (fix) {
                PU_GSYNC();
                for (int u = tid; u < nu; u += T) {
                    int k = u < nd ? d.data_bin[u] : d.pilot_bin[u - nd];
                    if (k > NFFT / 2) k -= NFFT;
                    const float tp = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(2.0f * 3.14159265358979323846, (double)k), (double)timing), (double)static_cast<float>(NFFT)));
                    float sn, cs;
                    nl::sincosf_ref(tp, &sn, &cs);
                    if (u < nd) S.Hd[u] = cmul(S.Hd[u], make_float2(cs, sn));
                    else S.Hp[u - nd] = cmul(S.Hp[u - nd], make_float2(cs, sn));
                }
            }
            PU_GSYNC();
        }

        // ---------------- equalize (channel_equalizer.cpp:728-840)
        const float noise_var = S.noise_var;
        if (differential) {
            const float timing = S.timing;
            const float2 ppc = S.ppc;
            for (int i = tid; i < nd; i += T) {
                const float2 rx = S.Fd[i], h = S.Hd[i];
                const float hp = cnorm(h);
                int k = d.data_bin[i];
                if (k > NFFT / 2) k -= NFFT;
                const float tp = static_cast<float>(__ddiv_rn(__dmul_rn(__dmul_rn(2.0f * 3.14159265358979323846, (double)k), (double)timing), (double)static_cast<float>(NFFT)));
                float2 tc = make_float2(1.0f, 0.0f);       // std::exp(Complex(0, 0)) == (1, 0)
                if (tp != 0.0f) {
                    float sn, cs;
                    nl::sincosf_ref(tp, &sn, &cs);
                    tc = make_float2(cs, sn);
                }
                float2 e;
                float nv;
                if (hp > 1e-6f) {
                    e = cmul(cmul(cdivs(cmul(rx, cconj(h)), hp), ppc), tc);   // :761
                    nv = __fdiv_rn(noise_var, hp);
                } else {
                    e = cmul(cmul(rx, ppc), tc);
                    nv = 100.0f;
                }
                S.eq[i] = e;
                S.cnv[i] = clampf(1e-6f, 100.0f, nv);
            }
        } else {
            for (int i = tid; i < nd; i += T) {
                const float2 rx = S.Fd[i], h = S.Hd[i];
                const float hp = cnorm(h);
                S.tmpa[i] = hp;
                const float den = __fadd_rn(hp, noise_var);
                if (den < 1e-10f) {
                    S.eq[i] = make_float2(0.0f, 0.0f);
                    S.cnv[i] = 100.0f;
                } else {
                    S.eq[i] = cdivs(cmul(cconj(h), rx), den);                                          // MMSE (:815)
                    S.cnv[i] = clampf(1e-6f, 100.0f, __fdiv_rn(noise_var, __fadd_rn(hp, 1e-6f)));
                }
            }
            PU_GSYNC();
            if (tid == 0) {   // deep-fade erasure threshold (:823-830): ordered sum
                float sum = 0.0f;
                for (int i = 0; i < nd; ++i) sum = __fadd_rn(sum, S.tmpa[i]);
                S.tmpb[0] = __fmul_rn(0.1f, __fdiv_rn(sum, static_cast<float>(nd)));
            }
            PU_GSYNC();
            const float thr = S.tmpb[0];
            for (int i = tid; i < nd; i += T)
                if (S.tmpa[i] < thr) S.cnv[i] = 100.0f;
        }
        PU_GSYNC();

        // ---------------- debug dump of this symbol's intermediates (tests only)
        if (dbg) {
            const int sd = s - training;
            float* rec = dbg + (frame * static_cast<size_t>(n_symbols - training) + sd) * (4 * nu + 3 * nd + kDbgScalars);
            for (int u = tid; u < nu; u += T) {
                const float2 f = u < nd ? S.Fd[u] : S.Fp[u - nd];
                const float2 h = u < nd ? S.Hd[u] : S.Hp[u - nd];
                rec[2 * u] = f.x; rec[2 * u + 1] = f.y;
                rec[2 * nu + 2 * u] = h.x; rec[2 * nu + 2 * u + 1] = h.y;
            }
            for (int i = tid; i < nd; i += T) {
                rec[4 * nu + 2 * i] = S.eq[i].x; rec[4 * nu + 2 * i + 1] = S.eq[i].y;
                rec[4 * nu + 2 * nd + i] = S.cnv[i];
            }
            if (tid == 0) {
                float* sc = rec + 4 * nu + 3 * nd;
                sc[0] = S.cfo_used; sc[1] = S.cfo_hz; sc[2] = S.noise_var; sc[3] = S.timing; sc[4] = S.snr_lin;
                sc[5] = S.ppc.x; sc[6] = S.ppc.y; sc[7] = S.cpc.x; sc[8] = S.cpc.y; sc[9] = static_cast<float>(S.snr_cnt);
            }
        }

        // ---------------- demodulateSymbol (demodulator.cpp:279-356) + soft_demap.hpp
        float* out = llr_out + frame * llr_stride;
        for (int i = tid; i < nd; i += T) {
            const float2 sym = S.eq[i];
            const float nv = __fmul_rn(S.cnv[i], d.ce_margin);
            float l[8];
            int nb = d.bps;
            if (differential) {
                const float2 prev = S.preveq[i];
                const float2 df = cmul(sym, cconj(prev));
                const float sp = __fmul_rn(cabs_ref(sym), cabs_ref(prev));
                S.preveq[i] = sym;
#pragma unroll
                for (int b = 0; b < 3; ++b) l[b] = 0.0f;
                if (!(sp < 1e-6f)) {
                    const float phase = nl::atan2f_ref(df.y, df.x);
                    if (d.mod == PU_MOD_DBPSK) {              // soft_demap.hpp:173-187
                        l[0] = clip_llr(__fdiv_rn(__fmul_rn(__fmul_rn(2.0f, sp), nl::cosf_ref(phase)), nv));
                    } else if (d.mod == PU_MOD_DQPSK) {       // :192-213
                        const float scale = __fdiv_rn(__fmul_rn(2.0f, sp), nv);
                        const float pi = 3.14159265358979f;
                        l[0] = clip_llr(__fmul_rn(scale, nl::sinf_ref(__fadd_rn(phase, pi / 4))));
                        l[1] = clip_llr(__fmul_rn(scale, nl::cosf_ref(__fmul_rn(2.0f, phase))));
                    } else {                                  // D8PSK :217-237
                        const float conf = __fdiv_rn(sp, nv);
                        l[0] = clip_llr(__fmul_rn(conf, nl::sinf_ref(phase)));
                        l[1] = clip_llr(__fmul_rn(conf, nl::sinf_ref(__fmul_rn(2.0f, phase))));
                        l[2] = clip_llr(__fmul_rn(conf, nl::sinf_ref(__fmul_rn(4.0f, phase))));
                    }
                }
            } else {
                const float I = sym.x, Q = sym.y;
                switch (d.mod) {
                    case PU_MOD_BPSK:      // :37-39
                        l[0] = clip_llr(__fdiv_rn(__fmul_rn(-2.0f, I), nv));
                        break;
                    case PU_MOD_QAM16: {   // :49-64
                        const float sc = __fdiv_rn(2.0f, nv);
                        l[0] = clip_llr(__fmul_rn(-sc, I));
                        l[1] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(I), 0.6324555320336759f)));
                        l[2] = clip_llr(__fmul_rn(-sc, Q));
                        l[3] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(Q), 0.6324555320336759f)));
                        break;
                    }
                    case PU_MOD_QAM32: {   // :68-121 max-log over the 4(I) x 8(Q) grid; the 32 distances are shared by the 5 bits
                        const float sc = __fdiv_rn(2.0f, nv);
                        const float qs = 0.1961161351381840f;
                        float d0[5], d1[5];
#pragma unroll
                        for (int b = 0; b < 5; ++b) { d0[b] = 1e10f; d1[b] = 1e10f; }
#pragma unroll
                        for (int qi = 0; qi < 8; ++qi) {
                            const int qg = qi ^ (qi >> 1);   // Q_GRAY = {0,1,3,2,6,7,5,4}
                            const float dq = __fsub_rn(Q, __fmul_rn(static_cast<float>(2 * qi - 7), qs));
                            const float dq2 = __fmul_rn(dq, dq);
#pragma unroll
                            for (int ii = 0; ii < 4; ++ii) {
                                const int ig = ii ^ (ii >> 1);   // I_GRAY = {0,1,3,2}
                                const float di = __fsub_rn(I, __fmul_rn(static_cast<float>(2 * ii - 3), qs));
                                const float dist = __fadd_rn(__fmul_rn(di, di), dq2);
                                const int bits = (qg << 2) | ig;
#pragma unroll
                                for (int b = 0; b < 5; ++b) {
                                    if (bits & (1 << (4 - b))) d1[b] = fminf(d1[b], dist);
                                    else d0[b] = fminf(d0[b], dist);
                                }
                            }
                        }
#pragma unroll
                        for (int b = 0; b < 5; ++b) l[b] = clip_llr(__fmul_rn(sc, __fsub_rn(d1[b], d0[b])));
                        break;
                    }
                    case PU_MOD_QAM64: {   // :124-141
                        const float sc = __fdiv_rn(2.0f, nv);
                        const float D4 = 0.6172134f, D2 = 0.3086067f;
                        l[0] = clip_llr(__fmul_rn(-sc, I));
                        l[1] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(I), D4)));
                        l[2] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(__fsub_rn(fabsf(I), D4)), D2)));
                        l[3] = clip_llr(__fmul_rn(-sc, Q));
                        l[4] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(Q), D4)));
                        l[5] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(__fsub_rn(fabsf(Q), D4)), D2)));
                        break;
                    }
                    case PU_MOD_QAM256: {  // :144-163
                        const float sc = __fdiv_rn(2.0f, nv);
                        const float D8 = 0.5163978f, D4 = 0.2581989f, D2 = 0.1290994f;
                        const float a1 = __fsub_rn(fabsf(I), D8), a2 = __fsub_rn(fabsf(a1), D4);
                        const float b1 = __fsub_rn(fabsf(Q), D8), b2 = __fsub_rn(fabsf(b1), D4);
                        l[0] = clip_llr(__fmul_rn(-sc, I));
                        l[1] = clip_llr(__fmul_rn(sc, a1));
                        l[2] = clip_llr(__fmul_rn(sc, a2));
                        l[3] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(a2), D2)));
                        l[4] = clip_llr(__fmul_rn(-sc, Q));
                        l[5] = clip_llr(__fmul_rn(sc, b1));
                        l[6] = clip_llr(__fmul_rn(sc, b2));
                        l[7] = clip_llr(__fmul_rn(sc, __fsub_rn(fabsf(b2), D2)));
                        break;
                    }
                    default: {             // QPSK :42-45
                        const float sc = __fdiv_rn(__fmul_rn(-2.0f, 0.7071067811865476f), nv);
                        l[0] = clip_llr(__fmul_rn(I, sc));
                        l[1] = clip_llr(__fmul_rn(Q, sc));
                        nb = 2;
                    }
                }
            }
            const int base = llr_pos + i * nb;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                if (b < nb) {
                    const int pos = base + b;
                    if (pos < llr_limit) {
                        const int dst = (d.llr_perm && pos < d.perm_len) ? d.llr_perm[pos] : pos;
                        out[dst] = l[b];
                    }
                }
            }
        }
        llr_pos += nd * d.bps;
        PU_GSYNC();
    }
    if (tid == 0 && !no_frame) {
        if (snr_db_out) snr_db_out[frame] = 10.0f * log10f(S.snr_lin);   // getEstimatedSNR, demodulator.cpp:797-799
        if (final_cfo_out) final_cfo_out[frame] = S.cfo_hz;              // getFrequencyOffset, :801-803
    }
}

// ofdm_diff.cu
bool ofdm_diff_supported(const OfdmDev& d, int n_symbols, int training);
cudaError_t ofdm_diff_launch(const OfdmDev& d, const float2* host_twiddle, const float* samples, size_t B, size_t frame_stride,
                             int n_symbols, int training, float* llr, size_t llr_stride, int llr_limit, float* snr_db,
                             float* final_cfo, cudaStream_t st);
// ofdm_fast512.cu
bool ofdm_fast512_supported(const OfdmDev& d, int n_symbols, int training, const float* samples, size_t frame_stride, size_t B, size_t llr_stride);
cudaError_t ofdm_fast512_launch(const OfdmDev& d, const float* samples, size_t B, size_t frame_stride, int n_symbols, int training,
                                float* llr, size_t llr_stride, int llr_limit, float* snr_db, float* final_cfo, int sm_count, cudaStream_t st);

// ofdm_diff512.cu
bool ofdm_diff512_supported(const OfdmDev& d, int n_symbols, int training, const float* samples, size_t frame_stride, size_t B);
cudaError_t ofdm_diff512_launch(const OfdmDev& d, const float2* host_twiddle, const float* samples, size_t B, size_t frame_stride,
                                int n_symbols, int training, float* llr, size_t llr_stride, int llr_limit, float* snr_db,
                                float* final_cfo, int sm_count, cudaStream_t st);

// ofdm_acquire.cu
struct AcqDev {
    int nfft, log2n, cp, sym_len;
    float sample_rate, sync_threshold;
    const float2* twiddle;
    const float* lts_i;
    const float* lts_q;
    float lts_energy_ref;
    float lts_threshold;
};
cudaError_t ofdm_acquire_launch(const AcqDev& a, const float* samples, size_t B, size_t frame_stride, int L, int chunk, int4* out_int,
                                float* out_cfo, cudaStream_t st);

// ofdm_tx_gpu.cu
struct TxDev {
    int nfft, cp, sym_len, guard, n_data, n_pilot, bps, differential;
    int pre_len, n_sym, frame_len;
    int osc_start;
    float scale;
    int il_inv;
    LdpcEncDev enc;
    const int* data_bin;
    const int* pilot_bin;
    const float* pilot_sign;
    const float2* twiddle;
    const float2* osc;
    const float* preamble;
    const float2* points;
};
cudaError_t ofdm_tx_launch(const TxDev& t, const uint8_t* frames, size_t frame_stride, int frame_bytes, int n_cw, int bpc, size_t B, float peak,
                           float* out, size_t out_stride, cudaStream_t st);
std::vector<float> ofdm_modulate_frame(const OfdmPlan& p, int layout, const uint8_t* data, size_t n_bytes);   // ofdm_tx.cpp
cfloat ofdm_constellation_point(uint32_t bits, uint32_t mod);

// estimateCFOFromTraining(samples, num_symbols, coarse_cfo_hz = 0) (src/ofdm/ofdm_sync.cpp:278-380), what processPresynced runs when no
// CFO was set (demodulator.cpp:920-925): a LOCAL mixer (NCO restarted at phase 0 = the head of the tabulated oscillator) brings the first
// two training symbols to baseband, then P = sum conj(z1) z2, E1 = sum |z1|^2, E2 = sum |z2|^2 over their FFT parts -- ordered fp32 sums,
// one lane each -- quality gate |P| / sqrt(E1 E2 + 1e-10) >= 0.3, CFO = arg(P) fs / (2 pi sym_len) clamped to +- fs / (2 sym_len).
// One warp per frame; dynamic shared memory: 2 * nfft float2 per warp.
__global__ void ofdm_training_cfo_kernel(OfdmDev d, const float* __restrict__ samples, size_t frame_stride, size_t B, float* __restrict__ cfo_out) {
    extern __shared__ __align__(16) unsigned char tcfo_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t b = static_cast<size_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (b >= B) return;
    float2* z1 = reinterpret_cast<float2*>(tcfo_smem) + static_cast<size_t>(warp) * 2 * d.nfft;
    float2* z2 = z1 + d.nfft;
    const float* x = samples + b * frame_stride;
    for (int i = lane; i < d.nfft; i += 32) {
        const int n1 = d.cp + i, n2 = d.sym_len + d.cp + i;
        const float2 o1 = __ldg(&d.nco[n1]), o2 = __ldg(&d.nco[n2]);
        const float s1 = __ldg(&x[n1]), s2 = __ldg(&x[n2]);
        z1[i] = make_float2(__fmul_rn(o1.x, s1), __fmul_rn(-o1.y, s1));      // samples[i] * std::conj(osc)
        z2[i] = make_float2(__fmul_rn(o2.x, s2), __fmul_rn(-o2.y, s2));
    }
    __syncwarp();
    float2 P = make_float2(0.0f, 0.0f);
    float E = 0.0f;
    if (lane == 0) for (int i = 0; i < d.nfft; ++i) P = cadd(P, cmul(cconj(z1[i]), z2[i]));
    if (lane == 1) for (int i = 0; i < d.nfft; ++i) E = __fadd_rn(E, cnorm(z1[i]));
    if (lane == 2) for (int i = 0; i < d.nfft; ++i) E = __fadd_rn(E, cnorm(z2[i]));
    const float E1 = __shfl_sync(0xffffffffu, E, 1), E2 = __shfl_sync(0xffffffffu, E, 2);
    if (lane != 0) return;
    const float corr_mag = __fdiv_rn(cabs_ref(P), __fsqrt_rn(__fadd_rn(__fmul_rn(E1, E2), 1e-10f)));
    float cfo = 0.0f;
    if (corr_mag >= 0.3f) {
        const float phase = refmath::atan2f_ref(P.y, P.x);
        const double den = __dmul_rn(__dmul_rn(2.0, 3.14159265358979323846), static_cast<double>(d.sym_len));
        cfo = static_cast<float>(__ddiv_rn(static_cast<double>(__fmul_rn(phase, d.sample_rate)), den));
        const float max_cfo = __fdiv_rn(d.sample_rate, __fmul_rn(2.0f, static_cast<float>(d.sym_len)));
        cfo = fmaxf(-max_cfo, fminf(max_cfo, cfo));
    }
    cfo_out[b] = cfo;
}

// frame windows of acquired frames: data symbols start at data_start and run to the end of the row
__global__ void acquire_windows_kernel(const int4* __restrict__ acq, size_t B, int L, int sym_len, int llr_per_symbol, int llr_stride,
                                       int* __restrict__ start, int* __restrict__ nsym, int* __restrict__ n_llr) {
    const size_t b = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (b >= B) return;
    const int4 a = acq[b];
    const int n = a.x ? max(0, (L - a.z) / sym_len) : 0;
    start[b] = a.x ? a.z : 0;
    nsym[b] = n;
    if (n_llr) n_llr[b] = min(n * llr_per_symbol, llr_stride);
}

}  // namespace pu

void pu_ldpc_encoder_view(const pu_ldpc* h, int* k, int* m, const uint8_t** cn_ninfo, const uint16_t** cn_check, const uint16_t** cn_var);   // ldpc_decode.cu

struct pu_ofdm {
    pu_ctx* ctx = nullptr;
    int device = 0;   // copy of ctx->device: the handle may outlive its context
    pu::OfdmPlan plan;
    pu::OfdmDev dev{};
    pu::DevMem d_tw, d_nco, d_dbin, d_pbin, d_zc, d_psign, d_ilo, d_ihi, d_ia, d_perm;
    pu::DevMem d_lts_i, d_lts_q;          // LTS passband templates of refineLTSTiming (built on first use)
    pu::DevMem d_chirp;                   // dual-chirp templates: up sin, up cos, down sin, down cos (built on first use)
    pu::ChirpDev chirp{};
    bool chirp_ready = false;

    // sync::ChirpSync::generateTemplate (src/sync/chirp_sync.hpp:706-735) with OFDMChirpWaveform::getChirpConfig
    // (src/waveform/ofdm_chirp_waveform.cpp:39-49): 300 -> 2700 Hz in 500 ms, 100 ms gaps
    pu_status ensure_chirp() {
        if (chirp_ready) return PU_OK;
        std::vector<float> t;
        pu::chirp_templates_host(static_cast<float>(plan.cfg.sample_rate), t, chirp);
        pu_status st = d_chirp.upload(t.data(), t.size());
        if (st != PU_OK) return st;
        pu::chirp_dev_bind(chirp, static_cast<const float*>(d_chirp.p));
        chirp_ready = true;
        return PU_OK;
    }
    pu::DevMem d_tx_osc, d_tx_pre[2], d_tx_points;   // transmitter tables (built on first use; preamble per layout)
    int tx_pre_len[2] = {-1, -1};
    size_t tx_osc_len = 0;
    int tx_il_inv = 0;                               // pu_ofdm_set_tx_interleave (TxDev::il_inv)
    pu::AcqDev acq{};
    bool acq_ready = false;

    // generateSequences (src/ofdm/demodulator.cpp:99-132): LTS in the frequency domain -> inverse FFT -> cyclic prefix ->
    // passband templates; energy_ref as refineLTSTiming accumulates it (ofdm_sync.cpp:405-411)
    pu_status ensure_acquire() {
        if (acq_ready) return PU_OK;
        const pu::OfdmPlan& p = plan;
        std::vector<pu::cfloat> f(p.nfft, pu::cfloat(0, 0));
        for (size_t i = 0; i < p.data_bin.size(); ++i) f[p.data_bin[i]] = p.sync_seq[i % p.sync_seq.size()];
        for (size_t i = 0; i < p.pilot_bin.size(); ++i) f[p.pilot_bin[i]] = pu::cfloat(p.pilot_sign[i], 0.0f);
        const size_t n = f.size();
        for (size_t i = 0, rev = 0; i + 1 < n; ++i) {          // fft_impl(inverse), src/dsp/fft.cpp:89-121
            if (i < rev) std::swap(f[i], f[rev]);
            size_t bit = n >> 1;
            while (bit <= rev) { rev -= bit; bit >>= 1; }
            rev += bit;
        }
        for (size_t span = 2; span <= n; span <<= 1) {
            const size_t half = span >> 1, stride = n / span;
            for (size_t blk = 0; blk < n; blk += span)
                for (size_t k = 0; k < half; ++k) {
                    const pu::cfloat t = std::conj(p.twiddle[k * stride]) * f[blk + k + half];
                    f[blk + k + half] = f[blk + k] - t;
                    f[blk + k] = f[blk + k] + t;
                }
        }
        const float scale = 1.0f / static_cast<float>(n);
        for (auto& v : f) v *= scale;
        const int P = p.nfft + p.cp;
        std::vector<pu::cfloat> osc = p.nco(static_cast<float>(p.cfg.center_freq), static_cast<size_t>(P) + 1);
        std::vector<float> li(P), lq(P);
        for (int i = 0; i < P; ++i) {
            const pu::cfloat bb = i < p.cp ? f[p.nfft - p.cp + i] : f[i - p.cp];
            const pu::cfloat mixed = bb * osc[i];
            li[i] = mixed.real();
            lq[i] = mixed.imag();
        }
        float e = 0.0f;
        for (int i = 0; i < P; ++i) { e += li[i] * li[i]; e += lq[i] * lq[i]; }
        e *= 0.5f;
        pu_status st;
        if ((st = d_lts_i.upload(li.data(), li.size())) != PU_OK) return st;
        if ((st = d_lts_q.upload(lq.data(), lq.size())) != PU_OK) return st;
        acq.nfft = p.nfft; acq.log2n = p.log2n; acq.cp = p.cp; acq.sym_len = p.sym_len;
        acq.sample_rate = static_cast<float>(p.cfg.sample_rate);
        acq.sync_threshold = 0.80f;                              // ModemConfig::sync_threshold default, include/ultra/types.hpp:188
        acq.twiddle = static_cast<const float2*>(d_tw.p);
        acq.lts_i = static_cast<const float*>(d_lts_i.p);
        acq.lts_q = static_cast<const float*>(d_lts_q.p);
        acq.lts_energy_ref = e;
        acq.lts_threshold = p.nfft >= 1024 ? 0.05f : 0.35f;      // ofdm_sync.cpp:451
        acq_ready = true;
        return PU_OK;
    }
    int max_symbols = 0;
    int last_kernel = 0;
    int precision = PU_PRECISION_EXACT;
    bool fast() const { return precision == PU_PRECISION_FAST; }
    size_t smem_bytes = 0;

    pu_status ensure_nco(int n_symbols) {
        if (n_symbols <= max_symbols) return PU_OK;
        const int want = std::max(n_symbols, 32);
        std::vector<pu::cfloat> t = plan.nco(static_cast<float>(plan.cfg.center_freq), static_cast<size_t>(want + 1) * plan.sym_len);
        pu_status s = d_nco.upload(t.data(), static_cast<size_t>(want) * plan.sym_len);
        if (s != PU_OK) return s;
        dev.nco = static_cast<const float2*>(d_nco.p);
        dev.nco_len = want * plan.sym_len;
        max_symbols = want;
        return PU_OK;
    }
};

extern "C" {

pu_status pu_ofdm_create(pu_ctx* ctx, const pu_modem_config* cfg, pu_ofdm** out) {
    PU_REQUIRE(ctx && cfg && out, "pu_ofdm_create: NULL argument");
    *out = nullptr;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    std::unique_ptr<pu_ofdm> h(new (std::nothrow) pu_ofdm());
    if (!h) return PU_ERR_NOMEM;
    h->ctx = ctx;
    h->device = ctx->device;
    const char* why = "";
    if (!pu::make_ofdm_plan(*cfg, &h->plan, &why)) {
        pu::set_error("pu_ofdm_create: %s", why);
        return PU_ERR_UNSUPPORTED;
    }
    const pu::OfdmPlan& p = h->plan;
    std::vector<pu::cfloat> zc(p.n_data);
    for (int i = 0; i < p.n_data; ++i) zc[i] = p.sync_seq[i % p.cfg.num_carriers];   // channel_equalizer.cpp:141
    pu_status s;
    if ((s = h->d_tw.upload(p.twiddle.data(), p.twiddle.size())) != PU_OK) return s;
    if ((s = h->d_dbin.upload(p.data_bin.data(), p.data_bin.size())) != PU_OK) return s;
    if ((s = h->d_pbin.upload(p.pilot_bin.data(), p.pilot_bin.size())) != PU_OK) return s;
    if ((s = h->d_zc.upload(zc.data(), zc.size())) != PU_OK) return s;
    if ((s = h->d_psign.upload(p.pilot_sign.data(), p.pilot_sign.size())) != PU_OK) return s;
    if ((s = h->d_ilo.upload(p.interp_lo.data(), p.interp_lo.size())) != PU_OK) return s;
    if ((s = h->d_ihi.upload(p.interp_hi.data(), p.interp_hi.size())) != PU_OK) return s;
    if ((s = h->d_ia.upload(p.interp_alpha.data(), p.interp_alpha.size())) != PU_OK) return s;
    pu::OfdmDev& d = h->dev;
    d.nfft = p.nfft; d.log2n = p.log2n; d.cp = p.cp; d.sym_len = p.sym_len;
    d.n_data = p.n_data; d.n_pilot = p.n_pilot; d.bps = p.bps; d.mod = static_cast<int>(p.cfg.modulation);
    d.ce_margin = p.ce_margin;
    d.sample_rate = static_cast<float>(p.cfg.sample_rate);
    d.twiddle = static_cast<const float2*>(h->d_tw.p);
    d.data_bin = static_cast<const int*>(h->d_dbin.p);
    d.pilot_bin = static_cast<const int*>(h->d_pbin.p);
    d.zc = static_cast<const float2*>(h->d_zc.p);
    d.pilot_sign = static_cast<const float*>(h->d_psign.p);
    d.interp_lo = static_cast<const int*>(h->d_ilo.p);
    d.interp_hi = static_cast<const int*>(h->d_ihi.p);
    d.interp_alpha = static_cast<const float*>(h->d_ia.p);
    d.llr_perm = nullptr;
    d.perm_len = 0;
    h->smem_bytes = sizeof(float2) * (p.nfft + p.nfft / 8) + sizeof(float) * ((p.sym_len + 3) & ~3) + sizeof(pu::RxShared);
    if ((s = h->ensure_nco(32)) != PU_OK) return s;
    *out = h.release();
    return PU_OK;
}

void pu_ofdm_destroy(pu_ofdm* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h;
}

int pu_ofdm_symbol_samples(const pu_ofdm* h) { return h ? h->plan.sym_len : -1; }
int pu_ofdm_data_carriers(const pu_ofdm* h) { return h ? h->plan.n_data : -1; }
int pu_ofdm_pilot_carriers(const pu_ofdm* h) { return h ? h->plan.n_pilot : -1; }
int pu_ofdm_bits_per_symbol(const pu_ofdm* h) { return h ? h->plan.n_data * h->plan.bps : -1; }
int pu_ofdm_last_kernel(const pu_ofdm* h) { return h ? h->last_kernel : -1; }

int pu_ofdm_carrier_bins(const pu_ofdm* h, int32_t* bins, int cap) {
    if (!h) return -1;
    int n = 0;
    for (int b : h->plan.data_bin) { if (n < cap) bins[n] = b; ++n; }
    for (int b : h->plan.pilot_bin) { if (n < cap) bins[n] = b; ++n; }
    return n;
}

pu_status pu_ofdm_set_precision(pu_ofdm* h, pu_precision mode) {
    PU_REQUIRE(h, "pu_ofdm_set_precision: NULL handle");
    PU_REQUIRE(mode == PU_PRECISION_EXACT || mode == PU_PRECISION_FAST, "pu_ofdm_set_precision: unknown mode");
    h->precision = mode;
    return PU_OK;
}
int pu_ofdm_get_precision(const pu_ofdm* h) { return h ? (h->fast() ? PU_PRECISION_FAST : PU_PRECISION_EXACT) : -1; }

pu_status pu_ofdm_set_deinterleave(pu_ofdm* h, size_t bits_per_symbol, size_t total_bits) {
    PU_REQUIRE(h, "pu_ofdm_set_deinterleave: NULL handle");
    PU_CUDA_TRY(cudaSetDevice(h->ctx->device));
    if (bits_per_symbol == 0) {
        h->dev.llr_perm = nullptr;
        h->dev.perm_len = 0;
        return PU_OK;
    }
    // ChannelInterleaver::deinterleave: output[inverse_permutation_[i]] = soft_bits[i] (ldpc_decoder.cpp:612-620)
    std::vector<uint32_t> perm(total_bits), inv(total_bits);
    pu_status s = pu_channel_interleaver_perm(bits_per_symbol, total_bits, perm.data(), inv.data(), nullptr);
    if (s != PU_OK) return s;
    std::vector<int> dst(inv.begin(), inv.end());
    if ((s = h->d_perm.upload(dst.data(), dst.size())) != PU_OK) return s;
    h->dev.llr_perm = static_cast<const int*>(h->d_perm.p);
    h->dev.perm_len = static_cast<int>(total_bits);
    return PU_OK;
}

pu_status pu_ofdm_set_tx_interleave(pu_ofdm* h, size_t bits_per_symbol) {
    PU_REQUIRE(h, "pu_ofdm_set_tx_interleave: NULL handle");
    h->tx_il_inv = bits_per_symbol ? static_cast<int>(pu::channel_interleaver_inverse_step(bits_per_symbol)) : 0;
    return PU_OK;
}

static pu_status launch_ofdm(pu_ofdm* h, const float* d_samples, size_t B, size_t L, int training,
                             const float* d_cfo, const float* d_phase, float* d_llr, size_t llr_stride,
                             float* d_snr, float* d_fcfo, float* d_dbg, cudaStream_t st,
                             const int* d_fstart = nullptr, const int* d_fnsym = nullptr) {
    const pu::OfdmPlan& p = h->plan;
    const int n_symbols = static_cast<int>(L / p.sym_len);
    pu_status s = h->ensure_nco(n_symbols);
    if (s != PU_OK) return s;
    const int total_llr = std::max(0, n_symbols - training) * p.n_data * p.bps;
    const int limit = static_cast<int>(std::min<size_t>(llr_stride, static_cast<size_t>(total_llr)));
    const unsigned grid = static_cast<unsigned>(B);
    (void)cudaGetLastError();
    if (!d_fstart && !d_fnsym && !d_cfo && !d_phase && !d_dbg && pu::ofdm_diff_supported(h->dev, n_symbols, training) &&
        pu::ofdm_diff512_supported(h->dev, n_symbols, training, d_samples, L, B)) {
        if (h->fast() && pu::ofdm_fast512_supported(h->dev, n_symbols, training, d_samples, L, B, llr_stride)) {
            // PU_PRECISION_FAST: the same pipeline with FMA-contracted butterflies (ofdm_fast512.cu)
            const cudaError_t e = pu::ofdm_fast512_launch(h->dev, d_samples, B, L, n_symbols, training, d_llr, llr_stride, limit, d_snr, d_fcfo,
                                                          h->ctx->sm_count, st);
            h->last_kernel = 5;
            h->ctx->launches.fetch_add(1);
            PU_CUDA_TRY(e);
            return PU_OK;
        }
        // 512-FFT differential no-pilot mode: persistent TMA-staged packed-fp32 kernel (ofdm_diff512.cu)
        const cudaError_t e = pu::ofdm_diff512_launch(h->dev, reinterpret_cast<const float2*>(p.twiddle.data()), d_samples, B, L, n_symbols,
                                                      training, d_llr, llr_stride, limit, d_snr, d_fcfo, h->ctx->sm_count, st);
        h->last_kernel = 3;
        h->ctx->launches.fetch_add(1);
        PU_CUDA_TRY(e);
        return PU_OK;
    }
    if (!d_fstart && !d_fnsym && !d_cfo && !d_phase && !d_dbg && pu::ofdm_diff_supported(h->dev, n_symbols, training)) {
        // differential no-pilot mode with setFrequencyOffset(0): symbols are independent -> warp-FFT kernel (ofdm_diff.cu)
        static_assert(sizeof(pu::cfloat) == sizeof(float2), "twiddle layout");
        const cudaError_t e = pu::ofdm_diff_launch(h->dev, reinterpret_cast<const float2*>(p.twiddle.data()), d_samples, B, L, n_symbols,
                                                   training, d_llr, llr_stride, limit, d_snr, d_fcfo, st);
        h->last_kernel = 2;
        h->ctx->launches.fetch_add(1);
        PU_CUDA_TRY(e);
        return PU_OK;
    }
    pu::WgTw twa;
    for (int m = 0; m < 16; ++m) {
        const pu::cfloat w = (32 * m < p.nfft / 2) ? p.twiddle[32 * m] : pu::cfloat(0.0f, 0.0f);
        twa.a[m] = make_float2(w.real(), w.imag());
    }
    // Warp-granular variant (one frame per warp): needs every used bin within +-CW of DC (the pruned pass B of the warp FFT)
    const int cw = p.nfft == 512 ? 16 : 32;
    bool near_dc = true;
    for (int b : p.data_bin) near_dc = near_dc && ((b >= 1 && b < cw) || b > p.nfft - cw);
    for (int b : p.pilot_bin) near_dc = near_dc && ((b >= 1 && b < cw) || b > p.nfft - cw);
    if (!d_dbg && near_dc) {
        // one CTA per SM with as many frames as shared memory holds, warps re-aligned at every symbol (r29: M3 32QAM 3.16 -> 2.49 ms,
        // M1 16QAM 7.19 -> 6.08 ms per 53k frames against small CTAs of 3-4 warps without the barrier)
        const int warps = p.nfft == 512 ? 16 : 14;
        const size_t buf_f2 = static_cast<size_t>(p.nfft + (p.nfft >> (p.nfft == 512 ? 4 : 5)) + 2 * cw);
        const unsigned group = static_cast<unsigned>((buf_f2 * sizeof(float2) + sizeof(pu::RxShared) + 15) & ~size_t(15));
        const unsigned wgrid = static_cast<unsigned>((B + warps - 1) / warps);
        const bool diff = pu::is_differential(p.cfg.modulation);
        using WK = void (*)(pu::OfdmDev, pu::WgTw, const float*, size_t, size_t, int, int, const float*, const float*, float*, size_t, int,
                            float*, float*, float*, unsigned, const int*, const int*);
        const bool fastk = h->fast();     // PU_PRECISION_FAST: FMA butterflies + MUFU rotator sin/cos (see the kernel's FAST parameter)
        const WK wk = fastk ? (p.nfft == 512 ? (diff ? pu::ofdm_presynced_kernel<512, true, 1, true> : pu::ofdm_presynced_kernel<512, true, 2, true>)
                                             : (diff ? pu::ofdm_presynced_kernel<1024, true, 1, true> : pu::ofdm_presynced_kernel<1024, true, 2, true>))
                            : (p.nfft == 512 ? (diff ? pu::ofdm_presynced_kernel<512, true, 1> : pu::ofdm_presynced_kernel<512, true, 2>)
                                             : (diff ? pu::ofdm_presynced_kernel<1024, true, 1> : pu::ofdm_presynced_kernel<1024, true, 2>));
        static std::atomic<uint64_t> attrw[8];      // per kernel instance, one bit per device (pu_async.cuh: smem_optin)
        PU_CUDA_TRY(pu::smem_optin(attrw[(fastk ? 4 : 0) + (p.nfft == 512 ? 0 : 2) + (diff ? 0 : 1)], wk, 232448));
        wk<<<wgrid, warps * 32, static_cast<size_t>(warps) * group, st>>>(h->dev, twa, d_samples, L, B, n_symbols, training, d_cfo, d_phase, d_llr,
                                                                           llr_stride, limit, d_snr, d_fcfo, nullptr, group, d_fstart, d_fnsym);
        h->last_kernel = fastk ? 6 : 4;
        h->ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        return PU_OK;
    }
    if (p.nfft == 512) {
        static std::atomic<uint64_t> attr512{0};
        PU_CUDA_TRY(pu::smem_optin(attr512, pu::ofdm_presynced_kernel<512, false, 0>, 65536));
        pu::ofdm_presynced_kernel<512, false, 0><<<grid, 64, h->smem_bytes, st>>>(h->dev, twa, d_samples, L, B, n_symbols, training, d_cfo, d_phase,
                                                                            d_llr, llr_stride, limit, d_snr, d_fcfo, d_dbg, 0u, d_fstart, d_fnsym);
    } else {
        static std::atomic<uint64_t> attr1024{0};
        PU_CUDA_TRY(pu::smem_optin(attr1024, pu::ofdm_presynced_kernel<1024, false, 0>, 65536));
        pu::ofdm_presynced_kernel<1024, false, 0><<<grid, 128, h->smem_bytes, st>>>(h->dev, twa, d_samples, L, B, n_symbols, training, d_cfo, d_phase,
                                                                              d_llr, llr_stride, limit, d_snr, d_fcfo, d_dbg, 0u, d_fstart, d_fnsym);
    }
    h->last_kernel = 1;
    h->ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_ofdm_presynced_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, int training_symbols,
                                  const float* cfo_hz, const float* cfo_phase, float* llr_out, size_t llr_stride,
                                  float* snr_db, float* final_cfo_hz, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ofdm_presynced_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && llr_out, "pu_ofdm_presynced_batch: NULL data pointer");
    PU_REQUIRE(training_symbols >= 0, "pu_ofdm_presynced_batch: negative training_symbols");
    const pu::OfdmPlan& p = h->plan;
    PU_REQUIRE(L >= static_cast<size_t>(p.sym_len) * static_cast<size_t>(training_symbols),
               "pu_ofdm_presynced_batch: frame shorter than its training symbols");
    PU_REQUIRE(llr_stride > 0, "pu_ofdm_presynced_batch: llr_stride is zero");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_DEVICE)
        return launch_ofdm(h, samples, B, L, training_symbols, cfo_hz, cfo_phase, llr_out, llr_stride, snr_db, final_cfo_hz, nullptr, st);

    pu::HostStage hs(ctx, st, B);
    const float *d_x, *d_cfo, *d_ph;
    float *d_llr, *d_snr, *d_fcfo;
    hs.in(&d_x, samples, L);
    hs.in(&d_cfo, cfo_hz, 1);
    hs.in(&d_ph, cfo_phase, 1);
    hs.out(&d_llr, llr_out, llr_stride);
    hs.out(&d_snr, snr_db, 1);
    hs.out(&d_fcfo, final_cfo_hz, 1);
    return hs.run([&](size_t nb) {
        return launch_ofdm(h, d_x, nb, L, training_symbols, d_cfo, d_ph, d_llr, llr_stride, d_snr, d_fcfo, nullptr, st);
    });
}

pu_status pu_ofdm_chirp_receive_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, float threshold, float* llr_out,
                                      size_t llr_stride, int32_t* n_llr, int32_t* sync_info, float* sync_values, float* snr_db,
                                      pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ofdm_chirp_receive_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && sync_info && sync_values, "pu_ofdm_chirp_receive_batch: NULL data pointer");
    PU_REQUIRE(!llr_out || (n_llr && llr_stride > 0), "pu_ofdm_chirp_receive_batch: llr_out needs n_llr and llr_stride");
    PU_REQUIRE(L < (1u << 30), "pu_ofdm_chirp_receive_batch: frame too long");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu_status s = h->ensure_chirp();
    if (s != PU_OK) return s;
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const pu::OfdmPlan& p = h->plan;
    if (threshold <= 0.0f) threshold = 0.15f;        // the callers' value, tools/test_iwaveform.cpp:133
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float* d_x;
        float *d_val, *d_llr, *d_snr;
        int32_t *d_info, *d_n;
        hs.in(&d_x, samples, L);
        hs.out(&d_info, sync_info, 4);
        hs.out(&d_val, sync_values, 4);
        hs.out(&d_llr, llr_out, llr_stride);
        hs.out(&d_n, llr_out ? n_llr : nullptr, 1);
        hs.out(&d_snr, llr_out ? snr_db : nullptr, 1);
        return hs.run([&](size_t nb) {
            return pu_ofdm_chirp_receive_batch(h, d_x, nb, L, threshold, d_llr, llr_stride, d_n, d_info, d_val, d_snr, PU_MEM_DEVICE, st);
        });
    }
    pu::DevMem dstart, dnsym, dcfo, dph;
    std::vector<int32_t> zi(B, 0);
    if ((s = dstart.upload(zi.data(), B)) != PU_OK) return s;
    if ((s = dnsym.upload(zi.data(), B)) != PU_OK) return s;
    if ((s = dcfo.upload(zi.data(), B)) != PU_OK) return s;
    if ((s = dph.upload(zi.data(), B)) != PU_OK) return s;
    (void)cudaGetLastError();
    PU_CUDA_TRY(pu::chirp_detect_launch(h->chirp, samples, B, L, static_cast<int>(L), threshold, p.sym_len, reinterpret_cast<int4*>(sync_info),
                                        reinterpret_cast<float4*>(sync_values), static_cast<int*>(dstart.p), static_cast<int*>(dnsym.p),
                                        static_cast<float*>(dcfo.p), static_cast<float*>(dph.p), llr_out ? n_llr : nullptr, p.n_data * p.bps,
                                        static_cast<int>(llr_stride), st));
    ctx->launches.fetch_add(1);
    if (llr_out) {
        // OFDMChirpWaveform::process (:170-199): setFrequencyOffsetWithPhase(cfo, accumulated phase); processPresynced(span, 2)
        s = launch_ofdm(h, samples, B, L, 2, static_cast<const float*>(dcfo.p), static_cast<const float*>(dph.p), llr_out, llr_stride, snr_db, nullptr,
                        nullptr, st, static_cast<const int*>(dstart.p), static_cast<const int*>(dnsym.p));
        if (s != PU_OK) return s;
    }
    PU_CUDA_TRY(cudaStreamSynchronize(st));           // the scratch buffers above are freed on return
    return PU_OK;
}

pu_status pu_chirp_phase_cycles(uint64_t cycles[8]) {
    PU_REQUIRE(cycles, "pu_chirp_phase_cycles: NULL output");
    unsigned long long v[8] = {};
    PU_CUDA_TRY(pu::chirp_phase_cycles(v));
    for (int i = 0; i < 8; ++i) cycles[i] = v[i];
    return PU_OK;
}

pu_status pu_chirp_search_stats(uint64_t* searches, uint64_t* rounds, uint64_t* fine_runs) {
    unsigned long long v[3] = {0, 0, 0};
    PU_CUDA_TRY(pu::chirp_search_stats(v));
    if (searches) *searches = v[0];
    if (rounds) *rounds = v[1];
    if (fine_runs) *fine_runs = v[2];
    return PU_OK;
}

pu_status pu_chirp_generate(float sample_rate, float tx_cfo_hz, float* out, size_t out_cap, size_t* out_len) {
    PU_REQUIRE(out_len && sample_rate > 0, "pu_chirp_generate: bad argument");
    // sync::ChirpSync::generate (src/sync/chirp_sync.hpp:58-108), host side: [up chirp][gap][down chirp][gap]
    const float f_start = 300.0f, f_end = 2700.0f, duration_ms = 500.0f, gap_ms = 100.0f, amplitude = 0.5f;
    const size_t n = static_cast<size_t>(sample_rate * duration_ms / 1000.0f), gap = static_cast<size_t>(sample_rate * gap_ms / 1000.0f);
    const size_t total = 2 * n + 2 * gap;
    *out_len = total;
    if (!out) return PU_OK;
    PU_REQUIRE(out_cap >= total, "pu_chirp_generate: output buffer too small");
    std::fill(out, out + total, 0.0f);
    const float T = duration_ms / 1000.0f, k = (f_end - f_start) / T;
    const float fu = f_start + tx_cfo_hz, fd = f_end + tx_cfo_hz;
    for (size_t i = 0; i < n; ++i) {
        const float t = static_cast<float>(i) / sample_rate;
        const float phase = static_cast<float>(2.0f * 3.14159265358979323846 * (fu * t + 0.5f * k * t * t));
        out[i] = amplitude * std::sin(phase);
    }
    for (size_t i = 0; i < n; ++i) {
        const float t = static_cast<float>(i) / sample_rate;
        const float phase = static_cast<float>(2.0f * 3.14159265358979323846 * (fd * t - 0.5f * k * t * t));
        out[n + gap + i] = amplitude * std::sin(phase);
    }
    return PU_OK;
}

}  // extern "C"

namespace pu {
namespace {
// The transmitter behind pu_ofdm_tx_batch (n_cw = 1, bpc = k / 8) and pu_frame_tx_batch: B frames of frame_bytes bytes -> n_cw codewords
// each (bpc frame bytes in CW0) -> one OFDM frame per row.  B == 0 or out == NULL: *frame_len only.
pu_status ofdm_tx_frames(pu_ofdm* h, const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes, int n_cw, int bpc, size_t B,
                         int layout, float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream) {
    const pu::OfdmPlan& p = h->plan;
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu::TxDev t{};
    pu_ldpc_encoder_view(code, &t.enc.k, &t.enc.m, &t.enc.cn_ninfo, &t.enc.cn_check, &t.enc.cn_var);
    pu_status s;
    if (h->tx_pre_len[layout] < 0) {                 // generateTrainingSymbols / generatePreamble: payload independent
        std::vector<float> pre = pu::ofdm_modulate_frame(p, layout, nullptr, 0);
        if ((s = h->d_tx_pre[layout].upload(pre.data(), pre.size())) != PU_OK) return s;
        h->tx_pre_len[layout] = static_cast<int>(pre.size());
    }
    if (!h->d_tx_points.p) {
        const uint32_t mod = p.cfg.modulation;
        std::vector<pu::cfloat> pts(static_cast<size_t>(1) << p.bps);
        for (uint32_t v = 0; v < pts.size(); ++v) {
            if (mod == PU_MOD_DBPSK) pts[v] = (v & 1) ? pu::cfloat(-1, 0) : pu::cfloat(1, 0);
            else if (mod == PU_MOD_DQPSK) { static const pu::cfloat st4[4] = {{1, 0}, {0, 1}, {-1, 0}, {0, -1}}; pts[v] = st4[v & 3]; }
            else if (mod == PU_MOD_D8PSK) {
                const float pi = 3.14159265358979f;
                const float ang = static_cast<float>(v & 7) * (pi / 4.0f) + pi / 8.0f;
                pts[v] = pu::cfloat(std::cos(ang), std::sin(ang));
            } else pts[v] = pu::ofdm_constellation_point(v, mod);
        }
        if ((s = h->d_tx_points.upload(pts.data(), pts.size())) != PU_OK) return s;
    }
    const int per_sym = p.n_data * p.bps;
    t.n_sym = (n_cw * PU_LDPC_N + per_sym - 1) / per_sym;
    t.pre_len = h->tx_pre_len[layout];
    t.frame_len = t.pre_len + t.n_sym * p.sym_len;
    *frame_len = static_cast<size_t>(t.frame_len);
    if (B == 0 || !out) return PU_OK;                // length query
    PU_REQUIRE(frames && out_stride >= static_cast<size_t>(t.frame_len), "pu_ofdm_tx_batch: output rows shorter than a frame");
    t.osc_start = layout == 0 ? t.pre_len : 2 * (p.nfft + p.cp);
    if (h->tx_osc_len < static_cast<size_t>(t.frame_len)) {
        std::vector<pu::cfloat> osc = p.nco(static_cast<float>(p.cfg.center_freq) + p.cfg.tx_cfo_hz, static_cast<size_t>(t.frame_len) + 1);
        if ((s = h->d_tx_osc.upload(osc.data(), static_cast<size_t>(t.frame_len))) != PU_OK) return s;
        h->tx_osc_len = static_cast<size_t>(t.frame_len);
    }
    t.nfft = p.nfft; t.cp = p.cp; t.sym_len = p.sym_len; t.guard = static_cast<int>(p.cfg.symbol_guard);
    t.n_data = p.n_data; t.n_pilot = p.n_pilot; t.bps = p.bps; t.differential = pu::is_differential(p.cfg.modulation) ? 1 : 0;
    t.scale = p.cfg.output_scale;
    t.il_inv = h->tx_il_inv;
    t.data_bin = static_cast<const int*>(h->d_dbin.p); t.pilot_bin = static_cast<const int*>(h->d_pbin.p);
    t.pilot_sign = static_cast<const float*>(h->d_psign.p); t.twiddle = static_cast<const float2*>(h->d_tw.p);
    t.osc = static_cast<const float2*>(h->d_tx_osc.p); t.preamble = static_cast<const float*>(h->d_tx_pre[layout].p);
    t.points = static_cast<const float2*>(h->d_tx_points.p);
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    (void)cudaGetLastError();
    const int fb = static_cast<int>(frame_bytes);
    auto launch = [&](const uint8_t* d_frames, size_t d_frame_stride, size_t nb, float* d_tx, size_t d_out_stride) -> pu_status {
        PU_CUDA_TRY(pu::ofdm_tx_launch(t, d_frames, d_frame_stride, fb, n_cw, bpc, nb, peak, d_tx, d_out_stride, st));
        ctx->launches.fetch_add(1);
        return PU_OK;
    };
    if (space == PU_MEM_DEVICE) return launch(frames, frame_stride, B, out, out_stride);
    // host memory: the padding of every output row beyond *frame_len is not staged and stays as it was
    pu::HostStage hs(ctx, st, B);
    const uint8_t* d_frames;
    float* d_tx;
    hs.in(&d_frames, frames, frame_bytes, frame_stride);
    hs.inout(&d_tx, out, static_cast<size_t>(t.frame_len), out_stride);
    return hs.run([&](size_t nb) { return launch(d_frames, frame_bytes, nb, d_tx, static_cast<size_t>(t.frame_len)); });
}
}  // namespace
}  // namespace pu

extern "C" {

pu_status pu_ofdm_tx_batch(pu_ofdm* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes, size_t B,
                           int layout, float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream) {
    PU_REQUIRE(h && code && frame_len, "pu_ofdm_tx_batch: NULL argument");
    PU_REQUIRE(layout == 0 || layout == 1, "pu_ofdm_tx_batch: layout must be 0 (training) or 1 (Schmidl-Cox preamble)");
    const int k = pu_ldpc_info_bits(code);
    PU_REQUIRE(payload_bytes * 8 <= static_cast<size_t>(k) && payload_bytes <= payload_stride, "pu_ofdm_tx_batch: payload longer than one codeword's information bits");
    return pu::ofdm_tx_frames(h, code, payload, payload_stride, payload_bytes, 1, k / 8, B, layout, peak, out, out_stride, frame_len, space, stream);
}

pu_status pu_frame_tx_batch(pu_ofdm* h, const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes, size_t B, int layout,
                            float peak, float* out, size_t out_stride, size_t* frame_len, size_t* n_codewords, pu_memspace space, void* stream) {
    PU_REQUIRE(h && code && frame_len && n_codewords, "pu_frame_tx_batch: NULL argument");
    PU_REQUIRE(layout == 0 || layout == 1, "pu_frame_tx_batch: layout must be 0 (training) or 1 (Schmidl-Cox preamble)");
    const int rate = pu_ldpc_rate(code);
    const uint64_t ncw = pu::frame_codewords(rate, frame_bytes);
    *n_codewords = static_cast<size_t>(ncw);
    PU_REQUIRE(ncw <= 255, "pu_frame_tx_batch: frame needs more than 255 codewords");
    PU_REQUIRE(B == 0 || frame_bytes <= frame_stride, "pu_frame_tx_batch: frame longer than its row");
    return pu::ofdm_tx_frames(h, code, frames, frame_stride, frame_bytes, static_cast<int>(ncw), pu::frame_bytes_per_codeword(rate), B, layout, peak,
                              out, out_stride, frame_len, space, stream);
}

pu_status pu_ofdm_acquire_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, size_t chunk, float sync_threshold,
                                int32_t* sync_info, float* coarse_cfo_hz, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ofdm_acquire_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && sync_info && coarse_cfo_hz, "pu_ofdm_acquire_batch: NULL data pointer");
    PU_REQUIRE(chunk > 0, "pu_ofdm_acquire_batch: chunk is zero");
    if (L > 40000) {   // 2 * OVERLAP_SAMPLES: beyond it the reference trims its buffer between calls (demodulator.cpp:593-597)
        pu::set_error("pu_ofdm_acquire_batch: frames longer than 40000 samples are not supported");
        return PU_ERR_UNSUPPORTED;
    }
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu_status s = h->ensure_acquire();
    if (s != PU_OK) return s;
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    pu::AcqDev a = h->acq;
    if (sync_threshold > 0.0f) a.sync_threshold = sync_threshold;
    (void)cudaGetLastError();
    if (space == PU_MEM_DEVICE) {
        PU_CUDA_TRY(pu::ofdm_acquire_launch(a, samples, B, L, static_cast<int>(L), static_cast<int>(std::min<size_t>(chunk, L)),
                                            reinterpret_cast<int4*>(sync_info), coarse_cfo_hz, st));
        ctx->launches.fetch_add(1);
        return PU_OK;
    }
    pu::HostStage hs(ctx, st, B);
    const float* d_x;
    int32_t* d_info;
    float* d_cfo;
    hs.in(&d_x, samples, L);
    hs.out(&d_info, sync_info, 4);
    hs.out(&d_cfo, coarse_cfo_hz, 1);
    return hs.run([&](size_t nb) { return pu_ofdm_acquire_batch(h, d_x, nb, L, chunk, sync_threshold, d_info, d_cfo, PU_MEM_DEVICE, st); });
}

pu_status pu_ofdm_process_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, size_t chunk, float sync_threshold,
                                float* llr_out, size_t llr_stride, int32_t* n_llr, int32_t* sync_info, float* coarse_cfo_hz,
                                float* snr_db, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ofdm_process_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && llr_out && n_llr, "pu_ofdm_process_batch: NULL data pointer");
    PU_REQUIRE(llr_stride > 0, "pu_ofdm_process_batch: llr_stride is zero");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const pu::OfdmPlan& p = h->plan;
    pu_status s;
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float* d_x;
        float *d_llr, *d_snr, *d_cfo;
        int32_t *d_n, *d_info;
        hs.in(&d_x, samples, L);
        hs.out(&d_llr, llr_out, llr_stride);
        hs.out(&d_n, n_llr, 1);
        hs.out(&d_snr, snr_db, 1);
        hs.out(&d_info, sync_info, 4);
        hs.out(&d_cfo, coarse_cfo_hz, 1);
        return hs.run([&](size_t nb) {
            return pu_ofdm_process_batch(h, d_x, nb, L, chunk, sync_threshold, d_llr, llr_stride, d_n, d_info, d_cfo, d_snr, PU_MEM_DEVICE, st);
        });
    }
    // device scratch: acquisition results, frame windows
    pu::DevMem dacq, dcfo, dstart, dnsym;
    std::vector<int32_t> zi(B * 4, 0);
    if ((s = dacq.upload(zi.data(), zi.size())) != PU_OK) return s;
    if ((s = dcfo.upload(zi.data(), B)) != PU_OK) return s;
    if ((s = dstart.upload(zi.data(), B)) != PU_OK) return s;
    if ((s = dnsym.upload(zi.data(), B)) != PU_OK) return s;
    {
        // The search is replayed on the first 2 * OVERLAP_SAMPLES = 40 000 samples only: beyond them the reference starts trimming
        // its buffer between calls (demodulator.cpp:551-555,593-597), which a whole-frame batch cannot replay.  A frame that
        // synchronises inside that prefix -- every frame of the tools -- may be as long as it likes: the SYNCED state runs on L.
        if ((s = h->ensure_acquire()) != PU_OK) return s;
        pu::AcqDev a = h->acq;
        if (sync_threshold > 0.0f) a.sync_threshold = sync_threshold;
        const size_t avail = std::min<size_t>(L, 40000);
        (void)cudaGetLastError();
        PU_CUDA_TRY(pu::ofdm_acquire_launch(a, samples, B, L, static_cast<int>(avail), static_cast<int>(std::min<size_t>(chunk, avail)),
                                            static_cast<int4*>(dacq.p), static_cast<float*>(dcfo.p), st));
        ctx->launches.fetch_add(1);
    }
    pu::acquire_windows_kernel<<<static_cast<unsigned>((B + 255) / 256), 256, 0, st>>>(
        static_cast<const int4*>(dacq.p), B, static_cast<int>(L), p.sym_len, p.n_data * p.bps, static_cast<int>(llr_stride),
        static_cast<int*>(dstart.p), static_cast<int*>(dnsym.p), n_llr);
    ctx->launches.fetch_add(1);
    // SYNCED state (demodulator.cpp:665-690): no LTS channel estimate, mixer restarted at the first data symbol, CFO = the
    // Schmidl-Cox estimate with zero rotator phase -- the presynced path with zero training symbols on the frame's window
    s = launch_ofdm(h, samples, B, L, 0, static_cast<const float*>(dcfo.p), nullptr, llr_out, llr_stride, snr_db, nullptr, nullptr, st,
                    static_cast<const int*>(dstart.p), static_cast<const int*>(dnsym.p));
    if (s != PU_OK) return s;
    if (sync_info) PU_CUDA_TRY(cudaMemcpyAsync(sync_info, dacq.p, B * 4 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    if (coarse_cfo_hz) PU_CUDA_TRY(cudaMemcpyAsync(coarse_cfo_hz, dcfo.p, B * sizeof(float), cudaMemcpyDeviceToDevice, st));
    PU_CUDA_TRY(cudaStreamSynchronize(st));   // the scratch buffers above are freed on return
    return PU_OK;
}

pu_status pu_ofdm_training_cfo_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, int training_symbols, float* cfo_hz,
                                     pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ofdm_training_cfo_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && cfo_hz, "pu_ofdm_training_cfo_batch: NULL data pointer");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const pu::OfdmPlan& p = h->plan;
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float* d_x;
        float* d_c;
        hs.in(&d_x, samples, L);
        hs.out(&d_c, cfo_hz, 1);
        return hs.run([&](size_t nb) { return pu_ofdm_training_cfo_batch(h, d_x, nb, L, training_symbols, d_c, PU_MEM_DEVICE, st); });
    }
    if (training_symbols < 2 || L < 2 * static_cast<size_t>(p.sym_len)) {          // ofdm_sync.cpp:279-282 (and nothing to correlate)
        PU_CUDA_TRY(cudaMemsetAsync(cfo_hz, 0, B * sizeof(float), st));
    } else {
        const pu_status s = h->ensure_nco(2);
        if (s != PU_OK) return s;
        const int warps = 4;
        const size_t smem = static_cast<size_t>(warps) * 2 * p.nfft * sizeof(float2);
        static std::atomic<uint64_t> attr{0};
        PU_CUDA_TRY(pu::smem_optin(attr, pu::ofdm_training_cfo_kernel, 96 * 1024));
        (void)cudaGetLastError();
        pu::ofdm_training_cfo_kernel<<<static_cast<unsigned>((B + warps - 1) / warps), warps * 32, smem, st>>>(h->dev, samples, L, B, cfo_hz);
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
    }
    return PU_OK;
}

pu_status pu_ofdm_presynced_debug(pu_ofdm* h, const float* samples, size_t L, int training_symbols, float cfo_hz,
                                  float cfo_phase, float* llr_out, size_t llr_cap, float* records, size_t records_cap,
                                  int* n_data_symbols) {
    PU_REQUIRE(h && samples && llr_out && records, "pu_ofdm_presynced_debug: NULL argument");
    const pu::OfdmPlan& p = h->plan;
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int n_symbols = static_cast<int>(L / p.sym_len);
    const int nds = std::max(0, n_symbols - training_symbols);
    const int nu = p.n_data + p.n_pilot;
    const size_t rec = static_cast<size_t>(4 * nu + 3 * p.n_data + pu::kDbgScalars);
    PU_REQUIRE(records_cap >= rec * nds, "pu_ofdm_presynced_debug: records buffer too small");
    if (n_data_symbols) *n_data_symbols = nds;
    // one frame through the general presynced kernel, which records every symbol's intermediate values
    pu::HostStage hs(ctx, st, 1);
    const float cp[2] = {cfo_hz, cfo_phase};
    const float *d_x, *d_c;
    float *d_llr, *d_rec;
    hs.in(&d_x, samples, L);
    hs.in(&d_c, cp, 2);
    hs.out(&d_llr, llr_out, llr_cap);
    hs.out(&d_rec, records, rec * nds);
    return hs.run([&](size_t) { return launch_ofdm(h, d_x, 1, L, training_symbols, d_c, d_c + 1, d_llr, llr_cap, nullptr, nullptr, d_rec, st); });
}

}  // extern "C"

pu_ctx* pu_ofdm_context(pu_ofdm* h) { return h ? h->ctx : nullptr; }

// Which samples of a presynced frame the demodulation kernel reads when a zero-CFO call takes the ofdm_diff512 path (launch_ofdm):
// symbols [first, n_symbols), samples [cp, cp + nfft) of each.  The host-buffer pipeline (linksim.cu) copies only those.  Returns
// false when the call would take another kernel (which may read anything).
bool pu_ofdm_diff512_window(pu_ofdm* h, const float* d_samples, size_t B, size_t L, int training, int* first, int* n_symbols, int* sym_len,
                            int* cp, int* nfft) {
    if (!h) return false;
    const pu::OfdmPlan& p = h->plan;
    const int ns = static_cast<int>(L / p.sym_len);
    if (ns < 1 || static_cast<size_t>(ns) * p.sym_len != L) return false;
    if (h->ensure_nco(ns) != PU_OK) return false;
    if (!pu::ofdm_diff_supported(h->dev, ns, training) || !pu::ofdm_diff512_supported(h->dev, ns, training, d_samples, L, B)) return false;
    *first = training > 0 ? training - 1 : 0;
    *n_symbols = ns;
    *sym_len = p.sym_len;
    *cp = h->dev.cp;
    *nfft = p.nfft;
    return true;
}
