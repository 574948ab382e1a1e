// projectultra_b200/csrc/ofdm_diff512.cu — persistent, TMA-staged, packed-fp32 receive kernel for the 512-FFT
// differential no-pilot OFDM modes with zero CFO (the BASELINE.json headline: M1 512-FFT DQPSK R1/2).
//
// Same reference behaviour and the same arithmetic DAG as ofdm_diff.cu (OFDMDemodulator::processPresynced,
// src/ofdm/demodulator.cpp:854-985: toBaseband channel_equalizer.cpp:19-57 -> extractSymbol + radix-2 FFT :59-71,
// src/dsp/fft.cpp:89-121 -> H from the last LTS symbol :179-185 -> ZF equalise :747-770 -> demapD*PSK
// src/ofdm/soft_demap.hpp:173-237); every butterfly is still the reference's unfused (t = w*b, a+t, a-t) in the
// reference's stage order, so bins / H / equalised symbols / LLRs stay bit-identical.  What changes is the machine
// mapping, chosen from the r03 profile (ofdm_diff_kernel: 78 % issue-slot utilisation, 56 % of all instructions are
// scalar FMUL/FADD of the butterflies, 28 % of stall samples wait on the first LDG of a symbol) and from the first
// packed kernel (pairs of symbols of one frame per warp: half the instructions, but two CTA-wide barriers per frame
// and a few-thread exact-demapper tail left the SM idle 75 % of the time):
//   * A WARP OWNS TWO FRAMES and walks their symbols in order.  Each 64-bit register pair holds the same quantity of
//     frame f and frame f+1, and the butterflies are issued as sm_100 packed-fp32 instructions (FFMA2 / FADD2: two
//     IEEE-rn fp32 operations per issue slot).  ptxas contracts `mul.rn.f32x2` + `add.rn.f32x2` into one FFMA2 even
//     with --fmad=false (measured: tools/ubench/f32x2_bench.cu), which would break bit-exactness, so every product
//     is written as fma(a, b, Z) with Z = (-0, -0) passed as a KERNEL ARGUMENT: a*b + (-0) is exactly RN(a*b)
//     including the sign of a zero product, and ptxas cannot fold an unknown addend.
//   * NOTHING IS SHARED BETWEEN WARPS but the read-only NCO table: the lanes that end the FFT holding a used bin keep
//     H, 1/nv and the previous equalised symbol of their carrier in registers and equalise + demap right there, so
//     the kernel has no __syncthreads / named barrier at all after its prologue.
//   * butterflies whose twiddle is tw[0] = (1, -0) skip the multiplication: (1, -0) * b == b for every finite b up
//     to the sign of a zero component, and a zero whose sign could differ can only reach a bin when all 512 samples
//     of the symbol are zero (any other zero is produced by a cancellation x - x = +0 in both evaluations); then the
//     carrier is below the demapper's weak-signal gate (soft_demap.hpp:178,199,224) and its LLRs are 0 either way.
//   * PERSISTENT CTA per SM; every warp runs its own ring of cp.async.bulk (TMA) copies, one symbol of both frames
//     per stage, mbarrier complete_tx, refilled as soon as pass A has taken the samples into registers: no warp
//     waits on HBM latency and sample loads are conflict-free LDS.
//   * the <= 2 % of carriers that fail the saturation filter are queued per warp (equalised symbol, predecessor,
//     nv, destination) and the exact libm-restatement demapper runs on 32 queued carriers at a time with all lanes
//     busy, instead of on one or two lanes per symbol.
//   * one shared-memory transpose between the two FFT passes, the real and the imaginary halves one after the other
//     through a buffer of half the size (two more __syncwarp, twice the LDS/STS instructions, room for more warps).
// HBM traffic: every sample of the symbols that are used is read exactly once, LLRs are written once.
// Measured and not kept (profiles/r04_ofdm512_variants.txt, r05): a 3-stage ring (0.70 ms per 53 248 frames against 0.54 ms),
// a 128-bit transpose buffer of full size (0.69 ms), and 16 warps with the transpose done in place in the ring stage and the
// pass-B twiddles in shared memory to stay under 128 registers (0.56 ms: the kernel is not occupancy-bound).
#include <cfloat>

#include "ofdm_dev.cuh"
#include "ofdm_diff_demap.cuh"
#include "pu_async.cuh"
#include "pu_internal.h"

namespace pu {


constexpr int kP512MaxWarps = 12;       // frame pairs in flight per CTA (one warp each)
constexpr int kP512Stages = 2;          // ring depth of the per-warp sample staging
constexpr int kP512MaxSym = 40;
constexpr int kP512Buf = 512 + 32;      // transpose slots (u64) per warp: element p lives at p + (p >> 4)
constexpr size_t kP512SmemMax = 227 * 1024;

struct P512Tw { u64 re[8], im[8]; };    // pass-A twiddles tw[32 m] as broadcast pairs (w.x, w.x), (w.y, w.y)

struct C2 { u64 re, im; };              // one complex quantity of frames (f, f+1): re = (re_f, re_f1), im likewise

// t = w * b as GCC lowers std::complex<float> multiplication (ofdm_dev.cuh: cmul), for two symbols at once
__device__ __forceinline__ C2 cmul2(u64 wre, u64 wim, C2 b, u64 Z) {
    C2 t;
    t.re = sub2(fma2(wre, b.re, Z), fma2(wim, b.im, Z));
    t.im = add2(fma2(wre, b.im, Z), fma2(wim, b.re, Z));
    return t;
}
__device__ __forceinline__ void bfly2(C2& a, C2& b, u64 wre, u64 wim, u64 Z) {   // fft.cpp:108-110
    const C2 t = cmul2(wre, wim, b, Z);
    b.re = sub2(a.re, t.re); b.im = sub2(a.im, t.im);
    a.re = add2(a.re, t.re); a.im = add2(a.im, t.im);
}
__device__ __forceinline__ void bfly2_w0(C2& a, C2& b) {                         // twiddle tw[0] = (1, -0): t == b
    const C2 t = b;
    b.re = sub2(a.re, t.re); b.im = sub2(a.im, t.im);
    a.re = add2(a.re, t.re); a.im = add2(a.im, t.im);
}
__device__ __forceinline__ C2 bfly2_lo(C2 a, C2 b, u64 wre, u64 wim, u64 Z) {
    const C2 t = cmul2(wre, wim, b, Z);
    C2 r; r.re = add2(a.re, t.re); r.im = add2(a.im, t.im); return r;
}
__device__ __forceinline__ C2 bfly2_hi(C2 a, C2 b, u64 wre, u64 wim, u64 Z) {
    const C2 t = cmul2(wre, wim, b, Z);
    C2 r; r.re = sub2(a.re, t.re); r.im = sub2(a.im, t.im); return r;
}

constexpr int kP512Queue = 64;          // per-warp queue of carriers waiting for the exact demapper (flushed 32 at a time)
constexpr int kP512StageFloats = 1024;  // one ring stage: 512 samples (after the cyclic prefix) of frame f, then of frame f+1

struct P512Smem {     // offsets (bytes) into dynamic shared memory, computed identically on host and device
    size_t nco;                                              // CTA-wide: NCO slices of the processed symbols
    size_t warp0, warp_stride;                               // then one block per warp:
    size_t S, T, q_rx, q_rxp, q_h, q_frame, q_item, bars; //   offsets inside a warp block
    size_t total;
};
__host__ __device__ inline P512Smem p512_layout(int n_proc, int warps) {
    P512Smem L;
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += (bytes + 15) & ~size_t(15); return at; };
    L.nco = take(static_cast<size_t>(n_proc) * 512 * sizeof(float2));
    L.warp0 = (o + 127) & ~size_t(127);
    o = 0;
    L.S = take(static_cast<size_t>(kP512Stages) * kP512StageFloats * sizeof(float));
    L.T = take(kP512Buf * sizeof(float2));
    L.q_rx = take(kP512Queue * sizeof(float2));
    L.q_rxp = take(kP512Queue * sizeof(float2));
    L.q_h = take(kP512Queue * sizeof(float2));
    L.q_frame = take(kP512Queue * sizeof(unsigned));
    L.q_item = take(kP512Queue * sizeof(int));
    L.bars = take(static_cast<size_t>(kP512Stages) * sizeof(u64));
    L.warp_stride = (o + 127) & ~size_t(127);
    L.total = L.warp0 + static_cast<size_t>(warps) * L.warp_stride;
    return L;
}

__global__ void __launch_bounds__(kP512MaxWarps * 32, 1) ofdm_diff512_kernel(
    OfdmDev d, P512Tw twa, u64 Z, const float* __restrict__ samples, size_t frame_stride, size_t B, int n_symbols, int training,
    float* __restrict__ llr_out, size_t llr_stride, int llr_limit, float* __restrict__ snr_db_out, float* __restrict__ final_cfo_out) {
    constexpr int EPL = 16;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int W = blockDim.x >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nd = d.n_data;
    const int first = training > 0 ? training - 1 : 0;   // data H uses the LAST training symbol only (:179-185)
    const int n_proc = n_symbols - first;
    const P512Smem L = p512_layout(n_proc, W);
    constexpr int SS = kP512StageFloats;
    float2* nco_s = reinterpret_cast<float2*>(smem_raw + L.nco);                       // [n_proc][16][32] (cos, -sin)
    unsigned char* wb = smem_raw + L.warp0 + warp * L.warp_stride;
    float* S = reinterpret_cast<float*>(wb + L.S);
    u64* tb = reinterpret_cast<u64*>(wb + L.T);
    float2* q_rx = reinterpret_cast<float2*>(wb + L.q_rx);       // queued carriers: FFT bin of the symbol,
    float2* q_rxp = reinterpret_cast<float2*>(wb + L.q_rxp);     //   bin of the preceding symbol,
    float2* q_h = reinterpret_cast<float2*>(wb + L.q_h);         //   channel estimate of the carrier
    unsigned* q_frame = reinterpret_cast<unsigned*>(wb + L.q_frame);
    int* q_item = reinterpret_cast<int*>(wb + L.q_item);
    u64* bars = reinterpret_cast<u64*>(wb + L.bars);

    const int c = lane & 15, b8 = lane >> 4;
    const int nlo = nd / 2, nhi = nd - nlo;
    const int rlane = static_cast<int>(__brev(static_cast<unsigned>(lane)) >> 27);   // brev5(lane)
    const float zf = __uint_as_float(static_cast<unsigned>(Z));                        // -0.0f the compiler cannot see

    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < kP512Stages; ++i) mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // NCO slices of the processed symbols (loop invariant: resident in shared memory for the life of the CTA); entry
    // [sy][q][lane] belongs to sample cp + brev5(lane) + 32 brev4(q) of symbol first + sy: the lane-linear order of pass A
    for (int i = threadIdx.x; i < n_proc * 512; i += blockDim.x) {
        const int sy = i >> 9, q = (i >> 5) & 15, l = i & 31;
        const int n = static_cast<int>(__brev(static_cast<unsigned>(l)) >> 27) + 32 * static_cast<int>(__brev(static_cast<unsigned>(q)) >> 28);
        const float2 o = __ldg(&d.nco[static_cast<size_t>(first + sy) * d.sym_len + d.cp + n]);
        nco_s[i] = make_float2(o.x, -o.y);
    }
    __syncthreads();      // the only CTA-wide barrier: from here on every warp is an independent pipeline

    // ---- this warp's share of the batch: frame pairs gw, gw + GW, ...
    const size_t n_pairs = (B + 1) >> 1;
    const size_t gw = static_cast<size_t>(blockIdx.x) * W + warp, GW = static_cast<size_t>(gridDim.x) * W;
    const size_t n_mine = gw < n_pairs ? (n_pairs - gw + GW - 1) / GW : 0;
    const size_t total_steps = n_mine * n_proc;
    const uint32_t sym_bytes = 512 * sizeof(float);

    // producer cursor (lane 0 only uses it): step -> (pair, symbol)
    size_t ip_pair = gw;
    int ip_sym = 0;
    auto issue = [&](int stage) {
        const size_t f0 = 2 * ip_pair, f1 = (f0 + 1 < B) ? f0 + 1 : f0;     // odd tail: the upper half recomputes frame f (never stored)
        const size_t so = static_cast<size_t>(first + ip_sym) * d.sym_len + d.cp;
        mbar_expect_tx(&bars[stage], 2 * sym_bytes);
        bulk_g2s(S + stage * SS, samples + f0 * frame_stride + so, sym_bytes, &bars[stage]);
        bulk_g2s(S + stage * SS + 512, samples + f1 * frame_stride + so, sym_bytes, &bars[stage]);
        if (++ip_sym == n_proc) { ip_sym = 0; ip_pair += GW; }
    };
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < kP512Stages; ++i)
            if (static_cast<size_t>(i) < total_steps) issue(i);
    }

    // ---- per-lane twiddles of pass B as broadcast pairs (loop invariant).  Stage q pairs (j, j + 2^q); low outputs
    //      use k = c, high outputs k = c + 16 (2^q - 1); table index k << (4 - q).  Stage 9: k = c or c + 240.
    u64 wl_re[4], wl_im[4], wh_re[4], wh_im[4], wlast_re, wlast_im;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int sh = 4 - q;
        const float2 a = __ldg(&d.twiddle[c << sh]);
        const float2 b = __ldg(&d.twiddle[(c + 16 * ((1 << q) - 1)) << sh]);
        wl_re[q] = pk(a.x, a.x); wl_im[q] = pk(a.y, a.y);
        wh_re[q] = pk(b.x, b.x); wh_im[q] = pk(b.y, b.y);
    }
    {
        const float2 a = __ldg(&d.twiddle[b8 ? (c + 240) : c]);
        wlast_re = pk(a.x, a.x); wlast_im = pk(a.y, a.y);
    }
    // the carrier this lane ends the FFT with: bins 1..nhi on lanes (0, c), bins 512-nlo..511 on lanes (1, c)
    int idx = -1;
    if (b8 == 0) { if (c >= 1 && c <= nhi) idx = nlo + c - 1; }
    else { const int cc = 16 - c; if (c >= 1 && cc <= nlo) idx = nlo - cc; }
    const float2 zc = idx >= 0 ? __ldg(&d.zc[idx]) : make_float2(1.0f, 0.0f);
    const int bps = d.bps, mod = d.mod;
    const float2 one = make_float2(1.0f, 0.0f);
    const unsigned lt_mask = (1u << lane) - 1u;

    int qcount = 0;                                        // warp-uniform
    // Exact path for the first min(qcount, 32) queued carriers: equalize (:747-770, ZF with pilot_phase_correction == (1,0)
    // and timing_offset == 0) of the symbol and of its predecessor from their raw bins, then the libm-restatement demapper.
    auto flush = [&]() {
        const int n = qcount < 32 ? qcount : 32;
        if (lane < n) {
            float l[3];
            const int qi = q_item[lane];
            const int item = qi & 0x3fffffff;
            const bool first = (qi >> 30) != 0;
            const float2 hh = q_h[lane];
            const float hq = cnorm(hh);
            float nq = (hq > 1e-6f) ? clampf(1e-6f, 100.0f, __fdiv_rn(0.1f, hq)) : 100.0f;   // noise_variance stays 0.1 (:762-768)
            nq = __fmul_rn(nq, d.ce_margin);
            auto eq = [&](float2 r) {
                return (hq > 1e-6f) ? cmul(cmul(cdivs(cmul(r, cconj(hh)), hq), one), one)    // :761
                                    : cmul(cmul(r, one), one);
            };
            const float2 sym = eq(q_rx[lane]);
            const float2 prv = first ? one : eq(q_rxp[lane]);            // differential reference (1,0) (demodulator.cpp:251-255)
            demap_exact(mod, sym, prv, false, nq, l);                    // |(1,0)| == 1 exactly, so `first` is not needed there
            store_llrs(llr_out + static_cast<size_t>(q_frame[lane]) * llr_stride, item * bps, bps, l, llr_limit, d.llr_perm, d.perm_len);
        }
        const int rem = qcount - n;
        float2 ms = one, mp = one, mh = one; unsigned mf = 0; int mi = 0;
        if (lane < rem) { ms = q_rx[32 + lane]; mp = q_rxp[32 + lane]; mh = q_h[32 + lane]; mf = q_frame[32 + lane]; mi = q_item[32 + lane]; }
        __syncwarp();
        if (lane < rem) { q_rx[lane] = ms; q_rxp[lane] = mp; q_h[lane] = mh; q_frame[lane] = mf; q_item[lane] = mi; }
        __syncwarp();
        qcount = rem;
    };

    // per-frame state of this lane's carrier, [0] = frame f, [1] = frame f+1.  rxp holds the FFT bin of the previous symbol
    // (the channel estimate itself before the first data symbol, so that bin * conj(rxp) / |h|^2 is the equalised symbol
    // times the conjugate of the reference (1,0)); ihp = 1/|h|^2 (0 when the carrier is not equalised, which sends it to
    // the exact path).
    float2 h[2] = {one, one};
    float inv_nv[2] = {10.0f, 10.0f};
    C2 rxp = {pk(1.0f, 1.0f), pk(0.0f, 0.0f)};
    u64 ihp = pk(1.0f, 1.0f);

    size_t pair = gw;
    int sidx = 0, stage = 0;
    uint32_t parity = 0;
    for (size_t t = 0; t < total_steps; ++t) {
        const size_t f0 = 2 * pair;
        const bool have1 = f0 + 1 < B;
        const int s = first + sidx;
        mbar_wait(&bars[stage], parity);
        const float* x0 = S + stage * SS;
        const float* x1 = x0 + 512;
        const float2* nc = nco_s + sidx * 512 + lane;                 // [q][lane]: entry of sample brev5(lane) + 32 brev4(q)
        // ---- pass A: lane g owns bit-reversed positions 16 g .. 16 g + 15 = samples brev5(g) + 32 brev4(q)
        C2 v[EPL];
#pragma unroll
        for (int q = 0; q < EPL; ++q) {
            const int brq = static_cast<int>(__brev(static_cast<unsigned>(q)) >> 28);
            const int n = rlane + 32 * brq;
            const float xa = x0[n], xb = x1[n];
            const float2 o = nc[32 * q];                              // (cos, -sin)
            v[q].re = pk(__fmaf_rn(o.x, xa, zf), __fmaf_rn(o.x, xb, zf));   // samples[i] * conj(osc) (channel_equalizer.cpp:36)
            v[q].im = pk(__fmaf_rn(o.y, xa, zf), __fmaf_rn(o.y, xb, zf));
        }
        __syncwarp();                                                  // every lane has taken its samples out of the stage
        if (lane == 0 && t + kP512Stages < total_steps) issue(stage);     // refill it with the step a full ring ahead
#pragma unroll
        for (int tt = 1; tt <= 4; ++tt) {
            const int half = 1 << (tt - 1);
#pragma unroll
            for (int p2 = 0; p2 < EPL / 2; ++p2) {
                const int kq = p2 & (half - 1);
                const int a = ((p2 >> (tt - 1)) << tt) | kq;
                const int m = kq << (4 - tt);
                if (m == 0) bfly2_w0(v[a], v[a + half]);
                else bfly2(v[a], v[a + half], twa.re[m], twa.im[m], Z);
            }
        }
        // ---- transpose: p = 16 lane + q at slot p + (p >> 4); pass B: lane (b8, c) owns p = c + 16 j + 256 b8
#pragma unroll
        for (int q = 0; q < EPL; ++q) tb[17 * lane + q] = v[q].re;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < EPL; ++j) v[j].re = tb[c + 17 * j + 272 * b8];
        __syncwarp();
#pragma unroll
        for (int q = 0; q < EPL; ++q) tb[17 * lane + q] = v[q].im;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < EPL; ++j) v[j].im = tb[c + 17 * j + 272 * b8];
        __syncwarp();                                                  // the transpose buffer may be rewritten (next step / SNR scratch)
#pragma unroll
        for (int j = 0; j < EPL; j += 2) bfly2(v[j], v[j + 1], wl_re[0], wl_im[0], Z);
#pragma unroll
        for (int q = 1; q < 4; ++q) {
            const int step = 1 << (q + 1), hh = 1 << q;
#pragma unroll
            for (int j = 0; j < EPL; j += step) {
                v[j] = bfly2_lo(v[j], v[j + hh], wl_re[q], wl_im[q], Z);
                v[j + step - 1] = bfly2_hi(v[j + step - 1 - hh], v[j + step - 1], wh_re[q], wh_im[q], Z);
            }
        }
        // stage 9 pairs lane (0,c) [A] with lane (1,c) [B]: bin c = A0 + w B0 on lane (0,c); bin 496+c = A15 - w B15 on lane (1,c)
        const C2 send = b8 ? v[0] : v[EPL - 1];
        C2 recv;
        recv.re = __shfl_xor_sync(0xffffffffu, send.re, 16);
        recv.im = __shfl_xor_sync(0xffffffffu, send.im, 16);
        const C2 bin = b8 ? bfly2_hi(recv, v[EPL - 1], wlast_re, wlast_im, Z) : bfly2_lo(v[0], recv, wlast_re, wlast_im, Z);
        float2 rx[2];
        upk(bin.re, rx[0].x, rx[1].x); upk(bin.im, rx[0].y, rx[1].y);

        if (sidx == 0 && training == 0) { h[0] = h[1] = one; }        // a new frame pair starts without training symbols
        if (s < training || (sidx == 0 && training == 0)) {
            // estimateChannelFromLTS for data carriers (channel_equalizer.cpp:141,179-185) + the per-carrier constants of equalize,
            // straight from the registers of the lane that holds the carrier's bin of the last LTS symbol (s == training - 1)
            float ih[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (s < training) h[j] = (idx >= 0) ? cdiv(rx[j], zc) : one;
                const float hq = cnorm(h[j]);
                float nq = (hq > 1e-6f) ? clampf(1e-6f, 100.0f, __fdiv_rn(0.1f, hq)) : 100.0f;   // noise_variance stays 0.1 (:762-768)
                nq = __fmul_rn(nq, d.ce_margin);
                inv_nv[j] = __frcp_rn(nq);
                ih[j] = (hq > 1e-6f) ? __frcp_rn(hq) : 0.0f;
            }
            ihp = pk(ih[0], ih[1]);
            rxp.re = pk(h[0].x, h[1].x);
            rxp.im = pk(h[0].y, h[1].y);
            if (snr_db_out) {   // reporting-only SNR estimate of estimateChannelFromLTS (:208-225), getEstimatedSNR (demodulator.cpp:797-799)
                float* sc = reinterpret_cast<float*>(tb);
                if (idx >= 0) { sc[idx] = cabs_ref(h[0]); sc[32 + idx] = cabs_ref(h[1]); }
                __syncwarp();
                if (lane < 2 && (lane == 0 || have1)) {
                    float snr_lin = 1.0f;
                    if (training > 0) {
                        float sum = 0.0f;
                        for (int i = 0; i < nd; ++i) sum = __fadd_rn(sum, sc[32 * lane + i]);
                        const float avg = __fdiv_rn(sum, static_cast<float>(nd));
                        if (avg > 1e-6f) snr_lin = clampf(0.1f, 10000.0f, __fdiv_rn(__fmul_rn(avg, avg), 0.1f));
                    }
                    snr_db_out[f0 + lane] = 10.0f * log10f(snr_lin);
                }
                __syncwarp();
            }
            if (final_cfo_out && lane < 2 && (lane == 0 || have1)) final_cfo_out[f0 + lane] = 0.0f;
        }
        if (s >= training) {
            // ---- equalize (:747-770) + demodulateSymbol (demodulator.cpp:279-316) + soft_demap.hpp on the lane that owns the
            //      carrier, for both frames.  The equalised symbols themselves are only formed on the exact path (flush):
            //      sym * conj(prev) = bin * conj(previous bin) / |h|^2 up to rounding, and the saturation filter only needs
            //      that product to a few ulp (its margin is 4e-5 relative + 0.01 absolute), so it reads the raw bins.
            const int sd = s - training;
            const int item = sd * nd + idx;
            C2 e;
            e.re = fma2(bin.re, rxp.re, fma2(bin.im, rxp.im, Z));
            e.im = sub2(fma2(bin.im, rxp.re, Z), fma2(bin.re, rxp.im, Z));
            e.re = fma2(e.re, ihp, Z);
            e.im = fma2(e.im, ihp, Z);
            float2 dd[2], rp[2];
            upk(e.re, dd[0].x, dd[1].x); upk(e.im, dd[0].y, dd[1].y);
            upk(rxp.re, rp[0].x, rp[1].x); upk(rxp.im, rp[0].y, rp[1].y);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                bool need = false;
                if (idx >= 0 && (j == 0 || have1)) {
                    float l[3];
                    if (demap_saturated_fast(mod, dd[j], inv_nv[j], l, 4e-5f))
                        store_llrs(llr_out + (f0 + j) * llr_stride, item * bps, bps, l, llr_limit, d.llr_perm, d.perm_len);
                    else
                        need = true;
                }
                const unsigned m = __ballot_sync(0xffffffffu, need);
                if (m) {
                    if (need) {
                        const int pos = qcount + __popc(m & lt_mask);
                        q_rx[pos] = rx[j]; q_rxp[pos] = rp[j]; q_h[pos] = h[j];
                        q_frame[pos] = static_cast<unsigned>(f0 + j); q_item[pos] = item | (sd == 0 ? (1 << 30) : 0);
                    }
                    qcount += __popc(m);
                    __syncwarp();
                    if (qcount >= 32) flush();
                }
            }
            rxp = bin;
        }
        if (++sidx == n_proc) { sidx = 0; pair += GW; }
        if (++stage == kP512Stages) { stage = 0; parity ^= 1u; }
    }
    while (qcount > 0) flush();
}

// Warps per CTA: as many independent frame-pair pipelines as shared memory holds (NCO slices + one block per warp).
static int p512_warps(int n_proc) {
    int w = kP512MaxWarps;
    while (w > 1 && p512_layout(n_proc, w).total > kP512SmemMax) --w;
    return w;
}

// Returns true when the configuration / call is one this kernel covers (a superset of ofdm_diff_supported's
// conditions: 512-FFT, 16-byte aligned rows so that the bulk copies are legal).
bool ofdm_diff512_supported(const OfdmDev& d, int n_symbols, int training, const float* samples, size_t frame_stride, size_t B) {
    const bool differential = d.mod == PU_MOD_DBPSK || d.mod == PU_MOD_DQPSK || d.mod == PU_MOD_D8PSK;
    if (!differential || d.n_pilot != 0 || d.nfft != 512 || !d.nco) return false;
    if (n_symbols > kP512MaxSym || n_symbols < 1 || training < 0 || training > n_symbols) return false;
    if ((d.sym_len & 3) || (d.cp & 3) || (frame_stride & 3) || (reinterpret_cast<uintptr_t>(samples) & 15)) return false;
    if (B >= (size_t(1) << 32)) return false;                  // queued carriers carry their frame index as 32 bits
    const int first = training > 0 ? training - 1 : 0;
    if (n_symbols - first < 1) return false;
    const int nlo = d.n_data / 2, nhi = d.n_data - nlo;
    if (!(nlo < 16 && nhi < 16)) return false;
    return p512_layout(n_symbols - first, 1).total <= kP512SmemMax;
}

cudaError_t ofdm_diff512_launch(const OfdmDev& d, const float2* host_twiddle, const float* samples, size_t B, size_t frame_stride,
                                int n_symbols, int training, float* llr, size_t llr_stride, int llr_limit, float* snr_db,
                                float* final_cfo, int sm_count, cudaStream_t st) {
    P512Tw twa;
    for (int m = 0; m < 8; ++m) {
        const float2 w = host_twiddle[32 * m];
        uint32_t xr, xi;
        memcpy(&xr, &w.x, 4); memcpy(&xi, &w.y, 4);
        twa.re[m] = (static_cast<u64>(xr) << 32) | xr;
        twa.im[m] = (static_cast<u64>(xi) << 32) | xi;
    }
    const int first = training > 0 ? training - 1 : 0;
    const int warps = p512_warps(n_symbols - first);
    const P512Smem L = p512_layout(n_symbols - first, warps);
    static std::atomic<uint64_t> attr_done{0};
    {
        const cudaError_t e = smem_optin(attr_done, ofdm_diff512_kernel, static_cast<int>(kP512SmemMax));
        if (e != cudaSuccess) return e;
    }
    const size_t max_ctas = static_cast<size_t>(sm_count > 0 ? sm_count : 148);      // persistent: one CTA per SM
    const size_t want_ctas = ((B + 1) / 2 + warps - 1) / warps;
    const unsigned grid = static_cast<unsigned>(want_ctas < max_ctas ? want_ctas : max_ctas);
    const u64 Z = 0x8000000080000000ull;    // (-0.0f, -0.0f): see the header comment
    ofdm_diff512_kernel<<<grid, warps * 32, L.total, st>>>(d, twa, Z, samples, frame_stride, B, n_symbols, training, llr,
                                                                                         llr_stride, llr_limit, snr_db, final_cfo);
    return cudaGetLastError();
}

}  // namespace pu
