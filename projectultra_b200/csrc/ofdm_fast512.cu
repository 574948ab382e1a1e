// projectultra_b200/csrc/ofdm_fast512.cu — FMA-contracted form of the headline receive kernel (512-FFT differential
// no-pilot OFDM modes with zero CFO: BASELINE.json's M1 512-FFT DQPSK R1/2), selected with
// pu_ofdm_set_precision(h, PU_PRECISION_FAST).
//
// Same reference behaviour as ofdm_diff512.cu (OFDMDemodulator::processPresynced, src/ofdm/demodulator.cpp:854-985:
// toBaseband channel_equalizer.cpp:19-57 -> extractSymbol + FFT :59-71, src/dsp/fft.cpp:89-121 -> H from the last LTS
// symbol :179-185 -> ZF equalise :747-770 -> demapD*PSK src/ofdm/soft_demap.hpp:173-237), the same machine mapping (a warp
// owns two frames packed into f32x2 registers, per-warp TMA ring, two register passes with one shared-memory transpose,
// equalise + demap on the lane that owns the bin, exact libm demapper for the carriers that fail the saturation filter),
// but NOT the reference's rounding sequence.  BASELINE.json's north star asks for LLRs within 1e-4 relative and
// bit-exact hard decisions on frames decoded with margin, not for bit-identical FFT bins; ofdm_diff512.cu pays for
// bit-identical bins with an unfused radix-2 DAG (10 packed instructions per butterfly, every twiddle multiplication
// executed, products forced through fma(a, b, -0)) and was measured at 0.52 of the HBM roofline, latency/issue-bound
// (r41: 1 041 warp instructions per frame-pair symbol).  Here:
//   * every butterfly is fused multiply-adds: a' = a + w b costs two FFMA2 per component, and b' = a - w b = 2a - a'
//     ONE more -- stored NEGATED, as -(2a - a') = fma(a, -2, a'), because FFMA2 can negate its scalar-broadcast twiddle
//     operand for free but not a packed addend.  The sign of every element is a compile-time function of its index and
//     is folded into the twiddle signs of the next butterfly; after the transpose a lane's 16 values share one sign
//     (they are element c of 16 sub-transforms) and the pruned pass B keeps a fixed sign per lane, so the bin a lane
//     ends with is sigma_lane * (true bin).  Every consumer is invariant under that sign: |h|^2, |h|, bin * conj(previous
//     bin of the same lane), bin * conj(h) with h estimated on the same lane.  6 packed instructions per butterfly instead
//     of 10, 4 for twiddles 1 and -j, 6 for the (1 -+ j)/sqrt2 ones.
//   * ptxas folds a duplicated scalar into the packed instruction (`FFMA2 R, R.F32x2, -R.F32, R.F32x2`, immediates and
//     uniform registers likewise): twiddles are scalars (half the registers of the bit-exact kernel), pass-A twiddles
//     are immediates, and the NCO mix x[n] * conj(osc[n]) is fused into the first butterfly (6 instead of 8 + no MOVs).
//   * the differential product and the saturation filter run packed for both frames; LLR destinations (fused
//     deinterleave + output limit) come from a per-CTA shared-memory table instead of a global-memory gather.
// Parity statement (tests/test_ofdm_fast_gpu.py): saturated LLRs (>= 98 %) are exactly the reference's +-10; the others
// go through the same libm-restatement demapper as the bit-exact kernel on bins that differ from the reference's by
// less than the reference's own bins differ from a float64 DFT; LLRs within 1e-4 * max(|ref|, 0.5); decoded bytes
// identical on every frame the reference decodes with margin.
// Like ofdm_diff512.cu, the transpose moves the real and the imaginary halves one after the other through a buffer of half the
// size.  Measured and not kept: 16 warps with the transpose done in place in the ring stage (128 registers) ran at 0.3645 ms
// against 0.3618 ms per 53 248 frames for 12 warps with their own buffer (v02: with four warps per scheduler the FMA pipe
// (math-pipe throttle 0.94 per issue) and the shared-memory pipe (68 %) are the limits, not latency).
#include <cfloat>

#include "ofdm_dev.cuh"
#include "ofdm_diff_demap.cuh"
#include "pu_async.cuh"
#include "pu_internal.h"

namespace pu {

constexpr int kF512MaxWarps = 12;
constexpr int kF512Stages = 2;              // ring depth of the per-warp sample staging
constexpr int kF512MaxSym = 40;
constexpr int kF512Buf = 512 + 32;          // transpose slots per warp: element p lives at p + (p >> 4)
constexpr int kF512Queue = 64;              // per-warp queue of carriers waiting for the exact demapper (flushed 32 at a time)
constexpr int kF512StageFloats = 1024;      // one ring stage: 512 samples (behind the cyclic prefix) of frame f, then of frame f+1
constexpr size_t kF512SmemMax = 227 * 1024;

struct FC2 { u64 re, im; };                  // one complex quantity of frames (f, f+1)

__device__ __forceinline__ u64 bc(float a) { return pk(a, a); }   // ptxas folds this into a scalar-broadcast operand

struct F512Smem {      // byte offsets into dynamic shared memory, identical on host and device
    size_t nco;        // CTA-wide [n_proc][16][32] float2 (cos, -sin) in pass-A order
    size_t dst;        // CTA-wide [n_proc][32] 4 x u16: LLR destinations of the lane's carrier in that symbol (0xffff = none)
    size_t warp0, warp_stride;
    size_t S, T, q_rx, q_rxp, q_h, q_frame, q_item, bars;
    size_t total;
};
__host__ __device__ inline F512Smem f512_layout(int n_proc, int warps) {
    F512Smem L;
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += (bytes + 15) & ~size_t(15); return at; };
    L.nco = take(static_cast<size_t>(n_proc) * 512 * sizeof(float2));
    L.dst = take(static_cast<size_t>(n_proc) * 32 * 4 * sizeof(unsigned short));
    L.warp0 = (o + 127) & ~size_t(127);
    o = 0;
    L.S = take(static_cast<size_t>(kF512Stages) * kF512StageFloats * sizeof(float));
    L.T = take(kF512Buf * sizeof(float2));
    L.q_rx = take(kF512Queue * sizeof(float2));
    L.q_rxp = take(kF512Queue * sizeof(float2));
    L.q_h = take(kF512Queue * sizeof(float2));
    L.q_frame = take(kF512Queue * sizeof(unsigned));
    L.q_item = take(kF512Queue * sizeof(int));
    L.bars = take(static_cast<size_t>(kF512Stages) * sizeof(u64));
    L.warp_stride = (o + 127) & ~size_t(127);
    L.total = L.warp0 + static_cast<size_t>(warps) * L.warp_stride;
    return L;
}

// ---- pass-A butterflies on elements stored as (sign * value); signs are compile-time after unrolling --------------------
// W16^m = (cos(2 pi m / 16), -sin(2 pi m / 16))
__device__ __forceinline__ void f_bfly(FC2& A, FC2& B, const int m, const int sa, int& sb) {
    constexpr float R = 0.70710678118654752f, C1 = 0.92387953251128674f, S1 = 0.38268343236508977f;
    const float s = static_cast<float>(sa * sb);        // relative sign of the stored B against the stored A
    if (m == 0) {                 // t = b
        const FC2 a = A;
        if (s > 0) { A.re = add2(a.re, B.re); A.im = add2(a.im, B.im); B.re = sub2(a.re, B.re); B.im = sub2(a.im, B.im); }
        else       { A.re = sub2(a.re, B.re); A.im = sub2(a.im, B.im); B.re = add2(a.re, B.re); B.im = add2(a.im, B.im); }
        sb = sa;
    } else if (m == 4) {          // t = -j b = (b.im, -b.re)
        const FC2 a = A, b = B;
        if (s > 0) { A.re = add2(a.re, b.im); A.im = sub2(a.im, b.re); B.re = sub2(a.re, b.im); B.im = add2(a.im, b.re); }
        else       { A.re = sub2(a.re, b.im); A.im = add2(a.im, b.re); B.re = add2(a.re, b.im); B.im = sub2(a.im, b.re); }
        sb = sa;
    } else if (m == 2) {          // t = b (1 - j)/sqrt2 = ((b.re + b.im), (b.im - b.re)) / sqrt2
        const FC2 a = A;
        const u64 s1 = add2(B.re, B.im), s2 = sub2(B.im, B.re);
        A.re = fma2(s1, bc(s * R), a.re); B.re = fma2(s1, bc(-s * R), a.re);
        A.im = fma2(s2, bc(s * R), a.im); B.im = fma2(s2, bc(-s * R), a.im);
        sb = sa;
    } else if (m == 6) {          // t = b (-1 - j)/sqrt2 = ((b.im - b.re), -(b.re + b.im)) / sqrt2
        const FC2 a = A;
        const u64 s1 = sub2(B.im, B.re), s2 = add2(B.re, B.im);
        A.re = fma2(s1, bc(s * R), a.re); B.re = fma2(s1, bc(-s * R), a.re);
        A.im = fma2(s2, bc(-s * R), a.im); B.im = fma2(s2, bc(s * R), a.im);
        sb = sa;
    } else {                      // general twiddle: a' = a + w b (sign sa), b' = a - w b stored as -sa * b' = fma(A, -2, A')
        const float wr = m == 1 ? C1 : m == 3 ? S1 : m == 5 ? -S1 : -C1;
        const float wi = m == 1 ? -S1 : m == 3 ? -C1 : m == 5 ? -C1 : -S1;
        const FC2 a = A;
        A.re = fma2(B.re, bc(s * wr), fma2(B.im, bc(-s * wi), a.re));
        A.im = fma2(B.im, bc(s * wr), fma2(B.re, bc(s * wi), a.im));
        B.re = fma2(a.re, bc(-2.0f), A.re);
        B.im = fma2(a.im, bc(-2.0f), A.im);
        sb = -sa;
    }
}

// ---- pass-B butterflies: both inputs carry the same sign, which the result keeps -----------------------------------------
__device__ __forceinline__ FC2 f_lo(FC2 a, FC2 b, float wr, float wi) {      // a + w b
    FC2 r;
    r.re = fma2(b.re, bc(wr), fma2(b.im, bc(-wi), a.re));
    r.im = fma2(b.im, bc(wr), fma2(b.re, bc(wi), a.im));
    return r;
}
__device__ __forceinline__ FC2 f_hi(FC2 a, FC2 b, float wr, float wi) {      // a - w b
    FC2 r;
    r.re = fma2(b.re, bc(-wr), fma2(b.im, bc(wi), a.re));
    r.im = fma2(b.im, bc(-wr), fma2(b.re, bc(-wi), a.im));
    return r;
}

__global__ void __launch_bounds__(kF512MaxWarps * 32, 1) ofdm_fast512_kernel(
    OfdmDev d, const float* __restrict__ samples, size_t frame_stride, size_t B, int n_symbols, int training,
    float* __restrict__ llr_out, size_t llr_stride, int llr_limit, float* __restrict__ snr_db_out, float* __restrict__ final_cfo_out) {
    constexpr int EPL = 16;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int W = blockDim.x >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nd = d.n_data;
    const int first = training > 0 ? training - 1 : 0;   // data H uses the LAST training symbol only (:179-185)
    const int n_proc = n_symbols - first;
    const F512Smem L = f512_layout(n_proc, W);
    constexpr int SS = kF512StageFloats;
    float2* nco_s = reinterpret_cast<float2*>(smem_raw + L.nco);
    uint2* dst_s = reinterpret_cast<uint2*>(smem_raw + L.dst);                        // [n_proc][32]
    unsigned char* wb = smem_raw + L.warp0 + warp * L.warp_stride;
    float* S = reinterpret_cast<float*>(wb + L.S);
    u64* tb = reinterpret_cast<u64*>(wb + L.T);
    float2* q_rx = reinterpret_cast<float2*>(wb + L.q_rx);       // queued carriers: FFT bin of the symbol,
    float2* q_rxp = reinterpret_cast<float2*>(wb + L.q_rxp);     //   bin of the preceding symbol (or h),
    float2* q_h = reinterpret_cast<float2*>(wb + L.q_h);         //   channel estimate of the carrier
    unsigned* q_frame = reinterpret_cast<unsigned*>(wb + L.q_frame);
    int* q_item = reinterpret_cast<int*>(wb + L.q_item);
    u64* bars = reinterpret_cast<u64*>(wb + L.bars);

    const int c = lane & 15, b8 = lane >> 4;
    const int nlo = nd / 2, nhi = nd - nlo;
    const int rlane = static_cast<int>(__brev(static_cast<unsigned>(lane)) >> 27);   // brev5(lane)
    const int bps = d.bps, mod = d.mod;
    // the carrier this lane ends the FFT with: bins 1..nhi on lanes (0, c), bins 512-nlo..511 on lanes (1, c)
    int idx = -1;
    if (b8 == 0) { if (c >= 1 && c <= nhi) idx = nlo + c - 1; }
    else { const int cc = 16 - c; if (c >= 1 && cc <= nlo) idx = nlo - cc; }

    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < kF512Stages; ++i) mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // NCO slices of the processed symbols, resident for the life of the CTA; entry [sy][q][lane] belongs to sample
    // cp + brev5(lane) + 32 brev4(q) of symbol first + sy: the lane-linear order of pass A
    for (int i = threadIdx.x; i < n_proc * 512; i += blockDim.x) {
        const int sy = i >> 9, q = (i >> 5) & 15, l = i & 31;
        const int n = static_cast<int>(__brev(static_cast<unsigned>(l)) >> 27) + 32 * static_cast<int>(__brev(static_cast<unsigned>(q)) >> 28);
        const float2 o = __ldg(&d.nco[static_cast<size_t>(first + sy) * d.sym_len + d.cp + n]);
        nco_s[i] = make_float2(o.x, -o.y);
    }
    // LLR destinations: [sy][lane] = positions of the bps LLRs of (data symbol first + sy - training, this lane's carrier) in the
    // frame's output row after the fused deinterleave (pu_ofdm_set_deinterleave) and the output limit; 0xffff = not written
    for (int i = threadIdx.x; i < n_proc * 32; i += blockDim.x) {
        const int sy = i >> 5, l = i & 31;
        const int lc = l & 15, lb = l >> 4;
        int li = -1;
        if (lb == 0) { if (lc >= 1 && lc <= nhi) li = nlo + lc - 1; }
        else { const int cc = 16 - lc; if (lc >= 1 && cc <= nlo) li = nlo - cc; }
        const int sd = first + sy - training;
        unsigned e[4] = {0xffffu, 0xffffu, 0xffffu, 0xffffu};
        if (li >= 0 && sd >= 0) {
            for (int b = 0; b < bps; ++b) {
                const int pos = (sd * nd + li) * bps + b;
                if (pos < llr_limit) e[b] = static_cast<unsigned>((d.llr_perm && pos < d.perm_len) ? __ldg(&d.llr_perm[pos]) : pos);
            }
        }
        dst_s[i] = make_uint2(e[0] | (e[1] << 16), e[2] | (e[3] << 16));
    }
    __syncthreads();      // the only CTA-wide barrier: from here on every warp is an independent pipeline

    // ---- this warp's share of the batch: frame pairs gw, gw + GW, ...
    const size_t n_pairs = (B + 1) >> 1;
    const size_t gw = static_cast<size_t>(blockIdx.x) * W + warp, GW = static_cast<size_t>(gridDim.x) * W;
    const size_t n_mine = gw < n_pairs ? (n_pairs - gw + GW - 1) / GW : 0;
    const size_t total_steps = n_mine * n_proc;
    const uint32_t sym_bytes = 512 * sizeof(float);

    size_t ip_pair = gw;      // producer cursor (lane 0 only): step -> (pair, symbol)
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
        for (int i = 0; i < kF512Stages; ++i)
            if (static_cast<size_t>(i) < total_steps) issue(i);
    }

    // ---- per-lane twiddles of pass B (loop invariant scalars).  Stage q pairs (j, j + 2^q); low outputs use k = c, high
    //      outputs k = c + 16 (2^q - 1); table index k << (4 - q).  Stage 9: k = c or c + 240.
    float2 wl[4], wh[4], wlast;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int sh = 4 - q;
        wl[q] = __ldg(&d.twiddle[c << sh]);
        wh[q] = __ldg(&d.twiddle[(c + 16 * ((1 << q) - 1)) << sh]);
    }
    wlast = __ldg(&d.twiddle[b8 ? (c + 240) : c]);
    // known LTS symbol of this lane's carrier, pre-divided: h = bin / zc = bin * conj(zc) / |zc|^2
    float2 zq = make_float2(1.0f, 0.0f);
    if (idx >= 0) {
        const float2 z = __ldg(&d.zc[idx]);
        const float iz = 1.0f / (z.x * z.x + z.y * z.y);
        zq = make_float2(z.x * iz, z.y * iz);
    }
    const float2 one = make_float2(1.0f, 0.0f);
    const unsigned lt_mask = (1u << lane) - 1u;

    int qcount = 0;                                        // warp-uniform
    // Exact path for the first min(qcount, 32) queued carriers: equalize (:747-770, ZF with pilot_phase_correction == (1,0)
    // and timing_offset == 0) of the symbol and of its predecessor from their bins, then the libm-restatement demapper.
    auto flush = [&]() {
        const int n = qcount < 32 ? qcount : 32;
        if (lane < n) {
            float l[3];
            const int qi = q_item[lane];
            const bool first_sym = (qi >> 30) != 0;
            const float2 hh = q_h[lane];
            const float hq = cnorm(hh);
            float nq = (hq > 1e-6f) ? clampf(1e-6f, 100.0f, __fdiv_rn(0.1f, hq)) : 100.0f;   // noise_variance stays 0.1 (:762-768)
            nq = __fmul_rn(nq, d.ce_margin);
            auto eq = [&](float2 r) {
                return (hq > 1e-6f) ? cmul(cmul(cdivs(cmul(r, cconj(hh)), hq), one), one)    // :761
                                    : cmul(cmul(r, one), one);
            };
            const float2 sym = eq(q_rx[lane]);
            const float2 prv = first_sym ? one : eq(q_rxp[lane]);       // differential reference (1,0) (demodulator.cpp:251-255)
            demap_exact(mod, sym, prv, false, nq, l);
            const unsigned* dq = reinterpret_cast<const unsigned*>(dst_s) + 2 * (qi & 0xffff);
            const unsigned d01 = dq[0], d2 = dq[1];
            float* row = llr_out + static_cast<size_t>(q_frame[lane]) * llr_stride;
            if ((d01 & 0xffffu) != 0xffffu) row[d01 & 0xffffu] = l[0];
            if ((d01 >> 16) != 0xffffu) row[d01 >> 16] = l[1];
            if ((d2 & 0xffffu) != 0xffffu) row[d2 & 0xffffu] = l[2];
        }
        const int rem = qcount - n;
        float2 ms = one, mp = one, mh = one; unsigned mf = 0; int mi = 0;
        if (lane < rem) { ms = q_rx[32 + lane]; mp = q_rxp[32 + lane]; mh = q_h[32 + lane]; mf = q_frame[32 + lane]; mi = q_item[32 + lane]; }
        __syncwarp();
        if (lane < rem) { q_rx[lane] = ms; q_rxp[lane] = mp; q_h[lane] = mh; q_frame[lane] = mf; q_item[lane] = mi; }
        __syncwarp();
        qcount = rem;
    };

    // per-frame state of this lane's carrier, packed (frame f, frame f+1).  rxp holds the FFT bin of the previous symbol (the channel
    // estimate itself before the first data symbol, so that bin * conj(rxp) / |h|^2 is the equalised symbol times the conjugate of the
    // reference (1,0)); ihp = 1/|h|^2 (0 when the carrier is not equalised, which sends it to the exact path).
    float2 h[2] = {one, one};
    FC2 rxp = {pk(1.0f, 1.0f), pk(0.0f, 0.0f)};
    u64 ihp = pk(1.0f, 1.0f);
    u64 inv_nv2 = pk(10.0f, 10.0f);       // 1 / nv of the carrier, per frame

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
        // ---- pass A, stage 1 fused with the mixer: elements (2p, 2p+1) = samples (n, n + 256), twiddle 1
        FC2 v[EPL];
#pragma unroll
        for (int p2 = 0; p2 < EPL / 2; ++p2) {
            const int qa = 2 * p2, qb = qa + 1;
            const int na = rlane + 32 * static_cast<int>(__brev(static_cast<unsigned>(qa)) >> 28);
            const int nb = rlane + 32 * static_cast<int>(__brev(static_cast<unsigned>(qb)) >> 28);
            const u64 xa = pk(x0[na], x1[na]), xb = pk(x0[nb], x1[nb]);
            const float2 oa = nc[32 * qa], ob = nc[32 * qb];          // (cos, -sin): samples[i] * conj(osc) (channel_equalizer.cpp:36)
            const u64 pr = mul2(xa, bc(oa.x)), pi = mul2(xa, bc(oa.y));
            v[qa].re = fma2(xb, bc(ob.x), pr);  v[qa].im = fma2(xb, bc(ob.y), pi);
            v[qb].re = fma2(xb, bc(-ob.x), pr); v[qb].im = fma2(xb, bc(-ob.y), pi);
        }
        __syncwarp();                                                  // every lane has taken its samples out of the stage
        if (lane == 0 && t + kF512Stages < total_steps) issue(stage);     // refill it with the step a full ring ahead
        int sg[EPL];
#pragma unroll
        for (int q = 0; q < EPL; ++q) sg[q] = 1;
#pragma unroll
        for (int tt = 2; tt <= 4; ++tt) {
            const int half = 1 << (tt - 1);
#pragma unroll
            for (int p2 = 0; p2 < EPL / 2; ++p2) {
                const int kq = p2 & (half - 1);
                const int a = ((p2 >> (tt - 1)) << tt) | kq;
                f_bfly(v[a], v[a + half], kq << (4 - tt), sg[a], sg[a + half]);
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
        // ---- pass B, pruned to the two bins this lane pair produces.  Stage 5: full butterflies, odd elements stored negated.
#pragma unroll
        for (int j = 0; j < EPL; j += 2) {
            const FC2 a = v[j], b = v[j + 1];
            v[j] = f_lo(a, b, wl[0].x, wl[0].y);
            v[j + 1].re = fma2(a.re, bc(-2.0f), v[j].re);             // -(a - w b)
            v[j + 1].im = fma2(a.im, bc(-2.0f), v[j].im);
        }
#pragma unroll
        for (int q = 1; q < 4; ++q) {                                  // low chain: even elements (+); high chain: odd elements (-)
            const int step = 1 << (q + 1), hh = 1 << q;
#pragma unroll
            for (int j = 0; j < EPL; j += step) {
                v[j] = f_lo(v[j], v[j + hh], wl[q].x, wl[q].y);
                v[j + step - 1] = f_hi(v[j + step - 1 - hh], v[j + step - 1], wh[q].x, wh[q].y);
            }
        }
        // stage 9 pairs lane (0,c) [A] with lane (1,c) [B]: bin c = A0 + w B0 on lane (0,c); bin 496+c = A15 - w B15 on lane (1,c) (negated)
        const FC2 send = b8 ? v[0] : v[EPL - 1];
        FC2 recv;
        recv.re = __shfl_xor_sync(0xffffffffu, send.re, 16);
        recv.im = __shfl_xor_sync(0xffffffffu, send.im, 16);
        const FC2 bin = b8 ? f_hi(recv, v[EPL - 1], wlast.x, wlast.y) : f_lo(v[0], recv, wlast.x, wlast.y);

        if (sidx == 0 && training == 0) { h[0] = h[1] = one; }        // a new frame pair starts without training symbols
        if (s < training || (sidx == 0 && training == 0)) {
            // estimateChannelFromLTS for data carriers (channel_equalizer.cpp:141,179-185) + the per-carrier constants of equalize,
            // on the lane that holds the carrier's bin of the last LTS symbol (s == training - 1)
            float ih[2], inv[2];
            if (s < training) {
                float2 rx[2];
                upk(bin.re, rx[0].x, rx[1].x); upk(bin.im, rx[0].y, rx[1].y);
#pragma unroll
                for (int j = 0; j < 2; ++j)
                    h[j] = (idx >= 0) ? make_float2(fmaf(rx[j].x, zq.x, rx[j].y * zq.y), fmaf(rx[j].y, zq.x, -rx[j].x * zq.y)) : one;
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float hq = cnorm(h[j]);
                float nq = (hq > 1e-6f) ? clampf(1e-6f, 100.0f, __fdiv_rn(0.1f, hq)) : 100.0f;   // noise_variance stays 0.1 (:762-768)
                nq = __fmul_rn(nq, d.ce_margin);
                inv[j] = __frcp_rn(nq);
                ih[j] = (hq > 1e-6f) ? __frcp_rn(hq) : 0.0f;
            }
            ihp = pk(ih[0], ih[1]);
            inv_nv2 = pk(inv[0], inv[1]);
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
            // ---- equalize (:747-770) + demodulateSymbol (demodulator.cpp:279-316) + soft_demap.hpp on the lane that owns the carrier,
            //      both frames at once: d = sym * conj(prev) = bin * conj(previous bin) / |h|^2
            FC2 e;
            e.re = fma2(bin.re, rxp.re, mul2(bin.im, rxp.im));
            e.im = sub2(mul2(bin.im, rxp.re), mul2(bin.re, rxp.im));
            e.re = mul2(e.re, ihp);
            e.im = mul2(e.im, ihp);
            const uint2 dd = dst_s[sidx * 32 + lane];
            bool need0 = false, need1 = false;
            if (mod == PU_MOD_DQPSK) {
                // saturation filter of ofdm_diff_demap.cuh (demap_saturated_fast), packed: exact LLR laws sqrt2 (dx+dy)/nv and
                // 2 (dx^2-dy^2)/(nv sp); when both exceed 10.01 + 4e-5 scale the reference's clipLLR returns exactly +-10
                const u64 r2 = fma2(e.re, e.re, mul2(e.im, e.im));
                float r2a, r2b, isa, isb;
                upk(r2, r2a, r2b);
                asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(isa) : "f"(r2a));
                asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(isb) : "f"(r2b));
                const u64 inv_sp = pk(isa, isb);
                const u64 two_inv = add2(inv_nv2, inv_nv2);
                const u64 scale = mul2(mul2(r2, inv_sp), two_inv);
                const u64 sm = add2(e.re, e.im), df = sub2(e.re, e.im);
                const u64 a0 = mul2(sm, mul2(inv_nv2, bc(1.41421356f)));
                const u64 a1 = mul2(mul2(df, sm), mul2(two_inv, inv_sp));
                const u64 thr = fma2(scale, bc(4e-5f), bc(10.01f));
                float a0a, a0b, a1a, a1b, tha, thb;
                upk(a0, a0a, a0b); upk(a1, a1a, a1b); upk(thr, tha, thb);
                const bool ok0 = (r2a > 4e-12f) && (tha < 1e29f) && (fabsf(a0a) >= tha) && (fabsf(a1a) >= tha);
                const bool ok1 = (r2b > 4e-12f) && (thb < 1e29f) && (fabsf(a0b) >= thb) && (fabsf(a1b) >= thb);
                const bool act0 = idx >= 0, act1 = idx >= 0 && have1;
                float* row0 = llr_out + f0 * llr_stride;
                float* row1 = row0 + llr_stride;
                const unsigned da = dd.x & 0xffffu, db = dd.x >> 16;
                if (act0 && ok0) {
                    if (da != 0xffffu) row0[da] = copysignf(10.0f, a0a);
                    if (db != 0xffffu) row0[db] = copysignf(10.0f, a1a);
                }
                if (act1 && ok1) {
                    if (da != 0xffffu) row1[da] = copysignf(10.0f, a0b);
                    if (db != 0xffffu) row1[db] = copysignf(10.0f, a1b);
                }
                need0 = act0 && !ok0 && da != 0xffffu;
                need1 = act1 && !ok1 && da != 0xffffu;
            } else {
                float2 ee[2];
                float inv[2];
                upk(e.re, ee[0].x, ee[1].x); upk(e.im, ee[0].y, ee[1].y);
                upk(inv_nv2, inv[0], inv[1]);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    if (idx >= 0 && (j == 0 || have1) && (dd.x & 0xffffu) != 0xffffu) {
                        float l[3];
                        if (demap_saturated_fast(mod, ee[j], inv[j], l, 4e-5f)) {
                            float* row = llr_out + (f0 + j) * llr_stride;
                            row[dd.x & 0xffffu] = l[0];
                            if ((dd.x >> 16) != 0xffffu) row[dd.x >> 16] = l[1];
                            if ((dd.y & 0xffffu) != 0xffffu) row[dd.y & 0xffffu] = l[2];
                        } else if (j == 0) need0 = true;
                        else need1 = true;
                    }
                }
            }
            const unsigned m0 = __ballot_sync(0xffffffffu, need0), m1 = __ballot_sync(0xffffffffu, need1);
            if (m0 | m1) {
                float2 rx[2], rp[2];
                upk(bin.re, rx[0].x, rx[1].x); upk(bin.im, rx[0].y, rx[1].y);
                upk(rxp.re, rp[0].x, rp[1].x); upk(rxp.im, rp[0].y, rp[1].y);
                const int item = (sidx * 32 + lane) | (s == training ? (1 << 30) : 0);     // index into dst_s + "first data symbol" flag
                if (need0) {
                    const int pos = qcount + __popc(m0 & lt_mask);
                    q_rx[pos] = rx[0]; q_rxp[pos] = rp[0]; q_h[pos] = h[0]; q_frame[pos] = static_cast<unsigned>(f0); q_item[pos] = item;
                }
                qcount += __popc(m0);
                if (need1) {
                    const int pos = qcount + __popc(m1 & lt_mask);
                    q_rx[pos] = rx[1]; q_rxp[pos] = rp[1]; q_h[pos] = h[1]; q_frame[pos] = static_cast<unsigned>(f0 + 1); q_item[pos] = item;
                }
                qcount += __popc(m1);
                __syncwarp();
                if (qcount >= 32) flush();
            }
            rxp = bin;
        }
        if (++sidx == n_proc) { sidx = 0; pair += GW; }
        if (++stage == kF512Stages) { stage = 0; parity ^= 1u; }
    }
    while (qcount > 0) flush();
}

static int f512_warps(int n_proc) {
    int w = kF512MaxWarps;
    while (w > 1 && f512_layout(n_proc, w).total > kF512SmemMax) --w;
    return w;
}

// Same coverage as ofdm_diff512_supported (512-FFT differential no-pilot, 16-byte aligned rows for the bulk copies); the queue of
// the exact path indexes the destination table with 16 bits and LLR positions are stored as 16 bits.
bool ofdm_fast512_supported(const OfdmDev& d, int n_symbols, int training, const float* samples, size_t frame_stride, size_t B, size_t llr_stride) {
    const bool differential = d.mod == PU_MOD_DBPSK || d.mod == PU_MOD_DQPSK || d.mod == PU_MOD_D8PSK;
    if (!differential || d.n_pilot != 0 || d.nfft != 512 || !d.nco) return false;
    if (n_symbols > kF512MaxSym || n_symbols < 1 || training < 0 || training > n_symbols) return false;
    if ((d.sym_len & 3) || (d.cp & 3) || (frame_stride & 3) || (reinterpret_cast<uintptr_t>(samples) & 15)) return false;
    if (B >= (size_t(1) << 32)) return false;
    const int first = training > 0 ? training - 1 : 0;
    if (n_symbols - first < 1) return false;
    const int nlo = d.n_data / 2, nhi = d.n_data - nlo;
    if (!(nlo < 16 && nhi < 16)) return false;
    const size_t total_llr = static_cast<size_t>(n_symbols - training) * d.n_data * d.bps;
    if (total_llr >= 0xffffu || (d.llr_perm && static_cast<size_t>(d.perm_len) >= 0xffffu) || llr_stride == 0) return false;
    return f512_layout(n_symbols - first, 1).total <= kF512SmemMax;
}

cudaError_t ofdm_fast512_launch(const OfdmDev& d, const float* samples, size_t B, size_t frame_stride, int n_symbols, int training,
                                float* llr, size_t llr_stride, int llr_limit, float* snr_db, float* final_cfo, int sm_count, cudaStream_t st) {
    const int first = training > 0 ? training - 1 : 0;
    const int warps = f512_warps(n_symbols - first);
    const F512Smem L = f512_layout(n_symbols - first, warps);
    static std::atomic<uint64_t> attr_done{0};
    if (const cudaError_t e = smem_optin(attr_done, ofdm_fast512_kernel, static_cast<int>(kF512SmemMax)); e != cudaSuccess) return e;
    const size_t max_ctas = static_cast<size_t>(sm_count > 0 ? sm_count : 148);      // persistent: one CTA per SM
    const size_t want_ctas = ((B + 1) / 2 + warps - 1) / warps;
    const unsigned grid = static_cast<unsigned>(want_ctas < max_ctas ? want_ctas : max_ctas);
    ofdm_fast512_kernel<<<grid, warps * 32, L.total, st>>>(d, samples, frame_stride, B, n_symbols, training, llr, llr_stride, llr_limit, snr_db, final_cfo);
    return cudaGetLastError();
}

}  // namespace pu
