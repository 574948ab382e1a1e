// projectultra_b200/csrc/ldpc_decode.cu — batched flooding scaled-min-sum LDPC decoder for sm_100a and the
// pu_ldpc_* entry points of the C ABI.
//
// Reference behaviour: LDPCDecoder::Impl::decodeBP (src/fec/ldpc_decoder.cpp:153-259).  The schedule is
// FLOODING (all check->variable messages, then all totals, then all variable->check messages, then the
// syndrome), scale 0.75, v2c clamp +-50, stop on zero syndrome.  Results are bit-exact with the reference:
// only fp32 adds in the reference's order, one multiply by 0.75 and comparisons are involved, and this TU is
// compiled with -fmad=false.
//
// Kernel shape: one codeword per CTA, state in shared memory.
//   tot[k]      total LLR of every information bit (the only totals another thread needs)
//   c2v[6][m]   check->variable message of (edge e, check slot p) at e*m+p
//   par_llr[m], par_c2v[m]   channel LLR / message of the degree-1 parity bit owned by check slot p
// The variable->check message is never stored: v2c = clamp(tot - c2v_prev) is rebuilt by the check thread
// from the previous message it wrote itself, which is exactly the value ldpc_decoder.cpp:219-222 stores.
// The syndrome of iteration t is evaluated by the check threads of iteration t+1 while they read the totals
// anyway, and voted with one __syncthreads_or: two barriers per iteration.
#include <cfloat>
#include <cstdlib>
#include <memory>
#include <new>

#include "ldpc_code.h"
#include "pu_internal.h"

namespace pu {

struct LdpcDevTables {
    int k, m, dv_max;
    const uint8_t* cn_ninfo;
    const uint16_t* cn_check;
    const uint16_t* cn_var;
    const uint8_t* vn_deg;
    const uint16_t* vn_slot;
};

constexpr int kE = kMaxInfoEdgesPerCheck;

__device__ __forceinline__ float clamp_sym(float v, float lim) {
    // std::max(-50.0f, std::min(50.0f, v)), ldpc_decoder.cpp:222
    return fmaxf(-lim, fminf(lim, v));
}

__global__ void __launch_bounds__(512) ldpc_flood_kernel(LdpcDevTables t, const float* __restrict__ llr,
                                                         size_t llr_stride, uint8_t* __restrict__ info,
                                                         size_t info_stride, uint8_t* __restrict__ ok,
                                                         int32_t* __restrict__ iters, int max_iter) {
    extern __shared__ float smem[];
    const int K = t.k, M = t.m;
    float* c2v = smem;                // [kE][M]
    float* tot = c2v + kE * M;        // [K]
    float* lin = tot + K;             // [K]  channel LLR of the info bits
    float* par_llr = lin + K;         // [M]
    float* par_c2v = par_llr + M;     // [M]
    const int tid = threadIdx.x, T = blockDim.x;
    const float* x = llr + static_cast<size_t>(blockIdx.x) * llr_stride;

    for (int j = tid; j < K; j += T) {
        const float v = x[j];
        tot[j] = v;
        lin[j] = v;
    }
    for (int p = tid; p < M; p += T) {
        par_llr[p] = x[K + t.cn_check[p]];
        par_c2v[p] = 0.0f;
#pragma unroll
        for (int e = 0; e < kE; ++e) c2v[e * M + p] = 0.0f;
    }
    __syncthreads();

    int it = 0;
    int converged = 0;
    for (;; ++it) {
        const bool last = (it == max_iter);
        // iteration 0 consumes the raw channel LLRs (ldpc_decoder.cpp:169-173 does not clamp them)
        const float lim = (it == 0) ? INFINITY : 50.0f;
        int syn = 0;
        for (int p = tid; p < M; p += T) {
            const int ninfo = t.cn_ninfo[p];
            const float pc = par_c2v[p];
            const float ptot = __fadd_rn(par_llr[p], pc);          // total of the parity bit (:206-213)
            unsigned parity = ptot < 0.0f;
            float v[kE];
#pragma unroll
            for (int e = 0; e < kE; ++e) {
                v[e] = 0.0f;
                if (e < ninfo) {
                    const float te = tot[t.cn_var[e * M + p]];
                    parity ^= (te < 0.0f);
                    v[e] = clamp_sym(__fsub_rn(te, c2v[e * M + p]), lim);   // (:219-222)
                }
            }
            const float vp = clamp_sym(__fsub_rn(ptot, pc), lim);
            syn |= parity;
            if (!last) {
                // min / second-min / sign product over all edges of the row; "msg < 0" flips (:193), so -0 is +
                float m1 = fabsf(vp), m2 = FLT_MAX;
                int arg = kE;
                unsigned neg = vp < 0.0f;
#pragma unroll
                for (int e = 0; e < kE; ++e) {
                    if (e < ninfo) {
                        const float a = fabsf(v[e]);
                        neg ^= (v[e] < 0.0f);
                        if (a < m1) { m2 = m1; m1 = a; arg = e; }
                        else if (a < m2) { m2 = a; }
                    }
                }
                const float s1 = __fmul_rn(m1, 0.75f), s2 = __fmul_rn(m2, 0.75f);   // (:200)
#pragma unroll
                for (int e = 0; e < kE; ++e) {
                    if (e < ninfo) {
                        const float mag = (e == arg) ? s2 : s1;
                        const unsigned sg = neg ^ (v[e] < 0.0f);
                        c2v[e * M + p] = sg ? -mag : mag;
                    }
                }
                {
                    const float mag = (arg == kE) ? s2 : s1;
                    const unsigned sg = neg ^ (vp < 0.0f);
                    par_c2v[p] = sg ? -mag : mag;
                }
            }
        }
        const int any = __syncthreads_or(syn);   // syndrome of the totals produced by iteration it-1 (:227-235)
        if (it > 0 && !any) { converged = 1; --it; break; }
        if (last) break;
        for (int j = tid; j < K; j += T) {
            const int d = t.vn_deg[j];
            float s = lin[j];
            for (int dd = 0; dd < d; ++dd) s = __fadd_rn(s, c2v[t.vn_slot[dd * K + j]]);   // ascending check order
            tot[j] = s;
        }
        __syncthreads();
    }

    // k information bits MSB-first, last byte left-justified (:242-256)
    uint8_t* out = info + static_cast<size_t>(blockIdx.x) * info_stride;
    const int nbytes = (K + 7) >> 3;
    for (int b = tid; b < nbytes; b += T) {
        unsigned byte = 0;
        int cnt = 0;
        for (int j = b * 8; j < b * 8 + 8 && j < K; ++j, ++cnt) byte = (byte << 1) | (tot[j] < 0.0f ? 1u : 0u);
        out[b] = static_cast<uint8_t>(byte << (8 - cnt));
    }
    if (tid == 0) {
        if (ok) ok[blockIdx.x] = static_cast<uint8_t>(converged);
        if (iters) iters[blockIdx.x] = it;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Register-resident variant used for the five real code rates.  Thread p owns check slot p for the whole decode: its
// variable indices, the messages it sent last iteration and its parity bit's LLR/message live in registers, so an
// iteration reads only the totals of its info bits from shared memory and writes its new messages there.  Thread j
// (+ r*T) owns information bit j: channel LLR and message slots in registers.  VR = info bits per thread,
// DV = maximum variable degree.
//
// Exactness notes (all against ldpc_decoder.cpp:179-236):
//  * channel LLRs are canonicalised on load (x + 0.0f turns -0 into +0).  A total that starts from a value that is
//    not -0 can never become -0, and neither can v = total - c2v, so "v < 0" is exactly the sign bit and the sign
//    product of a row is an XOR of raw bit patterns.  The sign of a zero never reaches a comparison or a magnitude
//    in the reference, so this does not change any message, hard decision or iteration count.
//  * clamp(v, +-50) = sign(v) min(|v|, 50), and the message to edge e is 0.75 * (product of the other edges' signs) *
//    (minimum of the other edges' magnitudes) (:185-201): both are FMNMX.XORSIGN combines (minxs below), so signs are
//    never separated from magnitudes.  Ties between magnitudes need no care: every edge sees the minimum over the
//    OTHER edges, which is what the reference's scan yields.
//  * absent edges: variable-side message words that no check writes (degree <= d < DV, and every word of an empty slot) are
//    zeroed once and hold +0.0f (x + 0 == x for x != -0); check-side edges of rows shorter than their warp's longest row read a
//    total of +INF: no sign, and a magnitude that is never below the clamp limit, which cannot lower the first or second
//    minimum of a row that has two real edges (every row does).
struct LdpcRegDev {   // device view of LdpcLayout (ldpc_code.h)
    int k, m, kpad, inf_slot, msg_words, threads;
    const uint8_t* cn_ninfo;
    const uint16_t* cn_check;
    const uint16_t* cn_rd;     // [kE][threads]
    const uint16_t* cn_wr;     // [kE][threads]
    const uint16_t* var_slot;  // [k]
    const int16_t* slot_var;   // [kpad]
    const uint8_t* slot_deg;   // [kpad]
};

// sign(a) XOR sign(b) on min(|a|, |b|): one FMNMX.XORSIGN.  It is the min-sum combine of two messages (:185-197: the
// sign product and the minimum magnitude of a row at once), and with b = +limit it is the symmetric clamp (:222).
__device__ __forceinline__ float minxs(float a, float b) {
    float d;
    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

// One check pass of a row with NE info edges: new messages to every edge, and the XOR of the sign bits of the totals it read
// (bit 31 = the row's parity of the previous iteration's hard decisions).  FIRST = iteration 0: no message has been sent yet
// (prev = pc = 0, so the v2c messages are the totals themselves) and the channel LLRs are not clamped (:169-173).
template <int NE, bool FIRST>
__device__ __forceinline__ unsigned cn_update(const float* __restrict__ tot, float* __restrict__ msg, const int (&rd)[kE],
                                              const int (&wr)[kE], float (&prev)[kE], float par_llr, float& pc) {
    const float ptot = FIRST ? par_llr : __fadd_rn(par_llr, pc);   // total of the parity bit (:206-213)
    const float vp = FIRST ? ptot : __fsub_rn(ptot, pc);           // its v2c before the clamp (:219-222)
    unsigned px = __float_as_uint(ptot);                            // XOR of the totals' sign bits = parity of the hard decisions
    // c[0] = parity edge, c[1..NE] = info edges: the v2c messages, sign and magnitude together.  The clamp to +-50 (:222) is
    // applied to the two heads of the scans below only, c[0] (first term of every prefix) and c[NE] (first term of every
    // suffix): every output oth[e] combines a prefix and a suffix, or is one of them, so its operand set holds at least one
    // clamped head.  A combine takes the XOR of the signs, which a clamp does not touch, and the minimum of the magnitudes;
    // min(|v|, 50) commutes with the minimum, so one clamped operand gives min(50, minimum of all operands): each output is
    // exactly what clamping every operand gives.  The +INF totals of absent edges are covered too: unclamped they only add
    // an operand of magnitude >= 50.
    float c[NE + 1];
    c[0] = FIRST ? vp : minxs(vp, 50.0f);
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const float te = tot[rd[e]];
        px ^= __float_as_uint(te);
        const float v = FIRST ? te : __fsub_rn(te, prev[e]);
        c[e + 1] = (FIRST || e + 1 < NE) ? v : minxs(v, 50.0f);
    }
    // sign product and minimum magnitude over the OTHER edges of the row (:185-197) from prefix and suffix combines:
    // 3(n-2) FMNMX.XORSIGN for n edges, exact (neither a minimum nor an XOR depends on the order it is taken in)
    float oth[NE + 1];
    if (NE == 0) {
        oth[0] = FLT_MAX;
    } else {
        float pre[NE + 1], suf[NE + 1];
        pre[0] = c[0];
#pragma unroll
        for (int i = 1; i < NE; ++i) pre[i] = minxs(pre[i - 1], c[i]);
        suf[NE] = c[NE];
#pragma unroll
        for (int i = NE - 1; i >= 1; --i) suf[i] = minxs(suf[i + 1], c[i]);
        oth[0] = suf[1];
        oth[NE] = pre[NE - 1];
#pragma unroll
        for (int i = 1; i < NE; ++i) oth[i] = minxs(pre[i - 1], suf[i + 1]);
    }
    // sign * min_abs * 0.75f (:200)
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const float out = __fmul_rn(oth[e + 1], 0.75f);
        prev[e] = out;
        msg[wr[e]] = out;
    }
    pc = __fmul_rn(oth[0], 0.75f);
    return px;
}

// The syndrome part of a check pass alone (the pass after the last iteration sends no messages).
template <int NE>
__device__ __forceinline__ unsigned cn_syndrome(const float* __restrict__ tot, const int (&rd)[kE], float par_llr, float pc) {
    unsigned px = __float_as_uint(__fadd_rn(par_llr, pc));
#pragma unroll
    for (int e = 0; e < NE; ++e) px ^= __float_as_uint(tot[rd[e]]);
    return px;
}

// Variable pass: the total of every information bit this thread owns, messages summed in ascending check order (:208-213).
template <int VR, int DV, int T, int KP>
__device__ __forceinline__ void vn_update(const float* __restrict__ msg, float* __restrict__ tot, const float (&lin)[VR], int tid) {
#pragma unroll
    for (int r = 0; r < VR; ++r) {
        const int a = tid + r * T;
        if ((r + 1) * T <= KP || a < KP) {
            float s = lin[r];
#pragma unroll
            for (int d = 0; d < DV; ++d) s = __fadd_rn(s, msg[d * KP + a]);
            tot[a] = s;
        }
    }
}

// Shared memory: msg[d][a] = message from the d-th check (ascending check index) of the information bit in variable
// slot a; tot[a] = its total.  The variable pass reads msg[d * KP + a] with a = thread index: conflict-free by
// construction.  The check pass gathers tot[a] and scatters msg[rank * KP + a]; both hit bank a mod 32, and the
// layout (ldpc_code.cpp: make_ldpc_layout) makes the 32 lanes of a warp use 32 different banks on every edge.
//
// The whole decode is specialised on NE = the longest row of the warp (check slots are sorted by degree, so warps are
// nearly uniform): every warp runs its own copy, and all copies execute the same sequence of CTA-wide barriers (barrier 0
// counts arriving threads, not program counters; max_iter and the voted syndrome are uniform over the CTA).  KP, T and DV
// are compile-time, so every shared-memory access of the variable pass is base + immediate.  Threads past the last check
// slot run a dummy row (table defaults: reads of the +INF word, writes to the scratch words, a parity LLR of +0) whose total
// is never negative, so there is no per-thread predicate in the loop.
//
// Iteration 0 (unclamped, no syndrome to test) and the syndrome-only pass after the last iteration are peeled off, so the
// loop body is one check pass, the vote and one variable pass.  The syndrome voted in iteration it is that of the totals
// of iteration it-1 (:227-235): a zero syndrome there means it-1 iterations were run, and converged.
template <int NE, int VR, int DV, int T, int KP>
__device__ __forceinline__ void decode_loop(float* __restrict__ msg, float* __restrict__ tot, const int (&rd)[kE], const int (&wr)[kE],
                                            const float (&lin)[VR], float par_llr, int tid, int max_iter, int& it_out, int& converged) {
    it_out = 0;
    converged = 0;
    if (max_iter == 0) return;   // no iteration: the hard decisions of the channel LLRs, not converged
    float prev[kE];
    float pc = 0.0f;
    cn_update<NE, true>(tot, msg, rd, wr, prev, par_llr, pc);
    __syncthreads();
    vn_update<VR, DV, T, KP>(msg, tot, lin, tid);
    __syncthreads();
    int it = 1, any = 1;
    for (; it < max_iter; ++it) {
        any = __syncthreads_or(static_cast<int>(cn_update<NE, false>(tot, msg, rd, wr, prev, par_llr, pc)) < 0);   // sign bit
        if (!any) break;
        vn_update<VR, DV, T, KP>(msg, tot, lin, tid);
        __syncthreads();
    }
    if (any) any = __syncthreads_or(static_cast<int>(cn_syndrome<NE>(tot, rd, par_llr, pc)) < 0);   // it == max_iter
    converged = !any;
    it_out = any ? it : it - 1;
}

template <int VR, int DV, int T, int MINB, int KP>
__global__ void __launch_bounds__(T, MINB) ldpc_flood_reg_kernel(LdpcRegDev t, const float* __restrict__ llr, size_t llr_stride,
                                                          uint8_t* __restrict__ info, size_t info_stride,
                                                          uint8_t* __restrict__ ok, int32_t* __restrict__ iters, int max_iter) {
    extern __shared__ float smem[];
    constexpr int kMsgWords = DV * KP + (T + 31) / 32 * 32 * kMaxInfoEdgesPerCheck;     // + 32 scratch words per (warp, edge slot)
    const int K = t.k, M = t.m;
    float* msg = smem;                       // [DV][KP] + scratch row
    float* tot = smem + kMsgWords;           // [KP] + the +INF word
    const int tid = threadIdx.x;
    const float* x = llr + static_cast<size_t>(blockIdx.x) * llr_stride;

    int rd[kE], wr[kE];
#pragma unroll
    for (int e = 0; e < kE; ++e) {
        rd[e] = t.cn_rd[e * T + tid];
        wr[e] = t.cn_wr[e * T + tid];
    }
    const int ninfo = t.cn_ninfo[tid];                       // 0 past the last check slot
    const int chk = t.cn_check[tid];
    int sv[VR];
#pragma unroll
    for (int r = 0; r < VR; ++r) {
        const int a = tid + r * T;
        sv[r] = a < KP ? t.slot_var[a] : -1;
        if (a < KP) {   // the message words of slot a that no check writes; the others are written by the first check pass
            const int deg = t.slot_deg[a];
#pragma unroll
            for (int d = 0; d < DV; ++d)
                if (d >= deg) msg[d * KP + a] = 0.0f;
        }
    }
    const int nw = __reduce_max_sync(0xffffffffu, ninfo);   // longest row of this warp (slots are sorted by degree)
    if (tid < 32) tot[KP + tid] = INFINITY;                    // LdpcLayout::inf_slot: one +INF word per bank
    // channel LLRs canonicalised on load (+0.0f)
    const float par_llr = tid < M ? __fadd_rn(x[K + chk], 0.0f) : 0.0f;
    float lin[VR];
#pragma unroll
    for (int r = 0; r < VR; ++r) {
        const int a = tid + r * T;
        lin[r] = sv[r] >= 0 ? __fadd_rn(x[sv[r]], 0.0f) : 0.0f;
        if (a < KP) tot[a] = lin[r];
    }
    __syncthreads();

    int it = 0, converged = 0;
    switch (nw) {
        case 0: decode_loop<0, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        case 1: decode_loop<1, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        case 2: decode_loop<2, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        case 3: decode_loop<3, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        case 4: decode_loop<4, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        case 5: decode_loop<5, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
        default: decode_loop<6, VR, DV, T, KP>(msg, tot, rd, wr, lin, par_llr, tid, max_iter, it, converged); break;
    }
    __syncthreads();   // every warp has left its loop: the totals are final

    // k information bits MSB-first, last byte left-justified (:242-256): warp w packs bits r*T + 32w .. +31 into 4 bytes
    uint8_t* out = info + static_cast<size_t>(blockIdx.x) * info_stride;
    // (the slots are loaded here and not in the prologue: kept in registers through the loop, they would cost the R2/3 .. R5/6
    // instances registers and occupancy)
    const int nbytes = (K + 7) >> 3, lane = tid & 31;
    int vs[VR];   // slot of information bit j = tid + r*T (the +INF word past k)
#pragma unroll
    for (int r = 0; r < VR; ++r) vs[r] = tid + r * T < K ? t.var_slot[tid + r * T] : KP;
#pragma unroll
    for (int r = 0; r < VR; ++r) {
        if (r * T < K) {
            const unsigned bits = __brev(__ballot_sync(0xffffffffu, tot[vs[r]] < 0.0f));   // bit 31 = lowest j of the warp
            const int b = ((r * T + (tid & ~31)) >> 3) + lane;
            if (lane < 4 && b < nbytes) out[b] = static_cast<uint8_t>(bits >> (24 - 8 * lane));
        }
    }
    if (tid == 0) {
        if (ok) ok[blockIdx.x] = static_cast<uint8_t>(converged);
        if (iters) iters[blockIdx.x] = it;
    }
}

}  // namespace pu

struct pu_ldpc {
    pu_ctx* ctx = nullptr;
    int device = 0;   // copy of ctx->device: the handle may outlive its context
    int max_iter = 50;
    pu::LdpcCode code;
    pu::LdpcHostTables host;
    pu::DevMem d_ninfo, d_check, d_var, d_deg, d_slot;
    pu::LdpcLayout layout;
    pu::DevMem r_ninfo, r_check, r_rd, r_wr, r_vslot, r_svar, r_sdeg;
    pu::LdpcRegDev reg{};
    pu::LdpcDevTables dev{};
    int threads = 128;
    size_t smem_bytes = 0;
    int reg_threads = 0, reg_vr = 0, reg_dv = 0;   // launch shape of the register-resident kernel (0: generic kernel)
    size_t reg_smem = 0;
    int last_success = 0, last_iters = 0;

    pu_status load(int rate) {
        code = pu::build_ldpc_code(rate);
        host = pu::make_ldpc_tables(code);
        pu_status s;
        if ((s = d_ninfo.upload(host.cn_ninfo.data(), host.cn_ninfo.size())) != PU_OK) return s;
        if ((s = d_check.upload(host.cn_check.data(), host.cn_check.size())) != PU_OK) return s;
        if ((s = d_var.upload(host.cn_var.data(), host.cn_var.size())) != PU_OK) return s;
        if ((s = d_deg.upload(host.vn_deg.data(), host.vn_deg.size())) != PU_OK) return s;
        if ((s = d_slot.upload(host.vn_slot.data(), host.vn_slot.size())) != PU_OK) return s;
        dev.k = host.k;
        dev.m = host.m;
        dev.dv_max = host.dv_max;
        dev.cn_ninfo = static_cast<const uint8_t*>(d_ninfo.p);
        dev.cn_check = static_cast<const uint16_t*>(d_check.p);
        dev.cn_var = static_cast<const uint16_t*>(d_var.p);
        dev.vn_deg = static_cast<const uint8_t*>(d_deg.p);
        dev.vn_slot = static_cast<const uint16_t*>(d_slot.p);
        // a warp multiple that covers the m check slots in one round (two for R1/4, R1/2) with few idle lanes
        const int per_round = host.m > 256 ? (host.m + 1) / 2 : host.m;
        threads = (per_round + 31) / 32 * 32;
        smem_bytes = sizeof(float) * (static_cast<size_t>(pu::kE + 2) * host.m + 2 * static_cast<size_t>(host.k));
        layout = pu::make_ldpc_layout(code);
        if ((s = r_ninfo.upload(layout.cn_ninfo.data(), layout.cn_ninfo.size())) != PU_OK) return s;
        if ((s = r_check.upload(layout.cn_check.data(), layout.cn_check.size())) != PU_OK) return s;
        if ((s = r_rd.upload(layout.cn_rd.data(), layout.cn_rd.size())) != PU_OK) return s;
        if ((s = r_wr.upload(layout.cn_wr.data(), layout.cn_wr.size())) != PU_OK) return s;
        if ((s = r_vslot.upload(layout.var_slot.data(), layout.var_slot.size())) != PU_OK) return s;
        if ((s = r_svar.upload(layout.slot_var.data(), layout.slot_var.size())) != PU_OK) return s;
        if ((s = r_sdeg.upload(layout.slot_deg.data(), layout.slot_deg.size())) != PU_OK) return s;
        reg.k = layout.k; reg.m = layout.m; reg.kpad = layout.kpad; reg.inf_slot = layout.inf_slot;
        reg.msg_words = layout.msg_words; reg.threads = layout.threads;
        reg.cn_ninfo = static_cast<const uint8_t*>(r_ninfo.p);
        reg.cn_check = static_cast<const uint16_t*>(r_check.p);
        reg.cn_rd = static_cast<const uint16_t*>(r_rd.p);
        reg.cn_wr = static_cast<const uint16_t*>(r_wr.p);
        reg.var_slot = static_cast<const uint16_t*>(r_vslot.p);
        reg.slot_var = static_cast<const int16_t*>(r_svar.p);
        reg.slot_deg = static_cast<const uint8_t*>(r_sdeg.p);
        reg_threads = layout.threads;
        reg_vr = layout.vr;
        reg_dv = layout.dv;
        reg_smem = sizeof(float) * (static_cast<size_t>(layout.msg_words) + layout.tot_words);
        return PU_OK;
    }
};

static pu_status launch_decode(pu_ldpc* h, const float* d_llr, size_t llr_stride, size_t B, uint8_t* d_info,
                               size_t info_stride, uint8_t* d_ok, int32_t* d_iters, cudaStream_t st) {
    if (B == 0) return PU_OK;
    (void)cudaGetLastError();   // drop stale non-sticky errors so the check below reports this launch only
    const size_t kMaxGrid = 1u << 30;
    for (size_t off = 0; off < B; off += kMaxGrid) {
        const size_t nb = std::min(kMaxGrid, B - off);
#define PU_LDPC_REG_CASE(VR, DV, T, MINB, KP)                                                                        \
    if (!done && h->reg_vr == (VR) && h->reg_dv == (DV) && h->reg_threads == (T) && h->layout.kpad == (KP)) {      \
        pu::ldpc_flood_reg_kernel<VR, DV, T, MINB, KP><<<static_cast<unsigned>(nb), T, h->reg_smem, st>>>(           \
            h->reg, d_llr + off * llr_stride, llr_stride, d_info + off * info_stride, info_stride,                \
            d_ok ? d_ok + off : nullptr, d_iters ? d_iters + off : nullptr, h->max_iter);                         \
        done = true;                                                                                              \
    }
        bool done = false;
        {
            // the launch shapes of make_ldpc_layout for the five code rates (threads, variable slots, degrees are fixed by H)
            PU_LDPC_REG_CASE(1, 5, 352, 3, 352)    // R1/2: 324 checks, 3 CTAs of 11 warps per SM
            PU_LDPC_REG_CASE(2, 3, 224, 4, 448)    // R2/3: 216 checks
            PU_LDPC_REG_CASE(3, 3, 192, 5, 512)    // R3/4: 162 checks
            PU_LDPC_REG_CASE(5, 3, 128, 6, 576)    // R5/6: 108 checks
            PU_LDPC_REG_CASE(1, 13, 512, 2, 192)   // R1/4: 486 checks
        }
#undef PU_LDPC_REG_CASE
        if (!done)
            pu::ldpc_flood_kernel<<<static_cast<unsigned>(nb), h->threads, h->smem_bytes, st>>>(
                h->dev, d_llr + off * llr_stride, llr_stride, d_info + off * info_stride, info_stride,
                d_ok ? d_ok + off : nullptr, d_iters ? d_iters + off : nullptr, h->max_iter);
        h->ctx->launches.fetch_add(1);
    }
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

// device tables of the systematic encoder (ofdm_tx_gpu.cu): the decoder's check tables in slot order
void pu_ldpc_encoder_view(const pu_ldpc* h, int* k, int* m, const uint8_t** cn_ninfo, const uint16_t** cn_check, const uint16_t** cn_var) {
    *k = h->dev.k; *m = h->dev.m;
    *cn_ninfo = h->dev.cn_ninfo; *cn_check = h->dev.cn_check; *cn_var = h->dev.cn_var;
}
pu_ctx* pu_ldpc_context(const pu_ldpc* h) { return h->ctx; }

extern "C" {

pu_status pu_ldpc_create(pu_ctx* ctx, int code_rate, int max_iter, pu_ldpc** out) {
    PU_REQUIRE(ctx && out, "pu_ldpc_create: NULL argument");
    *out = nullptr;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    std::unique_ptr<pu_ldpc> h(new (std::nothrow) pu_ldpc());
    if (!h) return PU_ERR_NOMEM;
    h->ctx = ctx;
    h->device = ctx->device;
    h->max_iter = max_iter < 0 ? 50 : max_iter;   // Impl::max_iterations default, ldpc_decoder.cpp:43
    pu_status s = h->load(code_rate);
    if (s != PU_OK) return s;
    *out = h.release();
    return PU_OK;
}

void pu_ldpc_destroy(pu_ldpc* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h;
}

pu_status pu_ldpc_set_rate(pu_ldpc* h, int code_rate) {
    PU_REQUIRE(h, "pu_ldpc_set_rate: NULL handle");
    PU_CUDA_TRY(cudaSetDevice(h->ctx->device));
    PU_CUDA_TRY(cudaStreamSynchronize(h->ctx->stream));
    return h->load(code_rate);
}

pu_status pu_ldpc_set_max_iterations(pu_ldpc* h, int n) {
    PU_REQUIRE(h, "pu_ldpc_set_max_iterations: NULL handle");
    h->max_iter = n;   // the reference stores any int; a non-positive value means "no iterations"
    if (h->max_iter < 0) h->max_iter = 0;
    return PU_OK;
}

int pu_ldpc_rate(const pu_ldpc* h) { return h ? h->code.rate : -1; }
int pu_ldpc_info_bits(const pu_ldpc* h) { return h ? h->code.k : -1; }
int pu_ldpc_num_edges(const pu_ldpc* h) { return h ? h->code.n_edges : -1; }

int pu_ldpc_row(const pu_ldpc* h, int check, int32_t* vars, int cap) {
    if (!h || check < 0 || check >= h->code.m) return -1;
    const auto& row = h->code.rows[check];
    for (int e = 0; e < static_cast<int>(row.size()) && e < cap; ++e) vars[e] = row[e];
    return static_cast<int>(row.size());
}

pu_status pu_ldpc_decode_batch(pu_ldpc* h, const float* llr, size_t llr_stride, size_t B, uint8_t* info_bytes,
                               size_t info_stride, uint8_t* ok, int32_t* iters, pu_memspace space, void* stream) {
    PU_REQUIRE(h, "pu_ldpc_decode_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(llr && info_bytes, "pu_ldpc_decode_batch: NULL data pointer");
    PU_REQUIRE(llr_stride >= PU_LDPC_N, "pu_ldpc_decode_batch: llr_stride < 648");
    const size_t kb = static_cast<size_t>((h->code.k + 7) / 8);
    PU_REQUIRE(info_stride >= kb, "pu_ldpc_decode_batch: info_stride too small for k bits");
    pu_ctx* ctx = h->ctx;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_DEVICE) return launch_decode(h, llr, llr_stride, B, info_bytes, info_stride, ok, iters, st);

    pu::HostStage hs(ctx, st, B);
    const float* d_llr;
    uint8_t *d_info, *d_ok;
    int32_t* d_iters;
    hs.in(&d_llr, llr, PU_LDPC_N, llr_stride);
    hs.out(&d_info, info_bytes, kb, info_stride);
    hs.out(&d_ok, ok, 1);
    hs.out(&d_iters, iters, 1);
    return hs.run([&](size_t nb) { return launch_decode(h, d_llr, PU_LDPC_N, nb, d_info, kb, d_ok, d_iters, st); });
}

pu_status pu_ldpc_decode_soft(pu_ldpc* h, const float* llr, size_t n_llr, uint8_t* out, size_t out_cap,
                              size_t* out_len, int* last_success, int* last_iters) {
    PU_REQUIRE(h && out_len, "pu_ldpc_decode_soft: NULL argument");
    *out_len = 0;
    if (n_llr == 0) {   // ldpc_decoder.cpp:285-288
        h->last_success = 0;
        if (last_success) *last_success = 0;
        if (last_iters) *last_iters = h->last_iters;
        return PU_OK;
    }
    PU_REQUIRE(llr && out, "pu_ldpc_decode_soft: NULL data pointer");
    const size_t n = PU_LDPC_N, k = static_cast<size_t>(h->code.k), kb = (k + 7) / 8;
    const size_t nblk = (n_llr + n - 1) / n;
    const size_t need = nblk == 1 ? kb : (nblk * k + 7) / 8;
    PU_REQUIRE(out_cap >= need, "pu_ldpc_decode_soft: output buffer too small");
    // zero-padded block matrix (LLR 0 = erasure, :160-166 and :396-399)
    std::vector<float> padded(nblk * n, 0.0f);
    std::memcpy(padded.data(), llr, n_llr * sizeof(float));
    std::vector<uint8_t> info(nblk * kb), okv(nblk);
    std::vector<int32_t> itv(nblk);
    pu_status s = pu_ldpc_decode_batch(h, padded.data(), n, nblk, info.data(), kb, okv.data(), itv.data(), PU_MEM_HOST, nullptr);
    if (s != PU_OK) return s;
    if (nblk == 1) {
        std::memcpy(out, info.data(), kb);
        *out_len = kb;
        h->last_success = okv[0];
    } else {
        // bit-level concatenation of the k info bits of every block (:386-427)
        std::memset(out, 0, need);
        size_t pos = 0;
        for (size_t b = 0; b < nblk; ++b)
            for (size_t j = 0; j < k; ++j, ++pos)
                if ((info[b * kb + (j >> 3)] >> (7 - (j & 7))) & 1) out[pos >> 3] |= static_cast<uint8_t>(1u << (7 - (pos & 7)));
        *out_len = need;
        const bool partial = (n_llr % n) != 0;
        int success = 1;
        for (size_t b = 0; b + (partial ? 1 : 0) < nblk; ++b) success &= okv[b];
        if (partial) success = okv[nblk - 1];   // decodeBP on the padded tail overwrites last_success (:400, :178,233)
        h->last_success = success;
    }
    h->last_iters = itv[nblk - 1];              // lastIterations() reflects the last block decoded (:332)
    if (last_success) *last_success = h->last_success;
    if (last_iters) *last_iters = h->last_iters;
    return PU_OK;
}

pu_status pu_ldpc_decode_hard(pu_ldpc* h, const uint8_t* coded, size_t n_bytes, uint8_t* out, size_t out_cap,
                              size_t* out_len, int* last_success, int* last_iters) {
    PU_REQUIRE(h && out_len, "pu_ldpc_decode_hard: NULL argument");
    std::vector<float> llr(n_bytes * 8);
    for (size_t i = 0; i < n_bytes; ++i)
        for (int b = 7; b >= 0; --b) llr[i * 8 + (7 - b)] = ((coded[i] >> b) & 1) ? -6.0f : 6.0f;   // :272-278
    return pu_ldpc_decode_soft(h, llr.data(), llr.size(), out, out_cap, out_len, last_success, last_iters);
}

pu_status pu_ldpc_encode(int code_rate, const uint8_t* data, size_t n_bytes, uint8_t* out, size_t out_cap,
                         size_t* out_len) {
    PU_REQUIRE(out_len, "pu_ldpc_encode: NULL out_len");
    static thread_local pu::LdpcCode cache;
    static thread_local bool have = false;
    if (!have || cache.rate != code_rate) {
        cache = pu::build_ldpc_code(code_rate);
        have = true;
    }
    std::vector<uint8_t> cw = pu::ldpc_encode(cache, data, n_bytes);
    *out_len = cw.size();
    PU_REQUIRE(out_cap >= cw.size(), "pu_ldpc_encode: output buffer too small");
    if (!cw.empty()) std::memcpy(out, cw.data(), cw.size());
    return PU_OK;
}

static size_t gcd_sz(size_t a, size_t b) {
    while (b) { const size_t t = a % b; a = b; b = t; }
    return a;
}

pu_status pu_channel_interleaver_perm(size_t bps, size_t total, uint32_t* perm, uint32_t* inv, size_t* step_out) {
    PU_REQUIRE(total > 0 && bps > 0, "pu_channel_interleaver_perm: zero size");
    // findCoprimeStep, ldpc_decoder.cpp:547-572: first step >= 3*bits_per_symbol coprime with total
    size_t want = bps * 3;
    if (want >= total) want = total / 2;
    size_t step = 0;
    for (size_t s = want; s < total && !step; ++s)
        if (gcd_sz(s, total) == 1) step = s;
    for (size_t s = bps + 1; s < total && !step; ++s)
        if (gcd_sz(s, total) == 1) step = s;
    if (!step) step = bps + 1;
    if (step_out) *step_out = step;
    for (size_t i = 0; i < total; ++i) {
        const size_t d = (i * step) % total;
        if (perm) perm[i] = static_cast<uint32_t>(d);
        if (inv) inv[d] = static_cast<uint32_t>(i);
    }
    return PU_OK;
}

}  // extern "C"

namespace pu {

uint32_t channel_interleaver_inverse_step(size_t bits_per_symbol) {
    size_t step = 0;
    pu_channel_interleaver_perm(bits_per_symbol, PU_LDPC_N, nullptr, nullptr, &step);
    for (uint32_t x = 1; x < PU_LDPC_N; ++x)
        if (step * x % PU_LDPC_N == 1) return x;
    return 0;      // unreachable: the step is coprime with 648
}

void channel_interleave_codewords(size_t bits_per_symbol, uint8_t* coded, size_t n_cw) {
    const uint32_t inv = channel_interleaver_inverse_step(bits_per_symbol);
    uint8_t cw[PU_LDPC_N / 8];
    for (size_t c = 0; c < n_cw; ++c) {
        uint8_t* in = coded + c * (PU_LDPC_N / 8);
        std::memset(cw, 0, sizeof cw);
        for (uint32_t j = 0; j < PU_LDPC_N; ++j) {      // out[perm[i]] = in[i]: bit j is coded bit j * step^-1
            const uint32_t i = j * inv % PU_LDPC_N;
            cw[j >> 3] |= static_cast<uint8_t>(((in[i >> 3] >> (7 - (i & 7))) & 1u) << (7 - (j & 7)));
        }
        std::memcpy(in, cw, sizeof cw);
    }
}

}  // namespace pu

extern "C" {

pu_status pu_block_interleaver_perm(size_t rows, size_t cols, uint32_t* perm) {
    PU_REQUIRE(perm && rows && cols, "pu_block_interleaver_perm: bad argument");
    for (size_t i = 0; i < rows * cols; ++i) perm[i] = static_cast<uint32_t>((i % cols) * rows + i / cols);
    return PU_OK;
}

}  // extern "C"
