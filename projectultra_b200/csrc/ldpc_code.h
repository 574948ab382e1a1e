// projectultra_b200/csrc/ldpc_code.h — host-side construction of the reference's LDPC code and of the
// device tables the decoder kernel walks.
#pragma once
#include <cstdint>
#include <vector>

namespace pu {

constexpr int kLdpcN = 648;
constexpr int kMaxInfoEdgesPerCheck = 6;  // max_check_degree, src/fec/ldpc_decoder.cpp:87

struct LdpcCode {
    int rate = 0, k = 0, m = 0, n_edges = 0;
    // rows[i] = variable indices of check i in the reference's stored order: info bits in construction
    // order, optional fix-up bit, then the identity column k+i (src/fec/ldpc_decoder.cpp:89-128)
    std::vector<std::vector<int>> rows;
    int max_var_degree = 0;
};

// CodeRate enum -> (k, m); unknown rates fall back to R1/2 sizes (getCodeParams, ldpc_decoder.cpp:21-36)
void ldpc_code_params(int rate, int* k, int* m);
// H = [H_data | I] exactly as LDPCDecoder::Impl::buildMatrix (ldpc_decoder.cpp:64-137)
LdpcCode build_ldpc_code(int rate);
// systematic encoder, LDPCEncoder::encode (src/fec/ldpc_encoder.cpp:193-257)
std::vector<uint8_t> ldpc_encode(const LdpcCode& code, const uint8_t* data, size_t n_bytes);

// Flat tables in the layout ldpc_decode.cu expects.  Checks are visited in "slot" order p (sorted by
// descending info degree so that a warp sees one loop bound); messages of slot p, edge e live at e*m + p.
struct LdpcHostTables {
    int k = 0, m = 0, dv_max = 0;
    std::vector<uint8_t> cn_ninfo;   // [m]      info edges of slot p
    std::vector<uint16_t> cn_check;  // [m]      original check index of slot p (parity variable = k + check)
    std::vector<uint16_t> cn_var;    // [6][m]   info variable of (edge e, slot p), 0xFFFF if absent
    std::vector<uint8_t> vn_deg;     // [k]      degree of info variable j
    std::vector<uint16_t> vn_slot;   // [dv_max][k] message slot of j's d-th edge in ASCENDING CHECK ORDER
                                     //          (the accumulation order of ldpc_decoder.cpp:208-213)
};
LdpcHostTables make_ldpc_tables(const LdpcCode& code);

// Bank-conflict-free layout for the register-resident decoder kernel (ldpc_flood_reg_kernel in ldpc_decode.cu).
//   * thread p < m owns check slot p (checks sorted by descending info degree, 32 per warp);
//   * information bit j lives in "variable slot" a(j) < kpad: its total is tot[a], its d-th incoming message
//     (d = rank of the check among j's checks in ASCENDING CHECK ORDER, the accumulation order of
//     ldpc_decoder.cpp:208-213) is msg[d * kpad + a];
//   * a(j) and the order of the edges inside every check are chosen so that the 32 lanes of a warp touch 32
//     different shared-memory banks (a mod 32) on every edge instruction: variables get banks by local search
//     until no warp uses a bank more often than its longest row, then each warp's (check x bank) bipartite
//     multigraph is edge-coloured (Koenig) with one colour per edge instruction.  conflicts = what is left over.
struct LdpcLayout {
    int k = 0, m = 0, threads = 0, kpad = 0, dv = 0, vr = 0;
    int inf_slot = 0;      // tot[] word that holds +INF (absent check-side edges read it)
    int scratch_slot = 0;  // msg[] word that absorbs the writes of absent edges
    int tot_words = 0, msg_words = 0;
    std::vector<uint8_t> cn_ninfo;    // [threads] info edges of slot p (0 for p >= m)
    std::vector<uint16_t> cn_check;   // [threads] original check index of slot p
    std::vector<uint16_t> cn_rd;      // [6][threads] tot[] index read by edge e of slot p
    std::vector<uint16_t> cn_wr;      // [6][threads] msg[] index written by edge e of slot p
    std::vector<uint16_t> var_slot;   // [k]    a(j)
    std::vector<int16_t> slot_var;    // [kpad] j or -1
    std::vector<uint8_t> slot_deg;    // [kpad] checks of the bit in slot a (0 for an empty slot): msg[d * kpad + a] is written
                                      //        by a check exactly for d < slot_deg[a]
    int conflicts = 0;                // extra shared-memory wavefronts per iteration that the layout could not remove
};
LdpcLayout make_ldpc_layout(const LdpcCode& code);

}  // namespace pu
