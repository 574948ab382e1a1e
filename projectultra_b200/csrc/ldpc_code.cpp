// projectultra_b200/csrc/ldpc_code.cpp — see ldpc_code.h.
#include "ldpc_code.h"

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <random>
#include <stdexcept>

namespace pu {

void ldpc_code_params(int rate, int* k, int* m) {
    static const struct { int rate, k; } tab[] = {{0, 162}, {2, 324}, {3, 432}, {4, 486}, {5, 540}};
    *k = 324;
    for (const auto& t : tab)
        if (t.rate == rate) *k = t.k;
    *m = kLdpcN - *k;
}

LdpcCode build_ldpc_code(int rate) {
    LdpcCode c;
    c.rate = rate;
    ldpc_code_params(rate, &c.k, &c.m);
    const int k = c.k, m = c.m;
    c.rows.assign(m, {});

    // The pseudo-random graph is grown one information bit at a time from a generator seeded with the rate
    // enum (ldpc_decoder.cpp:72).  std::mt19937 is bit-exact across standard libraries; the shuffle is the
    // reference's hand-rolled Fisher-Yates (`rng() % i`, :100-103), not std::shuffle.
    std::mt19937 gen(static_cast<uint32_t>(0x12345678 + rate));
    const int per_bit = std::min(std::max(3, (4 * m) / k), m / 2);   // target_var_degree, :82-84
    std::vector<int> load(m, 0);
    std::vector<int> open;
    open.reserve(m);
    for (int bit = 0; bit < k; ++bit) {
        open.clear();
        for (int chk = 0; chk < m; ++chk)
            if (load[chk] < kMaxInfoEdgesPerCheck) open.push_back(chk);
        for (size_t top = open.size(); top > 1; --top) std::swap(open[top - 1], open[gen() % top]);
        const int take = std::min<int>(per_bit, static_cast<int>(open.size()));
        for (int d = 0; d < take; ++d) {
            c.rows[open[d]].push_back(bit);
            ++load[open[d]];
        }
    }
    for (int chk = 0; chk < m; ++chk)                 // empty-row fix-up draws from the same stream, :115-121
        if (c.rows[chk].empty()) c.rows[chk].push_back(static_cast<int>(gen() % k));
    std::vector<int> vdeg(k, 0);
    for (int chk = 0; chk < m; ++chk) {
        for (int v : c.rows[chk]) ++vdeg[v];
        c.rows[chk].push_back(k + chk);               // identity part, :124-128
        c.n_edges += static_cast<int>(c.rows[chk].size());
    }
    c.max_var_degree = *std::max_element(vdeg.begin(), vdeg.end());
    return c;
}

std::vector<uint8_t> ldpc_encode(const LdpcCode& code, const uint8_t* data, size_t n_bytes) {
    const size_t k = code.k, m = code.m, n = k + m, total = n_bytes * 8;
    std::vector<uint8_t> out;
    std::vector<uint8_t> word(n);
    for (size_t start = 0; start < total; start += k) {     // k bits per block, zero padded (:214-219)
        for (size_t j = 0; j < k; ++j) {
            const size_t b = start + j;
            word[j] = b < total ? (data[b >> 3] >> (7 - (b & 7))) & 1 : 0;
        }
        for (size_t i = 0; i < m; ++i) {                    // parity_i = XOR of row i's info bits (:221-230)
            uint8_t acc = 0;
            const auto& row = code.rows[i];
            for (size_t e = 0; e + 1 < row.size(); ++e) acc ^= word[row[e]];
            word[k + i] = acc;
        }
        for (size_t base = 0; base < n; base += 8) {        // MSB-first, 81 bytes per block (:237-250)
            uint8_t byte = 0;
            for (size_t b = 0; b < 8; ++b) byte = static_cast<uint8_t>((byte << 1) | (base + b < n ? word[base + b] : 0));
            out.push_back(byte);
        }
    }
    return out;
}

LdpcHostTables make_ldpc_tables(const LdpcCode& code) {
    LdpcHostTables t;
    t.k = code.k;
    t.m = code.m;
    const int k = code.k, m = code.m;
    std::vector<int> slot_of(m), order(m);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(),
                     [&](int a, int b) { return code.rows[a].size() > code.rows[b].size(); });
    t.cn_ninfo.resize(m);
    t.cn_check.resize(m);
    t.cn_var.assign(static_cast<size_t>(kMaxInfoEdgesPerCheck) * m, 0xFFFF);
    for (int p = 0; p < m; ++p) {
        const int chk = order[p];
        slot_of[chk] = p;
        const auto& row = code.rows[chk];
        const int ninfo = static_cast<int>(row.size()) - 1;
        if (ninfo > kMaxInfoEdgesPerCheck) throw std::logic_error("check degree exceeds table width");
        t.cn_ninfo[p] = static_cast<uint8_t>(ninfo);
        t.cn_check[p] = static_cast<uint16_t>(chk);
        for (int e = 0; e < ninfo; ++e) t.cn_var[static_cast<size_t>(e) * m + p] = static_cast<uint16_t>(row[e]);
    }
    // variable side: walk checks in ascending index so each list is already in the reference's summation order
    std::vector<std::vector<uint16_t>> per_var(k);
    for (int chk = 0; chk < m; ++chk) {
        const auto& row = code.rows[chk];
        for (size_t e = 0; e + 1 < row.size(); ++e)
            per_var[row[e]].push_back(static_cast<uint16_t>(e * m + slot_of[chk]));
    }
    t.dv_max = 0;
    for (const auto& v : per_var) t.dv_max = std::max<int>(t.dv_max, static_cast<int>(v.size()));
    t.vn_deg.resize(k);
    t.vn_slot.assign(static_cast<size_t>(std::max(t.dv_max, 1)) * k, 0xFFFF);
    for (int j = 0; j < k; ++j) {
        t.vn_deg[j] = static_cast<uint8_t>(per_var[j].size());
        for (size_t d = 0; d < per_var[j].size(); ++d) t.vn_slot[d * k + j] = per_var[j][d];
    }
    return t;
}

namespace {

// Proper edge colouring of a bipartite multigraph (left = checks of one warp, right = banks) with `ncol` colours by
// alternating-path recolouring.  Edges whose endpoints both have degree <= ncol always get a proper colour; edges at
// an over-full bank fall back to any colour that is free at the check (and count as a conflict).
struct WarpColouring {
    int ncol;
    std::vector<std::array<int, 8>> at_left, at_right;   // edge id occupying colour c at a vertex, or -1
    std::vector<int> el, er, colour;
    WarpColouring(int nleft, int nright, int ncol_) : ncol(ncol_) {
        std::array<int, 8> none;
        none.fill(-1);
        at_left.assign(nleft, none);
        at_right.assign(nright, none);
    }
    int free_at(const std::array<int, 8>& v) const {
        for (int c = 0; c < ncol; ++c)
            if (v[c] < 0) return c;
        return -1;
    }
    // Adds a properly coloured edge; returns false (and adds nothing) when bank r has no free colour left.
    bool add(int l, int r) {
        const int a = free_at(at_left[l]);
        const int b = free_at(at_right[r]);
        if (a < 0) throw std::logic_error("check has more edges than colours");
        if (b < 0) return false;
        const int id = static_cast<int>(el.size());
        el.push_back(l);
        er.push_back(r);
        colour.push_back(-1);
        if (at_right[r][a] >= 0) {
            // colour a is free at l but taken at r; b is free at r.  Swap a<->b along the alternating path that starts
            // at r with colour a (it cannot reach l: the graph is bipartite and a is free at l).
            std::vector<int> path;
            int v = r, want = a;
            bool on_right = true;
            for (;;) {
                const int e = on_right ? at_right[v][want] : at_left[v][want];
                if (e < 0) break;
                path.push_back(e);
                v = on_right ? el[e] : er[e];
                on_right = !on_right;
                want = (want == a) ? b : a;
                if (path.size() > el.size()) throw std::logic_error("edge colouring: alternating path does not end");
            }
            for (int e : path) {
                at_left[el[e]][colour[e]] = -1;
                at_right[er[e]][colour[e]] = -1;
            }
            for (int e : path) {
                colour[e] = (colour[e] == a) ? b : a;
                at_left[el[e]][colour[e]] = e;
                at_right[er[e]][colour[e]] = e;
            }
        }
        if (at_right[r][a] >= 0 || at_left[l][a] >= 0) throw std::logic_error("edge colouring: colour still taken");
        colour[id] = a;
        at_left[l][a] = id;
        at_right[r][a] = id;
        return true;
    }
    // An edge at an over-full bank: any colour free at the check (costs one extra wavefront).  Call after all add()s.
    int add_conflicting(int l) {
        const int a = free_at(at_left[l]);
        if (a < 0) throw std::logic_error("check has more edges than colours");
        at_left[l][a] = 1 << 30;
        return a;
    }
};

}  // namespace

LdpcLayout make_ldpc_layout(const LdpcCode& code) {
    LdpcLayout L;
    const int k = code.k, m = code.m;
    L.k = k;
    L.m = m;
    L.threads = (m + 31) / 32 * 32;
    L.dv = std::max(code.max_var_degree, 1);
    L.kpad = (k + 31) / 32 * 32;
    if (L.kpad - k < 16) L.kpad += 32;                       // slack for the bank assignment
    if (L.kpad % L.threads != 0 && L.kpad > L.threads) L.kpad = (L.kpad + 31) / 32 * 32;
    L.vr = (L.kpad + L.threads - 1) / L.threads;
    const int depth = L.kpad / 32;
    const int nwarps = L.threads / 32;

    // check slots: descending info degree (stable), 32 per warp
    std::vector<int> order(m);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return code.rows[a].size() > code.rows[b].size(); });
    std::vector<int> ne_w(nwarps, 0);
    for (int p = 0; p < m; ++p) ne_w[p / 32] = std::max<int>(ne_w[p / 32], static_cast<int>(code.rows[order[p]].size()) - 1);
    // edges of every warp and, per variable, the warps it touches
    std::vector<std::vector<int>> var_warps(k);
    for (int p = 0; p < m; ++p) {
        const auto& row = code.rows[order[p]];
        for (size_t e = 0; e + 1 < row.size(); ++e) var_warps[row[e]].push_back(p / 32);
    }

    // ---- bank assignment by local search: cost = sum over (warp, bank) of max(0, uses - longest row of the warp)
    std::mt19937 gen(0xB200u + static_cast<uint32_t>(code.rate));
    std::vector<int> bank(k), fill(32, 0);
    std::vector<std::vector<int>> uses(nwarps, std::vector<int>(32, 0));
    {
        std::vector<int> vars(k);
        std::iota(vars.begin(), vars.end(), 0);
        std::stable_sort(vars.begin(), vars.end(), [&](int a, int b) { return var_warps[a].size() > var_warps[b].size(); });
        for (int j : vars) {   // greedy: the bank that adds the least cost, ties to the emptiest bank
            int best = -1, best_cost = 1 << 30;
            for (int b = 0; b < 32; ++b) {
                if (fill[b] >= depth) continue;
                int c = 0;
                for (int w : var_warps[j]) c += (uses[w][b] + 1 > ne_w[w]) ? 1000 : uses[w][b];
                c = c * 64 + fill[b];
                if (c < best_cost) { best_cost = c; best = b; }
            }
            bank[j] = best;
            ++fill[best];
            for (int w : var_warps[j]) ++uses[w][best];
        }
    }
    auto total_cost = [&]() {
        int c = 0;
        for (int w = 0; w < nwarps; ++w)
            for (int b = 0; b < 32; ++b) c += std::max(0, uses[w][b] - ne_w[w]);
        return c;
    };
    auto move_delta = [&](int j, int to) {   // cost change of moving variable j to bank `to`
        const int from = bank[j];
        int d = 0;
        const auto& ws = var_warps[j];
        for (size_t x = 0; x < ws.size(); ++x) {
            bool dup = false;
            for (size_t y = 0; y < x; ++y) dup |= (ws[y] == ws[x]);
            if (dup) continue;
            const int w = ws[x];
            const int c = static_cast<int>(std::count(ws.begin(), ws.end(), w));
            d += std::max(0, uses[w][from] - c - ne_w[w]) - std::max(0, uses[w][from] - ne_w[w]);
            d += std::max(0, uses[w][to] + c - ne_w[w]) - std::max(0, uses[w][to] - ne_w[w]);
        }
        return d;
    };
    auto apply_move = [&](int j, int to) {
        for (int w : var_warps[j]) { --uses[w][bank[j]]; ++uses[w][to]; }
        --fill[bank[j]];
        ++fill[to];
        bank[j] = to;
    };
    int cost = total_cost();
    // members of every bank, to pick swap partners quickly
    auto bank_members = [&](int b) {
        std::vector<int> v;
        for (int q = 0; q < k; ++q)
            if (bank[q] == b) v.push_back(q);
        return v;
    };
    std::vector<std::vector<int>> warp_vars(nwarps);   // variables touched by each warp (with multiplicity)
    for (int j = 0; j < k; ++j)
        for (int w : var_warps[j]) warp_vars[w].push_back(j);
    for (int iter = 0; iter < 3000000 && cost > 0; ++iter) {
        // targeted move: an over-used (warp, bank) pair gives up one of its variables
        int j;
        if ((iter & 3) != 3) {
            const int w = static_cast<int>(gen() % nwarps);
            if (warp_vars[w].empty()) continue;
            j = warp_vars[w][gen() % warp_vars[w].size()];
            if (uses[w][bank[j]] <= ne_w[w]) continue;
        } else {
            j = static_cast<int>(gen() % k);
            if (var_warps[j].empty()) continue;
        }
        const int to = static_cast<int>(gen() % 32);
        if (to == bank[j]) continue;
        if (fill[to] < depth) {
            const int d = move_delta(j, to);
            if (d < 0 || (d == 0 && (gen() & 1))) { apply_move(j, to); cost += d; }
        } else {
            const std::vector<int> cand = bank_members(to);
            const int q = cand[gen() % cand.size()];
            const int from = bank[j];
            const int d1 = move_delta(j, to);
            apply_move(j, to);
            const int d2 = move_delta(q, from);
            if (d1 + d2 < 0 || (d1 + d2 == 0 && (gen() & 1))) { apply_move(q, from); cost += d1 + d2; }
            else apply_move(j, from);
        }
    }

    if (getenv("PU_LDPC_LAYOUT_DEBUG")) fprintf(stderr, "rate %d: bank-assignment cost %d (recount %d), depth %d\n", code.rate, cost, total_cost(), depth);
    // ---- variable slots: a = bank + 32 * row
    L.var_slot.assign(k, 0);
    L.slot_var.assign(L.kpad, -1);
    {
        std::vector<int> next(32, 0);
        for (int j = 0; j < k; ++j) {
            const int a = bank[j] + 32 * next[bank[j]]++;
            L.var_slot[j] = static_cast<uint16_t>(a);
            L.slot_var[a] = static_cast<int16_t>(j);
        }
    }
    // rank of every check among its variables' checks, ascending check index
    std::vector<int> seen(k, 0);
    std::vector<std::vector<int>> rank(m);
    for (int chk = 0; chk < m; ++chk) {
        const auto& row = code.rows[chk];
        rank[chk].resize(row.size() - 1);
        for (size_t e = 0; e + 1 < row.size(); ++e) rank[chk][e] = seen[row[e]]++;
    }
    L.slot_deg.assign(L.kpad, 0);
    for (int j = 0; j < k; ++j) L.slot_deg[L.var_slot[j]] = static_cast<uint8_t>(seen[j]);

    L.inf_slot = L.kpad;
    L.tot_words = L.kpad + 32;    // + one +INF word per bank
    L.scratch_slot = L.dv * L.kpad;
    L.msg_words = L.dv * L.kpad + (L.threads + 31) / 32 * 32 * kMaxInfoEdgesPerCheck;   // + scratch words of the absent edges: 32 per (warp, slot)
    L.cn_ninfo.assign(L.threads, 0);
    L.cn_check.assign(L.threads, 0);
    L.cn_rd.assign(static_cast<size_t>(kMaxInfoEdgesPerCheck) * L.threads, static_cast<uint16_t>(L.inf_slot));
    L.cn_wr.assign(static_cast<size_t>(kMaxInfoEdgesPerCheck) * L.threads, 0);
    for (int e = 0; e < kMaxInfoEdgesPerCheck; ++e)
        for (int p = 0; p < L.threads; ++p)
            L.cn_wr[static_cast<size_t>(e) * L.threads + p] = static_cast<uint16_t>(L.scratch_slot + ((p >> 5) * kMaxInfoEdgesPerCheck + e) * 32 + (p & 31));

    // ---- per warp: colour the (check, bank) multigraph; the colour of an edge is its instruction slot e
    L.conflicts = 0;
    for (int w = 0; w < nwarps; ++w) {
        const int p0 = w * 32, p1 = std::min(m, p0 + 32);
        if (p0 >= m || ne_w[w] == 0) continue;
        WarpColouring col(32, 32, ne_w[w]);
        struct Ref { int p, e_row, id; };
        std::vector<Ref> placed, deferred;
        for (int p = p0; p < p1; ++p) {
            const auto& row = code.rows[order[p]];
            for (size_t e = 0; e + 1 < row.size(); ++e) {
                if (col.add(p - p0, bank[row[e]])) placed.push_back({p, static_cast<int>(e), static_cast<int>(col.el.size()) - 1});
                else deferred.push_back({p, static_cast<int>(e), -1});
            }
        }
        auto emit = [&](int p, int e_row, int e_slot) {
            const int chk = order[p];
            const int j = code.rows[chk][e_row];
            const int a = L.var_slot[j];
            L.cn_rd[static_cast<size_t>(e_slot) * L.threads + p] = static_cast<uint16_t>(a);
            L.cn_wr[static_cast<size_t>(e_slot) * L.threads + p] = static_cast<uint16_t>(rank[chk][e_row] * L.kpad + a);
        };
        std::vector<char> real(static_cast<size_t>(kMaxInfoEdgesPerCheck) * 32, 0);
        std::vector<unsigned> used(kMaxInfoEdgesPerCheck, 0u);       // banks touched by the real edges of instruction slot e
        auto emit_real = [&](int p, int e_row, int e_slot) {
            emit(p, e_row, e_slot);
            real[static_cast<size_t>(e_slot) * 32 + (p - p0)] = 1;
            used[e_slot] |= 1u << (L.cn_rd[static_cast<size_t>(e_slot) * L.threads + p] & 31);
        };
        for (const Ref& r : placed) emit_real(r.p, r.e_row, col.colour[r.id]);
        for (const Ref& r : deferred) {
            emit_real(r.p, r.e_row, col.add_conflicting(r.p - p0));
            ++L.conflicts;
        }
        // absent edges (rows shorter than the warp's longest, lanes past the last check) read a +INF word in a bank that no real
        // edge of the same instruction uses (one shared read-only address: no extra wavefront) and write a scratch word of their
        // OWN: every (warp, instruction slot) has 32 scratch words in 32 banks, and an instruction has exactly as many unused banks as
        // it has absent edges, so every absent lane gets a distinct unused bank -- no wavefront added, and no two threads ever store
        // to the same word (a shared dump word is a write-write race, harmless but flagged by compute-sanitizer --tool racecheck)
        for (int e = 0; e < ne_w[w] && e < kMaxInfoEdgesPerCheck; ++e) {
            int fb = -1;
            for (int b = 0; b < 32; ++b)
                if (!(used[e] & (1u << b))) { fb = b; break; }
            if (fb < 0) continue;
            int nb = 0;
            for (int lane = 0; lane < 32 && p0 + lane < L.threads; ++lane) {
                if (real[static_cast<size_t>(e) * 32 + lane]) continue;
                while (nb < 32 && (used[e] & (1u << nb))) ++nb;
                const int wb = nb < 32 ? nb++ : fb;
                L.cn_rd[static_cast<size_t>(e) * L.threads + p0 + lane] = static_cast<uint16_t>(L.inf_slot + fb);
                L.cn_wr[static_cast<size_t>(e) * L.threads + p0 + lane] = static_cast<uint16_t>(L.scratch_slot + (w * kMaxInfoEdgesPerCheck + e) * 32 + wb);
            }
        }
    }
    for (int p = 0; p < m; ++p) {
        L.cn_ninfo[p] = static_cast<uint8_t>(code.rows[order[p]].size() - 1);
        L.cn_check[p] = static_cast<uint16_t>(order[p]);
    }
    return L;
}

}  // namespace pu
