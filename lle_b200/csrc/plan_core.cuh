// Planning core (plan.cu, lle_plan): exact shortest death-free joint plans by breadth-first search over joint states.
//
// A state is what TinyWorld (tiny_core.cuh) keeps in its record after reset or after a step; the search never rebuilds a
// record from a key (no set_state): every frontier entry carries its full record (<= 8 words) next to its key.
//   key        mixed-radix index of each agent's cell among the map's standable cells (not wall, not laser source, not void):
//              key = sum_a idx(a) * n_cells^a; with LLE_PLAN_ALL_GEMS also + collected-gem mask * n_cells^A.
//              K = n_cells^A (* 2^G) <= kPlanMaxKeys.
//   expansion  every joint action of the product of the agents' available actions (the record's availability cache): copy the
//              record, TinyWorld::step, drop the successor if an agent died, recompute the availability cache.
//   goal       n_arrived == A (and, with LLE_PLAN_ALL_GEMS, every gem collected).  A state where every agent has arrived is
//              never expanded (the episode is over).
//   parent     a key first reached at depth d+1 keeps, as its parent, the smallest (parent key, joint action index) among its
//              predecessors at depth d; joint action index = sum_a act[a] * 5^a.  The table word of a key is
//              depth << 42 | parent key << 10 | joint action index, lowered by a 64-bit min: a key reached at an earlier depth
//              keeps its entry, and the winner of a depth does not depend on the order of the claims.
//   stop       after the first depth that reaches a goal (the plan ends at its smallest goal key), when the next frontier is
//              empty, or after max_steps depths.  n_states counts the keys reached until then (the start included).
// The device kernel (plan.cu) and plan_map_host below run the same search: the same plan and counts whatever the schedule.
#pragma once
#include <vector>

#include "map_compiler.hpp"
#include "tiny_core.cuh"

#define LLE_PLAN_MAX_AGENTS 4
#define LLE_PLAN_MAX_STEPS 1024

namespace lle {

constexpr int64_t kPlanMaxKeys = int64_t(1) << 22;  // K of one map: the claim table has K entries of 8 bytes (32 MB at most)
constexpr uint64_t kPlanEmpty = ~uint64_t(0);

// What the search needs of one map, derived from its compiled blob by plan_prepare
struct PlanSpec {
    int A = 0, G = 0, W = 0, n_cells = 0, n_words = 0;
    bool all_gems = false;
    int64_t K = 0;
    TinyLayout L{};
    std::vector<uint16_t> cell_index;  // [H*W]: index among the standable cells, 0xFFFF elsewhere
};

// Check the limits of one map and derive its PlanSpec.  Returns LLE_OK or LLE_LIMIT_EXCEEDED / LLE_INVALID_ARGUMENT with *why.
inline int plan_prepare(const uint8_t* blob, bool all_gems, PlanSpec& s, const char** why) {
    const LleMapHeader* hdr = reinterpret_cast<const LleMapHeader*>(blob);
    if (hdr->random_starts) { *why = "the map has random start candidates"; return LLE_INVALID_ARGUMENT; }
    if (hdr->A > LLE_PLAN_MAX_AGENTS) { *why = "more than 4 agents"; return LLE_LIMIT_EXCEEDED; }
    const LleBeam* beams = reinterpret_cast<const LleBeam*>(blob + hdr->beams_off);
    int max_len = 0;
    for (int b = 0; b < hdr->NB; ++b) max_len = beams[b].len > max_len ? beams[b].len : max_len;
    const LleStateLayout L = lle_state_layout(hdr->A, hdr->G, hdr->NB, max_len);
    if (L.n_words > 8 || L.on_words != 1 || L.gem_words > 1) {
        *why = "the engine record exceeds 8 words, one word per beam (<= 32 cells) and one gem word (<= 32 gems)";
        return LLE_LIMIT_EXCEEDED;
    }
    s.A = hdr->A; s.G = hdr->G; s.W = hdr->W; s.n_words = L.n_words; s.all_gems = all_gems;
    s.L = TinyLayout{L.w_flags, L.w_avail, L.w_gems, L.w_on, L.stride, L.gem_words != 0};
    const uint32_t* cellinfo = reinterpret_cast<const uint32_t*>(blob + hdr->cellinfo_off);
    s.cell_index.assign((size_t)(hdr->H * hdr->W), 0xFFFFu);
    s.n_cells = 0;
    for (int c = 0; c < hdr->H * hdr->W; ++c) {
        const uint32_t kind = cellinfo[c] & 7u;
        if (kind != LLE_T_WALL && kind != LLE_T_VOID) s.cell_index[(size_t)c] = (uint16_t)s.n_cells++;
    }
    double K = 1;
    for (int a = 0; a < s.A; ++a) K *= s.n_cells;
    if (all_gems) K *= (double)(uint64_t(1) << s.G);
    if (K > (double)kPlanMaxKeys) { *why = "more than 2^22 joint states (n_cells^n_agents, times 2^n_gems with all_gems)"; return LLE_LIMIT_EXCEEDED; }
    s.K = (int64_t)K;
    return LLE_OK;
}

// The per-thread view of the search on one map: TinyWorld over a record reached through Rec
template <int A_, class Rec>
struct PlanWorld {
    TinyWorld<A_, Rec> w;
    const uint16_t* cell_index;
    uint32_t n_cells;
    bool all_gems;

    LLE_HD uint32_t avail_cache() const {
        uint32_t cache = 0;
        LLE_UNROLL
        for (int a = 0; a < A_; ++a) cache |= w.available(a) << (8 * a);
        return cache;
    }
    LLE_HD uint32_t key() {
        uint32_t k = 0;
        if (all_gems && w.L.has_gems) k = w.rec(w.L.w_gems);
        LLE_UNROLL
        for (int a = A_ - 1; a >= 0; --a) k = k * n_cells + cell_index[w.cellof(w.pos[a])];
        return k;
    }
    LLE_HD bool goal() { return w.n_arrived == (uint32_t)A_ && (!all_gems || !w.L.has_gems || w.rec(w.L.w_gems) == len_mask32(w.hdr->G)); }
    // World::reset into the record; returns the start key
    LLE_HD uint32_t reset() {
        w.reset();
        w.pack(avail_cache());
        return key();
    }
    // joint action `j` from the state in the record (which must not be over): false when an action is unavailable or an agent
    // dies; otherwise the record holds the successor and *k its key
    LLE_HD bool expand(uint32_t j, uint32_t* k) {
        w.unpack();
        const uint32_t cache = w.rec(w.L.w_avail);
        uint32_t act[A_], ev[A_];
        LLE_UNROLL
        for (int a = 0; a < A_; ++a) {
            act[a] = j % 5u;
            j /= 5u;
            if (!((cache >> (8 * a + act[a])) & 1u)) return false;
        }
        uint32_t n_gem, n_exit, n_died;
        w.step(act, ev, n_gem, n_exit, n_died);
        if (n_died) return false;
        w.pack(avail_cache());
        *k = key();
        return true;
    }
};

LLE_HD uint64_t plan_claim(uint32_t depth, uint32_t parent_key, uint32_t j) {
    return (uint64_t)depth << 42 | (uint64_t)parent_key << 10 | j;
}
// actions[max_steps][4] of the plan that ends in `goal` at depth `length` (rows past the plan and agents past A stay -1)
template <class Table>
LLE_HD void plan_walk_back(const Table& table, uint32_t goal, int length, int A, int8_t* actions) {
    uint32_t k = goal;
    for (int t = length - 1; t >= 0; --t) {
        const uint64_t e = table[k];
        uint32_t j = (uint32_t)(e & 1023u);
        for (int a = 0; a < A; ++a) {
            actions[4 * t + a] = (int8_t)(j % 5u);
            j /= 5u;
        }
        k = (uint32_t)((e >> 10) & 0xFFFFFFFFu);
    }
}

// ---- the search on the host: the same rules as lle_plan_kernel, one claim after the other (the CPU test-suite's reference)
struct PlanResult {
    int32_t length = -1;
    int64_t n_states = 0;
};
struct PlanArrayRec {
    uint32_t* base;
    uint32_t& operator()(int word) const { return base[word]; }
};

template <int A_>
PlanResult plan_map_host(const uint8_t* blob, const PlanSpec& s, int max_steps, int8_t* actions) {
    PlanResult r;
    const int nw = s.n_words;
    std::vector<uint64_t> table((size_t)s.K, kPlanEmpty);
    std::vector<uint32_t> cur, next;  // entries of 1 + nw words: key, record
    uint32_t rec[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    PlanWorld<A_, PlanArrayRec> pw;
    pw.w.rec = PlanArrayRec{rec};
    pw.w.L = s.L;
    pw.w.W = s.W;
    pw.w.bind(blob);
    pw.cell_index = s.cell_index.data();
    pw.n_cells = (uint32_t)s.n_cells;
    pw.all_gems = s.all_gems;
    const uint32_t k0 = pw.reset();
    table[k0] = 0;
    r.n_states = 1;
    pw.w.unpack();
    if (pw.goal()) { r.length = 0; return r; }
    if (pw.w.n_arrived == (uint32_t)A_) return r;
    cur.push_back(k0);
    cur.insert(cur.end(), rec, rec + nw);
    uint32_t J = 1;
    for (int a = 0; a < A_; ++a) J *= 5;
    for (int depth = 0; depth < max_steps && !cur.empty(); ++depth) {
        uint32_t best_goal = 0xFFFFFFFFu;
        next.clear();
        for (size_t e = 0; e < cur.size(); e += (size_t)(1 + nw)) {
            for (uint32_t j = 0; j < J; ++j) {
                for (int q = 0; q < nw; ++q) rec[q] = cur[e + 1 + (size_t)q];
                uint32_t k;
                if (!pw.expand(j, &k)) continue;
                const uint64_t claim = plan_claim((uint32_t)depth + 1, cur[e], j);
                const uint64_t old = table[k];
                if (claim < old) table[k] = claim;
                if (old != kPlanEmpty) continue;
                ++r.n_states;
                if (pw.goal()) { best_goal = k < best_goal ? k : best_goal; continue; }
                if (pw.w.n_arrived == (uint32_t)A_) continue;
                next.push_back(k);
                next.insert(next.end(), rec, rec + nw);
            }
        }
        if (best_goal != 0xFFFFFFFFu) {
            r.length = depth + 1;
            plan_walk_back(table, best_goal, r.length, A_, actions);
            return r;
        }
        cur.swap(next);
    }
    return r;
}

// lle_plan (include/lle_b200.h) on compiled maps: validates everything, then searches on the device (plan.cu)
int plan_run(const CompiledMap* const* maps, int32_t n_maps, int32_t max_steps, uint32_t flags, int32_t device, int32_t* length,
             int64_t* n_states, int8_t* actions);

}  // namespace lle
