// Expert core (expert.cu, lle_vec_expert_*): exact distance-to-goal tables over every reachable joint state of a map, with the
// optimal joint action of each state.
//
// State, key, step, goal and limits are those of the planner (plan_core.cuh: PlanWorld, plan_prepare).  Two phases:
//   forward    every state reachable from World::reset through death-free transitions, with no depth cap and without stopping
//              at the first goal; a state where every agent has arrived is not expanded.
//   backward   level d = 1, 2, ...: every reached state whose distance is still open scans its joint actions j = sum_a act[a] * 5^a
//              in increasing order; the first death-free successor whose word says dist d - 1 resolves it (dist d, joint j).  A word
//              written in level d holds d, never d - 1, so the result does not depend on the order of the states.  The build stops
//              after the first level that resolves nothing; the states still open have no death-free way to a goal.
// dist(s) is thus the length of a shortest death-free path from s to a goal, and joint(s) the smallest joint action index that
// starts one: the table is unique, and expert_map_host below (one item after the other) and the device build (expert.cu) give
// the same bytes.
//
// Table word of a key (32 bits): dist << 10 | joint for a resolved state (a goal: 0).  K <= 2^22 keys, so a distance (at most
// the number of reached states minus one) fits the 22 upper bits, and the sentinels below, whose joint field is >= 1021 (a joint
// action index is < 625), are no resolved word.
#pragma once
#include <vector>

#include "plan_core.cuh"

namespace lle {

constexpr uint32_t kExpertEmpty = 0xFFFFFFFFu;  // not reached
constexpr uint32_t kExpertOpen = 0xFFFFFFFEu;   // reached, distance not known yet
constexpr uint32_t kExpertNone = 0xFFFFFFFDu;   // reached, no death-free way to a goal

constexpr LLE_HD uint32_t expert_joint_count(int A) { return A == 1 ? 5u : A == 2 ? 25u : A == 3 ? 125u : 625u; }
// -2 not reached, -1 no way to a goal, else the distance
LLE_HD int32_t expert_dist(uint32_t w) { return w == kExpertEmpty ? -2 : w >= kExpertNone ? -1 : (int32_t)(w >> 10); }
// the word of a state when it is first reached (the successor just stepped into pw's record): a goal is resolved at once, a
// state where everybody has arrived without being a goal (missing gems with all_gems) is a dead end
template <int A_, class Rec>
LLE_HD uint32_t expert_first_word(PlanWorld<A_, Rec>& pw) {
    if (pw.goal()) return 0u;
    return pw.w.n_arrived == (uint32_t)A_ ? kExpertNone : kExpertOpen;
}
// One backward item: the state in pw's record (copied in by `load`) at level d.  Returns the resolved word, or kExpertOpen.
template <int A_, class Rec, class Load>
LLE_HD uint32_t expert_resolve(PlanWorld<A_, Rec>& pw, const uint32_t* table, uint32_t d, Load load) {
    constexpr uint32_t J = expert_joint_count(A_);
    for (uint32_t j = 0; j < J; ++j) {
        load();
        uint32_t k;
        if (!pw.expand(j, &k)) continue;
        const uint32_t w = table[k];
        if (w < kExpertNone && (w >> 10) == d - 1u) return d << 10 | j;
    }
    return kExpertOpen;
}

// ---- the build on the host: the same rules as the device build, one item after the other (the CPU test-suite's reference).
// table: K words (resized here).  Returns the number of reached states.
template <int A_>
int64_t expert_map_host(const uint8_t* blob, const PlanSpec& s, std::vector<uint32_t>& table) {
    const int nw = s.n_words;
    constexpr uint32_t J = expert_joint_count(A_);
    table.assign((size_t)s.K, kExpertEmpty);
    std::vector<uint32_t> states;  // reached states in order of discovery, 1 + nw words each: key, record
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
    pw.w.unpack();
    table[k0] = expert_first_word(pw);
    states.push_back(k0);
    states.insert(states.end(), rec, rec + nw);
    const size_t ew = (size_t)(1 + nw);
    auto load = [&](size_t e) {
        for (int q = 0; q < nw; ++q) rec[q] = states[e * ew + 1 + (size_t)q];
    };
    // forward: a breadth-first enumeration (depth by depth, as the device build runs it; the order changes nothing in the table)
    for (size_t e = 0; e < states.size() / ew; ++e) {
        load(e);
        pw.w.unpack();
        if (pw.w.n_arrived == (uint32_t)A_) continue;
        for (uint32_t j = 0; j < J; ++j) {
            load(e);
            uint32_t k;
            if (!pw.expand(j, &k) || table[k] != kExpertEmpty) continue;
            table[k] = expert_first_word(pw);
            states.push_back(k);
            states.insert(states.end(), rec, rec + nw);
        }
    }
    const int64_t n_states = (int64_t)(states.size() / ew);
    // backward levels over the open states
    std::vector<size_t> open, next;
    for (size_t e = 0; e < (size_t)n_states; ++e)
        if (table[states[e * ew]] == kExpertOpen) open.push_back(e);
    for (uint32_t d = 1; !open.empty(); ++d) {
        next.clear();
        for (size_t e : open) {
            const uint32_t w = expert_resolve(pw, table.data(), d, [&] { load(e); });
            if (w == kExpertOpen) next.push_back(e);
            else table[states[e * ew]] = w;
        }
        if (next.size() == open.size()) break;
        open.swap(next);
    }
    for (size_t e : open) table[states[e * ew]] = kExpertNone;
    return n_states;
}

// dist i32[n] / joint i16[n] of the API (include/lle_b200.h: lle_vec_expert_table) from table words
inline void expert_decode(const uint32_t* words, int64_t n, int32_t* dist, int16_t* joint) {
    for (int64_t i = 0; i < n; ++i) {
        const int32_t d = expert_dist(words[i]);
        if (dist) dist[i] = d;
        if (joint) joint[i] = d > 0 ? (int16_t)(words[i] & 1023u) : (int16_t)-1;
    }
}

// ---- the vec's side (vec_world.cu unwraps the handle; expert.cu builds and queries)
struct ExpertTables;  // device tables of one build, owned by the vec
void expert_free(ExpertTables* t);

struct ExpertVecView {
    int device = 0;
    int64_t N = 0;
    int A = 0, G = 0, W = 0;
    LleStateLayout L{};
    const uint32_t* records = nullptr;     // [N_pad][L.stride]
    const int32_t* map_of_env = nullptr;   // [N_pad] or null (every env on map 0)
    std::vector<const uint8_t*> blobs;     // device blob of every map, as the vec steps it
    std::vector<const CompiledMap*> maps;  // the same maps compiled on the host
};
// lle_vec_expert_build / _act / _table once vec_world.cu has checked the vec-level conditions
int expert_build(const ExpertVecView& v, uint32_t flags, int64_t* n_states, void* stream, ExpertTables** out);
int expert_act(const ExpertVecView& v, const ExpertTables* t, int8_t* actions, int32_t* dist, void* stream);
int expert_table(const ExpertTables* t, int32_t map_index, int32_t* dist, int16_t* joint, int64_t cap, int64_t* n_keys);

}  // namespace lle
