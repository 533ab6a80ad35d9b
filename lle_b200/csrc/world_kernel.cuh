// lle_b200 — the fused `World` step kernel for NVIDIA B200 (sm_100a).  Device code only.
//
// One launch advances N independent worlds by one joint action (or resets them, or forces a state) and
// writes every per-step output of the reference's `LLE.step`:
//   world.rs:435-475 (step) . world.rs:343-363 (availability) . reward_strategy.py:58-109 .
//   env.py:253-254 (done) . pyworld_state.rs:79-101 (state vector) . observations.py:254-266 (layered).
//
// Layout of the work (DESIGN.md §4) — "warp per world, lane per agent":
//   * A warp takes a ticket for a small group of consecutive worlds and handles them one after the other.
//   * The world's record (a few 32-bit words, contiguous in HBM) is copied into the warp's shared memory with
//     one coalesced load.  Lane a owns agent a: its position, its action, its event.  The per-agent flags
//     (alive / arrived / tile slot) are warp-uniform bitmasks maintained with __ballot_sync; the beam masks
//     (`LaserBeam.beam`) stay in shared memory and are updated with shared-memory atomics
//     (leave: OR of a suffix, pre_enter: AND of a prefix), which is order-independent exactly like the
//     reference's sequential loops (SURVEY App. A).  No thread ever scans a beam cell by cell: a per-cell
//     table gives the (at most four) beams through the cell and the agent's offset on each.
//   * The layered observation is not recomputed cell by cell either.  Each warp keeps observation tiles in
//     shared memory, initialised from the map's static plane; for the next world it un-patches the few cells
//     that depended on the previous occupant's state, patches the new ones (agents, lit laser cells,
//     uncollected gems) and hands the tile to the TMA engine with ONE `cp.async.bulk.global.shared::cta`
//     (SASS: UBLKCP) per tile.  The LSU never touches the 7.5 KB of an observation, and the store drains
//     while the warp already computes its next world.
//   * Small outputs (state vector, availability, reward, done, events, actions, err) are written by the warp
//     with coalesced stores straight from registers / the shared record.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "static_map.h"
#include "step_common.cuh"

namespace lle {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr unsigned kFull = 0xFFFFFFFFu;

enum Mode : int { MODE_STEP = 0, MODE_RESET = 1, MODE_SET_STATE = 2 };

// ---- map view -------------------------------------------------------------------------------------------
struct MapDev {
    const uint8_t* blob;
    const LleMapHeader* hdr;
    const uint32_t* cellinfo;
    const LleCellBeams* cellbeams;
    const LleBeam* beams;
    const LlePatch* patches;
    const float* stat;  // the static plane; int8_t elements when the map was compiled for an int8 observation
    const LleAgentPlane* agent_planes;
    const uint32_t* chunk_tbl;
    int n_patch, NB, obs_floats, n_ap;
    uint64_t gem_toplevel;
    __device__ __forceinline__ void bind(const uint8_t* b) {
        blob = b;
        hdr = reinterpret_cast<const LleMapHeader*>(b);
        cellinfo = reinterpret_cast<const uint32_t*>(b + hdr->cellinfo_off);
        cellbeams = reinterpret_cast<const LleCellBeams*>(b + hdr->cellbeams_off);
        beams = reinterpret_cast<const LleBeam*>(b + hdr->beams_off);
        patches = reinterpret_cast<const LlePatch*>(b + hdr->patch_off);
        stat = reinterpret_cast<const float*>(b + hdr->static_off);
        agent_planes = reinterpret_cast<const LleAgentPlane*>(b + hdr->ap_off);
        n_ap = hdr->n_ap;
        chunk_tbl = reinterpret_cast<const uint32_t*>(b + hdr->chunk_tbl_off);
        n_patch = hdr->n_patch;
        NB = hdr->NB;
        obs_floats = hdr->obs_floats;
        gem_toplevel = hdr->gem_toplevel;
    }
};

struct KParams {
    const uint8_t* const* blobs;  // device array [n_maps] of map blobs
    int32_t* map_of_env;          // device [N_pad] or nullptr: index of each env's current map blob.  With randomize_lasers the
                                  // blob table holds `n_variants` colourings per map (index = map * n_variants + variant) and a reset
                                  // rewrites the env's entry
    uint32_t* records;            // [N_pad][L.stride]
    LleStateLayout L;
    int64_t N, N_pad;
    int32_t A, G, NBmax, C, H, W, S, R, HW;
    float* obs;
    int64_t obs_stride;  // floats per env
    float* state;
    uint8_t* avail;
    float* reward;
    uint8_t* done;
    uint8_t* events;
    int8_t* actions;
    uint8_t* err;
    const int8_t* actions_in;
    const uint8_t* reset_mask;
    const int32_t* ss_pos;
    const uint8_t* ss_gems;
    const uint8_t* ss_alive;
    uint64_t seed, env_id_base, t;
    int32_t mode, auto_reset, lle_semantics, walkable, write_obs;
    // work decomposition / observation tiling
    int32_t Wd;            // lanes per world: the power of two >= n_agents (32/Wd worlds share a warp)
    int32_t group;         // worlds per ticket (multiple of E and of 32/Wd, divides 32)
    int32_t E;             // worlds per tile (n_chunks == 1)
    int32_t n_chunks;      // > 1: one world's block is streamed in chunks (E == 1)
    int32_t chunk_floats;  // floats per chunk, multiple of 4
    int32_t tile_floats;   // floats per shared-memory tile buffer
    int32_t n_buf;         // tile buffers per warp (1 or 2)
    int32_t warp_smem_bytes;
    uint32_t* sched;       // this launch's scheduler slot: [0] next (step, ticket) pair, [1] warps finished, [2] generation =
                           // completed uses of the slot (slots rotate; a launch may only touch its slot once the launch that
                           // used it before has re-armed it, see sched_gen)
    uint32_t sched_gen;    // generation this launch expects in sched[2]
    uint32_t sched_check;  // 0: the host saw the launch that used this slot before retire - no need to look at the generation
    uint32_t* retired_launch;  // host-mapped: number of launches of the vec (any mode) whose last warp has left
    uint32_t* retired_count;   // device counter behind it
    // The tables of map 0 resolved on the host (pointers into its blob): a batch on one map binds them from the parameters instead
    // of chasing blob table -> header -> tables through three dependent L2 round trips at the start of every warp.
    MapDev map0;
    int32_t has_map0, pad_map0;
    uint32_t* flags;       // [n_tickets] sequence number of the last step completed for the ticket's worlds
    uint32_t seq;          // sequence number of the (first) step of this launch; step q of a ticket needs flags >= q-1
    uint32_t n_tickets, n_warps_total;
    uint64_t* timeline;    // development aid: per warp {start, first store, last store, end} in ns (globaltimer), or nullptr
    int32_t n_steps;       // steps in this launch (> 1: rollout with device-sampled actions)
    // LaserSubgoal extras / PotentialShapedLLE
    float* extras;         // [N_pad][A][JE] or nullptr
    int32_t JE, pbrs_on;
    uint64_t extras_set, pbrs_set;  // bit b: source b is tracked
    double pbrs_gamma, pbrs_value;
    int8_t extras_beam[64];         // source index of extras column j
    // observation kind (static_map.h LLE_OBS_*): layered / perspective go through the tile renderer (write_obs), partial has
    // its own cell-by-cell renderer, state is written with the small outputs (state_obs: 1 = state, 2 = normalised)
    int32_t obs_kind, obs_param, state_obs, pad0;
    // Pipelined host stepping (lle_vec_pipeline_submit): the actions of this step arrive through a copy engine on
    // another stream, which then publishes `in_need` to *in_flag (stream memory op); the reward / done of this step are
    // duplicated into a ring slot that a third stream copies to the host once *out_flag >= out_value.
    const uint32_t* in_flag;
    uint32_t in_need, out_value;
    // Closed loop over parts of the batch (lle_vec_parts_*): the tickets of part k (part_tickets consecutive tickets) start once
    // part_in[32 k] >= in_need (a stream memory op of the host behind the copy of the part's actions into the staging buffer
    // actions_in points at), and the warp that completes the part's last ticket writes out_value to part_out[32 k]
    // (host-mapped) behind a system-scope fence: the reward / done of the part are in host memory (reward2 / done2).
    const uint32_t* part_in;
    uint32_t* part_out;
    uint32_t* part_count;  // device counters: tickets of the part completed in this step
    uint32_t part_tickets, part_last;  // tickets per part; index of the last part, which also takes the padding tickets behind N
    uint32_t* out_flag;
    float* reward2;
    uint8_t* done2;
    // host-mapped word that receives the sequence number of the last step of this launch when the launch retires: lets the
    // host see how many step launches are still in flight (a scheduling hint only, see launch_mode in vec_world.cu)
    volatile uint32_t* retired_seq;
    uint32_t reset_epoch;  // number of explicit resets of the vec so far: part of the start-sampling counter (random starts)
    int32_t randomize;     // LLE(randomize_lasers=True), env.py:198-200: every LLE-level reset recolours the sources at random
    int32_t n_variants;    // colourings per map: n_agents ^ n_sources (source b's colour = digit b in base n_agents)
    uint32_t refresh_only; // MODE_RESET launch that resets no env: re-exports observation / state / availability only
    // Step.info of LLE.step (env.py:174-188) and per-env episode statistics (lle_vec_options.episode_stats), or nullptr
    uint8_t* info;         // [N_pad][2 + A]: gems_collected, n_arrived, has-arrived flags of the transition just taken
    float* ep_return;      // [N_pad][R]  reward summed over the running episode
    int32_t* ep_length;    // [N_pad]     its steps so far
    float* last_return;    // [N_pad][R]  the same two of the last finished episode
    int32_t* last_length;  // [N_pad]
    int8_t* obs_i8;        // the observation rows of an int8 vec (lle_vec_options.obs_dtype; obs is then null).  Elements of
                           // either type are counted alike: obs_stride, tile_floats and chunk_floats count int8 elements there
};

// The observation rows as the kernel's element type OT (float, or int8_t for an int8 vec)
template <typename OT>
__device__ __forceinline__ OT* obs_rows(const KParams& p) {
    if constexpr (sizeof(OT) == 1) return p.obs_i8;
    else return p.obs;
}

// ---- PTX wrappers (TMA 1-D bulk store through the async proxy) ----------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}
// The same with an L2 eviction policy (createpolicy): observation rows are written once per step and not read by the kernel
__device__ __forceinline__ void bulk_store_hint(void* gdst, const void* ssrc, uint32_t bytes, uint64_t policy) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(s), "r"(bytes), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    return policy;
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// Ampere-style asynchronous 16-byte global -> shared copies (SASS: LDGSTS), used to (re)build a tile from the
// map's static plane without staging through registers
__device__ __forceinline__ void cp_async16(void* sdst, const void* gsrc) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}


// =============================================================================================================
// Sub-warp groups: a warp processes P = 32/Wd worlds at once, Wd = the power of two >= n_agents.  Lane
// (sub, gl) = (lane / Wd, lane % Wd) owns agent `gl` of the warp's world number `sub`.  Values that the
// reference keeps per world (alive / arrived / slot masks, counters) are group-uniform registers holding
// group-relative bit masks, maintained with group ballots; beam masks and the gem mask stay in the world's
// shared-memory record and are updated with shared-memory atomics.  Every phase takes a per-lane predicate
// (`on`: this lane's world takes part) so that worlds in one warp may diverge (errors, resets, extra passes)
// while the warp stays converged for the shuffles.
// =============================================================================================================
struct World {
    uint32_t* rec;      // this lane's world record in shared memory (layout L)
    LleStateLayout L;
    MapDev m;           // this lane's map (group-uniform)
    int A, W, Wd, gl;   // agents, map width, group width, lane within group
    uint32_t gbase, wmask, amask;
    // per lane
    uint32_t pos;
    uint64_t sub_e, sub_p;  // this agent's LaserSubgoal / PBRS "has stood on a laser of source b" flags
    // group-uniform
    uint32_t alive, arrived, slot, n_arrived, n_deads, done;

    __device__ __forceinline__ uint32_t gballot(bool pred) const { return (__ballot_sync(kFull, pred) >> gbase) & wmask; }
    __device__ __forceinline__ uint32_t gshfl(uint32_t v, int src) const { return __shfl_sync(kFull, v, src, Wd); }
    __device__ __forceinline__ uint32_t cell(uint32_t p) const { return (p >> 8) * (uint32_t)W + (p & 0xFFu); }
    __device__ __forceinline__ uint32_t* on_words(int b) const { return rec + L.w_on + b * L.on_words; }
    __device__ __forceinline__ bool on_bit(int b, int k) const { return (on_words(b)[k >> 5] >> (k & 31)) & 1u; }
    __device__ __forceinline__ uint64_t collected() const {
        uint64_t c = 0;
        if (L.gem_words >= 1) c = rec[L.w_gems];
        if (L.gem_words == 2) c |= (uint64_t)rec[L.w_gems + 1] << 32;
        return c;
    }
    // gl == 0 writes; callers synchronise
    __device__ __forceinline__ void set_collected(uint64_t c) {
        if (L.gem_words >= 1) rec[L.w_gems] = (uint32_t)c;
        if (L.gem_words == 2) rec[L.w_gems + 1] = (uint32_t)(c >> 32);
    }

    // World::available_actions cache (world.rs:37, refreshed by compute_available_actions :343-363)
    __device__ __forceinline__ uint32_t cached_avail() const {
        return gl < A ? (uint32_t)reinterpret_cast<const uint8_t*>(rec + L.w_avail)[gl] : 16u;
    }
    __device__ __forceinline__ void store_avail(uint32_t mask) {
        if (gl < A) reinterpret_cast<uint8_t*>(rec + L.w_avail)[gl] = (uint8_t)mask;
    }

    // sources (restricted to `set`) one of whose *listed* laser tiles (env/utils.py:6-11 via World::lasers) covers this
    // agent's cell: `agent_pos in pos_to_reward` of extras_generators.py:95 / reward_strategy.py:171
    __device__ __forceinline__ uint64_t subgoals_here(uint64_t set) const {
        uint64_t mm = 0;
        if (gl < A && set) {
            const LleCellBeams cb = m.cellbeams[cell(pos)];
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const uint32_t e = cb.e[n];
                if (e == LLE_NO_BEAM) break;
                if (be_listed(e)) mm |= 1ull << be_b(e);
            }
        }
        return mm & set;
    }
    // sum over the lanes of this world's group
    __device__ __forceinline__ uint32_t gsum(uint32_t v) const {
        for (int off = Wd >> 1; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off, Wd);
        return v;
    }

    // ---- record <-> registers
    __device__ __forceinline__ void unpack() {
        pos = 0;
        sub_e = sub_p = 0;
        if (L.sub_words && gl < A) {
            if (L.w_subp > L.w_sube) {
                sub_e = rec[L.w_sube + gl * L.sub_words];
                if (L.sub_words == 2) sub_e |= (uint64_t)rec[L.w_sube + gl * 2 + 1] << 32;
            }
            if (L.n_words > L.w_subp) {
                sub_p = rec[L.w_subp + gl * L.sub_words];
                if (L.sub_words == 2) sub_p |= (uint64_t)rec[L.w_subp + gl * 2 + 1] << 32;
            }
        }
        if (gl < A) {
            const uint32_t w = rec[gl >> 1];
            pos = (gl & 1) ? (w >> 16) : (w & 0xFFFFu);
        }
        if (!L.wide_flags) {
            const uint32_t f = rec[L.w_flags];
            alive = f & 0xFFu; arrived = (f >> 8) & 0xFFu; slot = (f >> 16) & 0xFFu;
            n_arrived = (f >> 24) & 0xFu; n_deads = (f >> 28) & 0x7u; done = f >> 31;
        } else {
            alive = rec[L.w_flags]; arrived = rec[L.w_flags + 1]; slot = rec[L.w_flags + 2];
            const uint32_t mm = rec[L.w_flags + 3];
            n_arrived = mm & 0xFFu; n_deads = (mm >> 8) & 0xFFu; done = (mm >> 16) & 1u;
        }
    }
    // writes positions and flags (beam and gem masks are already in place); all lanes must call it
    __device__ __forceinline__ void pack() {
        const uint32_t other = __shfl_down_sync(kFull, pos, 1, Wd);
        if (gl < A && !(gl & 1)) rec[gl >> 1] = pos | ((gl + 1 < A ? other : 0u) << 16);
        if (L.sub_words && gl < A) {
            if (L.w_subp > L.w_sube) {
                rec[L.w_sube + gl * L.sub_words] = (uint32_t)sub_e;
                if (L.sub_words == 2) rec[L.w_sube + gl * 2 + 1] = (uint32_t)(sub_e >> 32);
            }
            if (L.n_words > L.w_subp) {
                rec[L.w_subp + gl * L.sub_words] = (uint32_t)sub_p;
                if (L.sub_words == 2) rec[L.w_subp + gl * 2 + 1] = (uint32_t)(sub_p >> 32);
            }
        }
        if (gl == 0) {
            if (!L.wide_flags) {
                const uint32_t nd = n_deads > 7u ? 7u : n_deads;  // only "> 0" is ever observed (env.py:253-254)
                rec[L.w_flags] = alive | (arrived << 8) | (slot << 16) | (n_arrived << 24) | (nd << 28) | (done << 31);
            } else {
                rec[L.w_flags] = alive; rec[L.w_flags + 1] = arrived; rec[L.w_flags + 2] = slot;
                rec[L.w_flags + 3] = (n_arrived & 0xFFu) | ((n_deads > 255u ? 255u : n_deads) << 8) | (done << 16);
            }
        }
    }

    // ---- tile protocol, lane-parallel ---------------------------------------------------------------------
    // Tile::leave for the alive agents (tile.rs:52-61, laser.rs:199-202 + :157-162 + :50-55): every beam through
    // the agent's cell whose bit there is off is re-armed from that offset on (unless disabled); the slot clears.
    __device__ __forceinline__ void leave_all(bool on) {
        const bool active = on && gl < A && ((alive >> gl) & 1u);
        if (active) {
            const LleCellBeams cb = m.cellbeams[cell(pos)];
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const uint32_t e = cb.e[n];
                if (e == LLE_NO_BEAM) break;  // entries are packed from index 0
                if (be_enabled(e) && !on_bit(be_b(e), be_k(e))) {
                    const uint64_t msk = (~0ull << be_k(e)) & len_mask(be_len(e));
                    uint32_t* w = on_words(be_b(e));
                    if ((uint32_t)msk) atomicOr(w, (uint32_t)msk);
                    if (L.on_words == 2 && (uint32_t)(msk >> 32)) atomicOr(w + 1, (uint32_t)(msk >> 32));
                }
            }
        }
        slot &= ~gballot(active);
        __syncwarp();
    }
    // Tile::pre_enter at `target` (tile.rs:21-27, laser.rs:173-182): an alive agent cuts the enabled beams of its
    // own colour from its offset on.  `alive_flags` are the flags the reference sees at that point.
    __device__ __forceinline__ void pre_enter_all(bool on, uint32_t target, uint32_t alive_flags) {
        if (on && gl < A && ((alive_flags >> gl) & 1u)) {
            const LleCellBeams cb = m.cellbeams[cell(target)];
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const uint32_t e = cb.e[n];
                if (e == LLE_NO_BEAM) break;
                if (be_enabled(e) && be_colour(e) == gl) {
                    const uint64_t msk = (1ull << be_k(e)) - 1ull;
                    uint32_t* w = on_words(be_b(e));
                    atomicAnd(w, (uint32_t)msk);
                    if (L.on_words == 2) atomicAnd(w + 1, (uint32_t)(msk >> 32));
                }
            }
        }
        __syncwarp();
    }
    // Tile::enter at `target` (tile.rs:29-50, laser.rs:184-197, gem.rs:26-35, void.rs:13-22).  An on beam of
    // another colour stops the agent before the wrapped tile (alive -> dies, dead -> nothing; the base tile is
    // NOT entered).  Otherwise the base tile takes the agent.  Returns this lane's event code.
    __device__ __forceinline__ uint32_t enter_all(bool on, uint32_t target) {
        uint32_t code = EV_NONE;
        bool die = false, arrive = false, take_slot = false;
        if (on && gl < A) {
            const uint32_t c = cell(target);
            const LleCellBeams cb = m.cellbeams[c];
            bool lethal = false;
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const uint32_t e = cb.e[n];
                if (e == LLE_NO_BEAM) break;
                if (be_colour(e) != gl && on_bit(be_b(e), be_k(e))) lethal = true;
            }
            const bool is_alive = (alive >> gl) & 1u;
            if (lethal) {
                if (is_alive) { die = true; code = EV_DIED; }
            } else {
                take_slot = true;
                const uint32_t info = m.cellinfo[c];
                const uint32_t kind = info & 7u;
                if (kind == LLE_T_EXIT) {
                    if (!((arrived >> gl) & 1u)) { arrive = true; code = EV_EXIT; }
                } else if (kind == LLE_T_GEM) {
                    const uint32_t g = (info >> 8) & 63u;
                    uint32_t* gw = rec + L.w_gems + (g >> 5);
                    if (!((*gw >> (g & 31u)) & 1u)) {  // no two agents share a cell: no race on this bit
                        atomicOr(gw, 1u << (g & 31u));
                        code = EV_GEM;
                    }
                } else if (kind == LLE_T_VOID) {
                    if (is_alive) { die = true; code = EV_DIED; }
                }
            }
        }
        alive &= ~gballot(die);
        arrived |= gballot(arrive);
        slot |= gballot(take_slot);
        __syncwarp();
        return code;
    }
    // all tiles reset (tile.rs:75-84; laser.rs:168-171: an enabled beam ends fully on, a disabled one stays off)
    __device__ __forceinline__ void tiles_reset(bool on) {
        if (on) {
            for (int b = gl; b < m.NB; b += Wd) {
                const LleBeam bm = m.beams[b];
                const uint64_t v = bm.enabled ? len_mask(bm.len) : 0ull;
                on_words(b)[0] = (uint32_t)v;
                if (L.on_words == 2) on_words(b)[1] = (uint32_t)(v >> 32);
            }
            if (gl == 0) set_collected(0);
            slot = 0;
        }
        __syncwarp();
    }
    // World::reset (world.rs:411-432) with one start per agent (RNG-free, utils/mod.rs:63), then
    // RewardStrategy.reset / LLE.reset bookkeeping (env.py:191-203).
    // sample_different (src/utils/mod.rs:39-86) for maps whose agents have several start candidates (TOML v2 maps).  The
    // reference draws from rand::StdRng (unpinned); the stream here is this library's own contract, restated by the oracle:
    // attempt n = 0..15: agent a draws word (a & 3) of Philox4x32-10(counter = (env id, step, 0x40000000 | n << 8 | a >> 2,
    // reset epoch), key = seed) and starts probing its (row-major sorted) candidates at k = mulhi(word, count); agents are
    // served by increasing number of candidates (stable) and take the first candidate, cyclically from k, that no earlier
    // agent took; an agent without a free candidate fails the attempt.  After 16 failed attempts the assignment computed
    // by the map compiler (a bipartite matching, hdr->start) is used.
    __device__ __forceinline__ void sample_starts(bool on, uint32_t env_lo, uint32_t t32, uint32_t epoch, uint64_t seed) {
        const uint32_t* cidx = reinterpret_cast<const uint32_t*>(m.blob + m.hdr->cand_index_off);
        const uint16_t* cpos = reinterpret_cast<const uint16_t*>(m.blob + m.hdr->cand_pos_off);
        const bool mine = on && gl < A;
        uint32_t first = 0, n = 1;
        if (mine) { first = cidx[2 * gl]; n = cidx[2 * gl + 1]; }
        bool need = on;  // group-uniform
        for (uint32_t attempt = 0; attempt < 16u; ++attempt) {
            if (!__any_sync(kFull, need)) break;
            uint32_t r[4];
            philox4x32_10(env_lo, t32, 0x40000000u | (attempt << 8) | (uint32_t)(gl >> 2), epoch, (uint32_t)seed, (uint32_t)(seed >> 32), r);
            const uint32_t word = (gl & 3) == 0 ? r[0] : (gl & 3) == 1 ? r[1] : (gl & 3) == 2 ? r[2] : r[3];
            const uint32_t k = __umulhi(word, n);
            uint32_t my = 0xFFFFFFFFu;  // this agent's pick, once made
            bool failed = false;         // group-uniform
            for (int i = 0; i < A; ++i) {
                const int a = on ? (int)m.hdr->start_order[i] : 0;
                const uint32_t na = gshfl(n, a);
                uint32_t probe = 0;
                bool settled = !need || failed;  // group-uniform
                while (__any_sync(kFull, !settled)) {
                    uint32_t c = 0xFFFFFFFEu;
                    if (mine && gl == a) c = cpos[first + (k + probe) % n];
                    c = gshfl(c, a);
                    const bool clash = gballot(my == c) != 0;
                    if (!settled) {
                        if (!clash) {
                            if (gl == a) my = c;
                            settled = true;
                        } else if (++probe >= na) {
                            failed = true;
                            settled = true;
                        }
                    }
                }
            }
            if (need && !failed) {
                if (mine) pos = my;
                need = false;
            }
        }
    }
    // `sample`: compile-time switch of the start sampler — batches with random starts run on the general kernel, so the
    // fast kernel does not carry the sampler's code
    __device__ __forceinline__ void reset(bool on, uint64_t pbrs_set, uint32_t env_lo = 0, uint32_t t32 = 0, uint32_t epoch = 0,
                                          uint64_t seed = 0, bool sample = false) {
        tiles_reset(on);
        if (on) {
            alive = amask; arrived = 0; n_arrived = 0; n_deads = 0; done = 0;
            pos = gl < A ? (uint32_t)m.hdr->start[gl] : 0u;
        }
        if (sample && __any_sync(kFull, on && m.hdr->random_starts)) sample_starts(on && m.hdr->random_starts, env_lo, t32, epoch, seed);
        pre_enter_all(on, pos, alive);
        (void)enter_all(on, pos);  // events are dropped (world.rs:428-430)
        if (on) {
            sub_e = 0;                        // extras_generator.reset() (env.py:196); marked again when observed
            sub_p = subgoals_here(pbrs_set);  // PotentialShapedLLE.reset (reward_strategy.py:176-180): clear, then compute_potential()
        }
    }
    // World::compute_available_actions (world.rs:343-363) as a 5-bit mask indexed by Action value.
    __device__ __forceinline__ uint32_t available() const {
        const bool active = gl < A && ((alive >> gl) & 1u) && !((arrived >> gl) & 1u);
        uint32_t nbr = 0;
        if (active) nbr = (m.cellinfo[cell(pos)] >> 3) & 15u;
        for (int o = 0; o < A; ++o) {
            const uint32_t op = gshfl(pos, o);
            if (((slot >> o) & 1u) && o != gl) {  // Tile::is_occupied (tile.rs:97-99)
                const int d = (int)op - (int)pos;
                if (d == -256) nbr &= ~1u;
                else if (d == 256) nbr &= ~2u;
                else if (d == 1) nbr &= ~4u;
                else if (d == -1) nbr &= ~8u;
            }
        }
        return 16u | nbr;  // Stay is always listed
    }
    // LLE.available_actions with walkable_lasers == False (env.py:153-163): drop every listed action (STAY
    // included) whose target holds an on, listed (world.rs:159-172) laser of another colour.
    __device__ __forceinline__ uint32_t available_no_walk(uint32_t mask) const {
        uint32_t out = 0;
        if (gl < A) {
#pragma unroll
            for (int act = 0; act < 5; ++act) {
                if (!((mask >> act) & 1u)) continue;
                const LleCellBeams cb = m.cellbeams[cell(pos + act_delta(act))];
                bool blocked = false;
#pragma unroll
                for (int n = 0; n < 4; ++n) {
                    const uint32_t e = cb.e[n];
                    if (e != LLE_NO_BEAM && be_listed(e) && be_colour(e) != gl && on_bit(be_b(e), be_k(e))) blocked = true;
                }
                if (!blocked) out |= 1u << act;
            }
        }
        return out;
    }
    // World::step after validation (world.rs:454-472) for the worlds with `on`.  Returns this lane's event byte;
    // the counts are group-uniform.
    __device__ __forceinline__ uint32_t step(bool on, uint32_t act, uint32_t& n_gem, uint32_t& n_exit, uint32_t& n_died) {
        uint32_t np = (on && gl < A) ? pos + act_delta(act) : 0xFFFF0000u + gl;  // inactive lanes never collide
        // vertex conflicts (world.rs:365-378 + utils/mod.rs:18-36): every agent whose target is shared goes back
        for (;;) {
            bool dup = false;
            for (int o = 0; o < A; ++o) {
                const uint32_t other = gshfl(np, o);
                if (o != gl && other == np) dup = true;
            }
            dup = dup && on && gl < A;
            if (!__any_sync(kFull, dup)) break;
            if (dup) np = pos;
        }
        uint32_t ev = 0;
        n_gem = n_exit = n_died = 0;
        bool again = on;  // move_agents (world.rs:477-505), repeated while an agent of this world died (:468-472)
        for (uint32_t pass = 1;; ++pass) {
            leave_all(again);
            pre_enter_all(again, np, alive);
            const uint32_t code = enter_all(again, np);
            if (pass == 1) {
                ev = code;
                if (on && gl < A) pos = np;
            } else if (code != EV_NONE) {
                ev |= (pass > 63u ? 63u : pass) << 2;  // passes >= 2 can only emit deaths (SURVEY App. A)
            }
            const uint32_t died = gballot(code == EV_DIED);
            n_died += __popc(died);
            n_gem += __popc(gballot(code == EV_GEM));
            n_exit += __popc(gballot(code == EV_EXIT));
            again = again && died != 0;
            if (!__any_sync(kFull, again)) break;
        }
        return ev;
    }
    // SingleObjective / MultiObjective.compute_reward (reward_strategy.py:58-75, :90-109) and LLE.compute_done
    // (env.py:253-254): updates the counters (if `on`); component r of the reward.
    __device__ __forceinline__ void account(bool on, uint32_t n_exit, uint32_t n_died) {
        if (on) {
            n_arrived += n_exit;
            n_deads += n_died;
            done = (n_arrived == (uint32_t)A || n_deads > 0) ? 1u : 0u;
        }
    }
    __device__ __forceinline__ float reward_component(int r, int R, uint32_t n_gem, uint32_t n_exit, uint32_t n_died) const {
        const bool all_in = n_arrived == (uint32_t)A;
        if (R == 1) return (float)n_gem + (float)n_exit - (float)n_died + (all_in ? 1.0f : 0.0f);  // death override is dead code (:71-72)
        switch (r) {
            case 0: return n_died ? 0.0f : (float)n_gem;
            case 1: return n_died ? 0.0f : (float)n_exit;
            case 2: return -(float)n_died;
            default: return (!n_died && all_in) ? 1.0f : 0.0f;
        }
    }
    // Body of World::set_state after the argument checks (world.rs:541-594) for the worlds with `on`.  `target`
    // per lane; sg / sa requested gem and alive masks.  Returns ERR_OK, ERR_STATE_NOT_WALKABLE (nothing entered)
    // or ERR_STATE_MISMATCH per world (group-uniform).
    __device__ __forceinline__ uint32_t set_state_apply(bool on, uint32_t target, uint64_t sg, uint32_t sa, uint32_t& code,
                                                        uint32_t& n_gem, uint32_t& n_exit, uint32_t& n_died) {
        code = EV_NONE;
        n_gem = n_exit = n_died = 0;
        tiles_reset(on);
        if (on && gl == 0) set_collected(sg & m.gem_toplevel);  // only top-level Gem tiles can be force-collected (:550-554)
        const bool wall = on && gl < A && (m.cellinfo[cell(target)] & 7u) == LLE_T_WALL;
        const bool blocked = gballot(wall) != 0;  // :556-568
        const bool go = on && !blocked;
        __syncwarp();
        pre_enter_all(go, target, alive);  // with the agents' *current* alive flags (:555)
        if (go) {
            if (gl < A) pos = target;  // :571
            alive = amask;             // agent.reset() (:578)
            arrived = 0;
        }
        code = enter_all(go, pos);
        if (go) alive &= sa;  // forced death, no event (:583-585)
        n_died = __popc(gballot(code == EV_DIED));
        n_gem = __popc(gballot(code == EV_GEM));
        n_exit = __popc(gballot(code == EV_EXIT));
        if (!on) return ERR_OK;
        if (blocked) return ERR_STATE_NOT_WALKABLE;
        if (collected() != sg || alive != (sa & amask)) return ERR_STATE_MISMATCH;  // :588-594
        return ERR_OK;
    }
};

// ---- observation tile: descriptor bits read straight from a record ------------------------------------------
__device__ __forceinline__ bool rec_lit(const uint32_t* rec, const LleStateLayout& L, const LlePatch& pe) {
    if (pe.src == 0xFF)  // gem: lit while NOT collected (observations.py:260-263)
        return !((rec[L.w_gems + (pe.bit >> 5)] >> (pe.bit & 31)) & 1u);
    return (rec[L.w_on + pe.src * L.on_words + (pe.bit >> 5)] >> (pe.bit & 31)) & 1u;  // laser: lit while on (:256-259)
}
__device__ __forceinline__ uint32_t rec_pos(const uint32_t* rec, int a) {
    const uint32_t w = rec[a >> 1];
    return (a & 1) ? (w >> 16) : (w & 0xFFFFu);
}

// Per-lane register copy of the first 64 patch entries of the map being rendered (entries lane and lane + 32):
// the element index, the static value to restore (as the tile's element type OT), and where in a record the controlling bit lives.
template <typename OT>
struct PatchCache {
    uint32_t idx0, idx1;
    OT stat0, stat1;
    uint16_t word0, word1;  // record word holding the bit
    uint8_t bit0, bit1, gem0, gem1;
    bool valid0, valid1;
    __device__ __forceinline__ void load(const MapDev& rm, const LleStateLayout& L, int lane) {
        valid0 = lane < rm.n_patch;
        valid1 = lane + 32 < rm.n_patch;
        idx0 = idx1 = 0; stat0 = stat1 = (OT)0; word0 = word1 = 0; bit0 = bit1 = gem0 = gem1 = 0;
        if (valid0) {
            const LlePatch pe = rm.patches[lane];
            idx0 = pe.idx; stat0 = (OT)pe.stat; gem0 = pe.src == 0xFF; bit0 = pe.bit & 31;
            word0 = (uint16_t)(gem0 ? L.w_gems + (pe.bit >> 5) : L.w_on + pe.src * L.on_words + (pe.bit >> 5));
        }
        if (valid1) {
            const LlePatch pe = rm.patches[lane + 32];
            idx1 = pe.idx; stat1 = (OT)pe.stat; gem1 = pe.src == 0xFF; bit1 = pe.bit & 31;
            word1 = (uint16_t)(gem1 ? L.w_gems + (pe.bit >> 5) : L.w_on + pe.src * L.on_words + (pe.bit >> 5));
        }
    }
    // a laser cell is lit while its beam bit is on, a gem while it is NOT collected (observations.py:256-263)
    __device__ __forceinline__ bool lit0(const uint32_t* rec) const { return (((rec[word0] >> bit0) & 1u) ^ gem0) != 0; }
    __device__ __forceinline__ bool lit1(const uint32_t* rec) const { return (((rec[word1] >> bit1) & 1u) ^ gem1) != 0; }
};

// (Re)build elements [lo, hi) of one world's block from the map's static plane (observations.py:216-237) with
// asynchronous copies; pad elements beyond C*H*W are zero.  Completion: cp_async_wait_all() + __syncwarp().
// int8: the plane is zero-padded to the row stride and lo, hi are multiples of 16, so every piece is one 16-byte copy.
template <typename OT>
__device__ __forceinline__ void tile_rebuild_async(OT* sub_tile, const MapDev& rm, int lo, int hi, int lane) {
    const int nf = hi - lo;
    if constexpr (sizeof(OT) == 1) {
        const int8_t* stat = reinterpret_cast<const int8_t*>(rm.stat);
        for (int f = lane * 16; f < nf; f += 512) cp_async16(sub_tile + f, stat + lo + f);
    } else {
        for (int f = lane * 4; f < nf; f += 128) {
            const int gi = lo + f;
            if (gi + 3 < rm.obs_floats) {
                cp_async16(sub_tile + f, rm.stat + gi);
            } else {
                float4 v;
                v.x = gi + 0 < rm.obs_floats ? __ldg(rm.stat + gi + 0) : 0.f;
                v.y = gi + 1 < rm.obs_floats ? __ldg(rm.stat + gi + 1) : 0.f;
                v.z = gi + 2 < rm.obs_floats ? __ldg(rm.stat + gi + 2) : 0.f;
                v.w = gi + 3 < rm.obs_floats ? __ldg(rm.stat + gi + 3) : 0.f;
                *reinterpret_cast<float4*>(sub_tile + f) = v;
            }
        }
    }
}

// Dataflow ordering between steps.  A ticket's step q may start once the ticket's step q-1 is complete, whichever
// launch (programmatic dependent launches overlap) or warp ran it.  Completion is published with a gpu-scope release
// after every write of the ticket (records, outputs, and the observation bulk stores, which must have completed),
// and consumed with an acquire before the records are read (through L2).
__device__ __forceinline__ void ticket_release(uint32_t* flag, uint32_t seq) {
    asm volatile("fence.proxy.async;" ::: "memory");  // completed async-proxy (bulk) writes before the generic-proxy release
    // st.release orders every earlier write of this thread, and (cumulatively) of the lanes it synchronised with, before the flag
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(seq) : "memory");
}
__device__ __forceinline__ bool sys_flag_ready(const uint32_t* flag, uint32_t need) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    return (int32_t)(v - need) >= 0;
}
__device__ __forceinline__ bool ticket_ready(const uint32_t* flag, uint32_t need) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    return (int32_t)(v - need) >= 0;
}
// lle_vec_parts_*: count a completed ticket of its part; the last one publishes the part to the host.  A warp's stores to host
// memory (reward2 / done2) are ordered before its count by a gpu-scope release (they have left the SM; posted PCIe writes keep
// their order), the last warp acquires the counts, fences at system scope and writes the part's completion word.  The counter
// is cleared for the next step, whose tickets of this part cannot complete before the host has seen this word and fed the part
// again.  Out of line: only the parts loop gets here.
__device__ __noinline__ void part_ticket_done(uint32_t* part_count, uint32_t* part_out, uint32_t part_tickets, uint32_t part_last, uint32_t n_tickets,
                                              uint32_t ticket, uint32_t value) {
    const uint32_t part = min(ticket / part_tickets, part_last);
    const uint32_t n = part == part_last ? n_tickets - part_last * part_tickets : part_tickets;
    uint32_t before;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(before) : "l"(part_count + part) : "memory");
    if (before == n - 1u) {
        part_count[part] = 0;
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(part_out + part * 32), "r"(value) : "memory");
    }
}
template <bool PARTS>
__device__ __forceinline__ void ticket_done(const KParams& p, uint32_t ticket, uint32_t seq) {
    ticket_release(p.flags + ticket, seq);
    if constexpr (PARTS) part_ticket_done(p.part_count, p.part_out, p.part_tickets, p.part_last, p.n_tickets, ticket, p.out_value);
}
// The tickets of a part wait for the host's actions (lle_vec_parts_feed).  `fed_upto` (lane 0's register): tickets below it are
// known to be fed - a warp takes tickets in increasing order, so it looks at a part's word once.  Always true outside that mode.
template <bool PARTS>
__device__ __forceinline__ bool part_fed(const KParams& p, uint32_t ticket, uint32_t& fed_upto) {
    if (!PARTS || ticket < fed_upto) return true;
    const uint32_t part = min(ticket / p.part_tickets, p.part_last);
    // gpu scope: the word and the staged actions are written into device memory (L2) by the copy / front-end engines; a
    // system-scope acquire or fence here costs microseconds per use (measured: 97 -> 127 us per step with one fence.sys per part)
    if (!ticket_ready(p.part_in + part * 32, p.in_need)) return false;
    fed_upto = part == p.part_last ? p.n_tickets : (part + 1u) * p.part_tickets;
    return true;
}
// a host-supplied action; in a parts loop the staging buffer is rewritten by the copy engine while kernels run: through L2 only
template <bool PARTS>
__device__ __forceinline__ uint32_t load_action(const KParams& p, int64_t index) {
    return (uint32_t)(uint8_t)(PARTS ? __ldcv(p.actions_in + index) : p.actions_in[index]);
}
__device__ __forceinline__ bool sched_slot_armed(const uint32_t* gen, uint32_t want) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(gen) : "memory");
    return v == want;
}
// What a launch waits for before it takes its first pair.  Host-supplied actions still in flight on the copy stream (independent
// of this stream: no cycle).  And its scheduler slot: slots rotate over the launches, and programmatic dependent launch lets many
// small launches be resident at once, so the launch that used this slot kSchedSlots launches ago may still be running: wait until
// its last warp has re-armed the slot (it never waits for us, and all of its CTAs are resident by the time this launch may start:
// no cycle).
__device__ __forceinline__ void launch_wait(const KParams& p, int lane) {
    if (p.in_flag) {
        if (lane == 0)
            while (!sys_flag_ready(p.in_flag, p.in_need)) __nanosleep(100);
        __syncwarp();
    }
    if (p.sched_check) {
        if (lane == 0)
            while (!sched_slot_armed(p.sched + 2, p.sched_gen)) __nanosleep(32);
        __syncwarp();
    }
}
// Lane 0: the warp's next (step, ticket) pair (`first`: its first one).  On an idle device (the host saw every earlier launch
// retire: a closed loop) all CTAs are resident at once and a warp's first pair is its own index - no round trip to the launch's
// counter before it can start.  Not when launches overlap: CTAs then trickle in as their predecessors retire, and a pair pinned to
// a late CTA would hold up everything behind it.
__device__ __forceinline__ uint32_t take_pair(const KParams& p, bool first, uint32_t warp_global) {
    if (p.sched_check == 0) return first ? warp_global : p.n_warps_total + atomicAdd(&p.sched[0], 1u);  // behind the static pairs
    return atomicAdd(&p.sched[0], 1u);
}
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// LLE.reset with randomize_lasers (env.py:198-200): after world.reset() every source gets a random colour.  The reference
// draws random.randint(0, n_agents - 1) from Python's global generator (unpinned); the stream here is this library's
// contract: source b takes word (b & 3) of Philox4x32-10(counter = (env id, step, 0x20000000 | b >> 2, explicit-reset
// count), key = seed) and colour = mulhi(word, n_agents).  The colouring selects one of the map's precompiled variants
// (index = map * n_variants + sum colour_b * n_agents^b), recorded in map_of_env.  Out of line: resets are rare and the
// step kernel should not carry this in its registers.
__device__ __noinline__ int recolour_variant(int32_t* map_of_env, uint64_t env_id_base, uint64_t seed, uint32_t reset_epoch, int n_agents,
                                             int n_variants, int64_t env, uint64_t t_now, int n_sources, int map_id) {
    const int base = map_id / n_variants;
    int variant = 0, scale = 1;
    uint32_t r[4] = {0, 0, 0, 0};
    for (int b = 0; b < n_sources; ++b) {
        if ((b & 3) == 0)
            philox4x32_10((uint32_t)(env_id_base + (uint64_t)env), (uint32_t)t_now, 0x20000000u | (uint32_t)(b >> 2), reset_epoch,
                          (uint32_t)seed, (uint32_t)(seed >> 32), r);
        const uint32_t word = (b & 3) == 0 ? r[0] : (b & 3) == 1 ? r[1] : (b & 3) == 2 ? r[2] : r[3];
        variant += (int)__umulhi(word, (uint32_t)n_agents) * scale;
        scale *= n_agents;
    }
    const int next = base * n_variants + variant;
    __stcg(map_of_env + env, next);
    return next;
}

// Episode statistics of one reward component / of the episode length (lle_vec_options.episode_stats).  Out of line: the step
// kernel should not carry this in its registers when the option is off.
__device__ __noinline__ void episode_stat_reward(float* running, float* last, float v, bool paid, bool done, bool cleared) {
    float acc = cleared ? 0.0f : *running;
    if (paid) {
        acc = __fadd_rn(acc, v);
        if (done) { *last = acc; acc = 0.0f; }
    }
    *running = acc;
}
__device__ __noinline__ void episode_stat_length(int32_t* running, int32_t* last, bool paid, bool done, bool cleared) {
    int32_t len = cleared ? 0 : *running;
    if (paid) {
        ++len;
        if (done) { *last = len; len = 0; }
    }
    *running = len;
}

// End of a launch, lane 0 of every warp: count the warp out; the last warp re-arms the launch's scheduler slot for a later
// launch (generation word, see sched_slot_armed) and publishes the launch to the host.  With host-facing stepping
// (lle_vec_pipeline_submit) reward / done went straight into pinned host memory: every warp fences them at system scope before
// it is counted, and the last one writes the step number into the slot's completion word, which the host polls.
__device__ __forceinline__ void launch_epilogue(const KParams& p, bool is_step) {
    if (p.out_flag) __threadfence_system();
    else __threadfence();
    const uint32_t finished = atomicAdd(&p.sched[1], 1u);
    if (finished == p.n_warps_total - 1) {
        p.sched[0] = 0;
        p.sched[1] = 0;
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.sched + 2), "r"(p.sched_gen + 1u) : "memory");
        if (is_step && p.retired_seq) *p.retired_seq = p.seq + (uint32_t)p.n_steps - 1u;
        if (p.retired_launch) *p.retired_launch = atomicAdd(p.retired_count, 1u) + 1u;  // a lower bound of the launches that have retired
        if (p.out_flag) {
            __threadfence_system();
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.out_flag), "r"(p.out_value) : "memory");
        }
    }
}

#ifndef LLE_MIN_CTAS
#define LLE_MIN_CTAS 5
#endif
// MODE: MODE_STEP / MODE_RESET / MODE_SET_STATE, compiled separately so the step kernel carries no set_state code.
// FAST: the common shape — one map for the whole batch, one whole world per tile, a single tile buffer, at most 64
// patch entries and a record of at most 32 words.  The tile then never changes map or chunk, so the tag / freshness
// bookkeeping of the general path disappears and the per-tile work is a handful of shared-memory accesses.
// KIND: 0 general, 1 FAST (above), 2 general with the feature-driven renderer of partial observations (sparse maps).
// PARTS: the step kernel of a parts loop (lle_vec_parts_*): tickets wait for their part's actions and completed parts are
// published to the host.  A separate instantiation: the plain step kernel carries none of it.
// OT: the observation's element type, float or int8_t (lle_vec_options.obs_dtype).  An int8 vec renders the same tiles in bytes:
// the static plane, patch values and one-hots are byte stores and every bulk store moves a quarter of the bytes.  Partial
// observations are float only.
template <int MODE, int KIND, bool PARTS = false, typename OT = float>
__global__ void __launch_bounds__(kThreads, LLE_MIN_CTAS) lle_world_kernel(const KParams p) {
    constexpr bool FAST = KIND == 1;
    constexpr bool BY_FEATURE = KIND == 2;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LleStateLayout L = p.L;
    const int A = p.A, stride = L.stride;
    uint8_t* wbase = smem_raw + (size_t)warp * p.warp_smem_bytes;
    OT* tiles = reinterpret_cast<OT*>(wbase);                                                // [n_buf][tile_floats]
    uint32_t* recs = reinterpret_cast<uint32_t*>(tiles + (size_t)p.n_buf * p.tile_floats);   // [group][stride]
    uint32_t* applied = recs + (size_t)p.group * stride;                                     // [n_buf][E][stride]
    int32_t* tags = reinterpret_cast<int32_t*>(applied + (size_t)p.n_buf * p.E * stride);    // [n_buf][E] map id, [n_buf] chunk
    int32_t* map_ids = tags + p.n_buf * p.E + p.n_buf;                                       // [group]
    int32_t* fresh = map_ids + p.group;  // [n_buf][E]: 1 = just rebuilt from the static plane (copies may be in flight)
    for (int k = lane; k < p.n_buf * p.E + p.n_buf; k += 32) tags[k] = -1;
    for (int k = lane; k < p.n_buf * p.E; k += 32) fresh[k] = 0;
    __syncwarp();

    const int Wd = p.Wd, P = 32 / Wd;
    World w;
    w.L = L;
    w.A = A;
    w.W = p.W;
    w.Wd = Wd;
    w.gl = lane & (Wd - 1);
    w.gbase = (uint32_t)(lane & ~(Wd - 1));
    w.wmask = Wd >= 32 ? ~0u : ((1u << Wd) - 1u);
    w.amask = A >= 32 ? ~0u : ((1u << A) - 1u);
    const int sub = lane / Wd, gl = w.gl;
    int bound_map = -1;       // map bound to this lane's World
    MapDev rm;                // map bound for rendering (warp-uniform)
    PatchCache<OT> pc;
    int render_map = -1;
    int buf = 0;
    bool tile_fresh = true;  // FAST: the tile was just (pre)built from the static plane
    // Programmatic dependent launch: let the next launch on the stream begin its prologue as soon as SM resources
    // free up; everything above and the static-plane prefetch below touch nothing the previous launch writes.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    uint32_t fresh_bits = 0;  // FAST: sub-tiles that hold a pristine static plane (nothing to un-patch yet)
    if constexpr (FAST) {
        if (p.map_of_env == nullptr) {  // one map for the whole batch: bind it once and prefetch its static plane
            if (p.has_map0) w.m = p.map0;
            else w.m.bind(p.blobs[0]);
            bound_map = 0;
            rm = w.m;
            render_map = 0;
            pc.load(rm, L, lane);
            for (int s = 0; s < p.E; ++s)  // lands while the first logic pass runs
                tile_rebuild_async(tiles + (size_t)s * p.obs_stride, rm, 0, (int)p.obs_stride, lane);
            asm volatile("cp.async.commit_group;" ::: "memory");
            for (int k = lane; k < p.E; k += 32) tags[k] = 0;
            fresh_bits = ~0u;
            __syncwarp();
        } else {
            tile_fresh = false;
        }
    }
    // Reset / set_state wait for the whole previous launch.  A step does not: it orders itself ticket by ticket with
    // the epoch flags, so its first tickets start while the previous step's last ones are still draining.
    if constexpr (MODE != MODE_STEP) asm volatile("griddepcontrol.wait;" ::: "memory");
    launch_wait(p, lane);
    const uint32_t warp_global = blockIdx.x * kWarps + warp;
    const uint32_t n_pairs = p.n_tickets * (uint32_t)p.n_steps;  // (step, ticket) pairs, handed out in order (the host keeps it < 2^31)
    uint64_t t_first = 0, t_last = 0;
    if (p.timeline && lane == 0) p.timeline[warp_global * 4] = globaltimer_ns();
    int step_index = 0;
    bool first = true;
    uint32_t owed_ticket = 0, owed_seq = 0;  // the previous ticket, whose completion is published once its stores are done
    bool owed = false;
    const bool single_step = p.n_steps == 1;
    bool first_pair = true;
    uint32_t fed_upto = 0;  // lle_vec_parts_*: tickets below this are known to have their actions
    for (;;) {
        uint32_t pair = 0;
        if (lane == 0) pair = take_pair(p, first_pair, warp_global);
        pair = __shfl_sync(kFull, pair, 0);
        first_pair = false;
        if (pair >= n_pairs) break;
        const uint32_t ticket = single_step ? pair : pair % p.n_tickets;
        step_index = single_step ? 0 : (int)(pair / p.n_tickets);
        const uint32_t my_seq = p.seq + (uint32_t)step_index;
        if constexpr (MODE == MODE_STEP) {
            bool flushed = false;
            if (lane == 0 && (!ticket_ready(p.flags + ticket, my_seq - 1u) || !part_fed<PARTS>(p, ticket, fed_upto))) {
                // Never block while owing a completion: the warp we are about to wait for may be waiting for ours (and the host
                // waits for whole parts before it feeds the next actions).
                if (owed) {
                    bulk_wait_all();
                    ticket_done<PARTS>(p, owed_ticket, owed_seq);
                    flushed = true;
                }
                while (!ticket_ready(p.flags + ticket, my_seq - 1u)) __nanosleep(64);
                while (!part_fed<PARTS>(p, ticket, fed_upto)) __nanosleep(200);
            }
            if (__shfl_sync(kFull, (int)flushed, 0)) owed = false;
        }
        const int64_t env0 = (int64_t)ticket * p.group;
        const uint64_t t_now = p.t + (uint64_t)step_index;
        {   // the ticket's records (contiguous, group x stride words) start moving into shared memory now, through L2 only
            // (rollout mode re-reads its own writes); the first pass below waits for them, later passes find them there
            const uint32_t* gsrc = p.records + env0 * stride;
            for (int k = lane * 4; k < p.group * stride; k += 128) cp_async16(recs + k, gsrc + k);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        if (!FAST && first && p.write_obs && p.n_chunks == 1 && p.obs_kind != LLE_OBS_PARTIAL) {
            // start filling this warp's tiles from the static plane of the first world's map now: the copies land
            // while the first logic pass runs
            first = false;
            const int mid = p.map_of_env ? __ldcg(p.map_of_env + env0) : 0;
            rm.bind(p.blobs[mid]);
            render_map = mid;
            pc.load(rm, L, lane);
            for (int b = 0; b < p.n_buf; ++b)
                for (int s = 0; s < p.E; ++s) {
                    tile_rebuild_async(tiles + (size_t)b * p.tile_floats + (size_t)s * p.obs_stride, rm, 0, (int)p.obs_stride, lane);
                    if (!FAST && lane == 0) { tags[b * p.E + s] = mid; fresh[b * p.E + s] = 1; }
                }
            if (lane == 0)
                for (int b = 0; b < p.n_buf; ++b) tags[p.n_buf * p.E + b] = 0;
            asm volatile("cp.async.commit_group;" ::: "memory");
        }

        // ================================================================== logic: P worlds at a time
        for (int g0 = 0; g0 < p.group; g0 += P) {
            const int g = g0 + sub;
            const int64_t env = env0 + g;  // N_pad is a multiple of the group size: always a world
            int map_id = 0;
            if (!FAST || p.map_of_env != nullptr) {
                map_id = p.map_of_env ? __ldcg(p.map_of_env + env) : 0;  // through L2: a reset of the previous (overlapped) step may have rewritten it
                if (map_id != bound_map) {
                    if (map_id == 0 && p.has_map0) w.m = p.map0;
                    else w.m.bind(p.blobs[map_id]);
                    bound_map = map_id;
                }
                if (gl == 0) map_ids[g] = map_id;
            }
            // LLE.reset with randomize_lasers (env.py:198-200): the worlds with `on` take a new colouring (recolour_variant,
            // above); the reset that precedes it ran with the previous colours, like the reference
            auto recolour = [&](bool on) {
                if constexpr (FAST) return;  // randomize_lasers runs on the general kernel (the host selects it): no cost here
                int next = map_id;
                if (on && gl == 0)
                    next = recolour_variant(p.map_of_env, p.env_id_base, p.seed, p.reset_epoch, A, p.n_variants, env, t_now, w.m.NB, map_id);
                map_id = __shfl_sync(kFull, next, (int)(lane & ~(Wd - 1)));
                if (on && map_id != bound_map) {
                    w.m.bind(p.blobs[map_id]);
                    bound_map = map_id;
                }
                if (on && gl == 0) map_ids[g] = map_id;
                __syncwarp();
            };
            uint32_t* rec = recs + (size_t)g * stride;
            if (g0 == 0) {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
            }
            w.rec = rec;
            w.unpack();

            uint32_t ev = 0, act = 4, err = ERR_OK, n_gem = 0, n_exit = 0, n_died = 0;
            double shaped = 0.0;
            bool touch = true;  // whether reward/done/events/err/actions are (re)written
            bool paid = false;  // whether a reward is due (a transition happened)
            const bool real = env < p.N;

            if constexpr (MODE == MODE_STEP) {
                const uint32_t av = w.cached_avail();
                if (p.actions_in) {
                    if (real && gl < A) act = load_action<PARTS>(p, env * A + gl);  // padding worlds just STAY
                } else {
                    uint32_t r[4];
                    philox4x32_10((uint32_t)(p.env_id_base + (uint64_t)env), (uint32_t)t_now, (uint32_t)(gl >> 2), (uint32_t)(t_now >> 32),
                                  (uint32_t)p.seed, (uint32_t)(p.seed >> 32), r);
                    const uint32_t word = (gl & 3) == 0 ? r[0] : (gl & 3) == 1 ? r[1] : (gl & 3) == 2 ? r[2] : r[3];
                    act = pick_action(word, av);
                }
                const bool bad = w.gballot(gl < A && (act > 4u || !((av >> act) & 1u))) != 0;
                if (p.lle_semantics && w.done) err = ERR_DONE;
                else if (bad) err = ERR_INVALID_ACTION;  // the world is left untouched (world.rs:444-453)
                paid = err == ERR_OK;
                ev = w.step(paid, act, n_gem, n_exit, n_died);
                w.account(paid, n_exit, n_died);
                if (p.pbrs_on) {  // PotentialShapedLLE.compute_reward (reward_strategy.py:145-158), python-float arithmetic
                    const uint32_t before = w.gsum((uint32_t)__popcll(w.sub_p));
                    if (paid) w.sub_p |= w.subgoals_here(p.pbrs_set);
                    const uint32_t after = w.gsum((uint32_t)__popcll(w.sub_p));
                    const uint32_t size = (uint32_t)A * (uint32_t)__popcll(p.pbrs_set & len_mask(w.m.NB));
                    const double prev = __dmul_rn((double)(size - before), p.pbrs_value);
                    const double curr = __dmul_rn((double)(size - after), p.pbrs_value);
                    shaped = __dsub_rn(__dmul_rn(p.pbrs_gamma, prev), curr);  // no fused multiply-add, like CPython
                }
            } else if constexpr (MODE == MODE_RESET) {
                const bool on = !p.refresh_only && (!p.reset_mask || !real || p.reset_mask[env]);
                w.reset(on, p.pbrs_set, (uint32_t)(p.env_id_base + (uint64_t)env), (uint32_t)t_now, p.reset_epoch, p.seed, !FAST);
                touch = on;
                if constexpr (!FAST)
                    if (p.randomize && __any_sync(kFull, on)) recolour(on);
            } else {  // MODE_SET_STATE: World::set_state (world.rs:515-597) + LLE.set_state (env.py:208-216)
                touch = real;  // padding worlds: nothing to force
                int si = 0, sj = 0;
                bool want_alive = false;
                if (real && gl < A) {
                    si = p.ss_pos[(env * A + gl) * 2];
                    sj = p.ss_pos[(env * A + gl) * 2 + 1];
                    want_alive = p.ss_alive[env * A + gl] != 0;
                }
                const uint32_t sa = w.gballot(want_alive) & w.amask;
                uint64_t sg = 0;
                for (int b0 = 0; b0 < p.G; b0 += Wd) {
                    const bool bit = real && b0 + gl < p.G && p.ss_gems[env * p.G + b0 + gl] != 0;
                    sg |= (uint64_t)w.gballot(bit) << b0;
                }
                if (real && p.lle_semantics) {  // reward_strategy.reset() precedes world.set_state (env.py:213)
                    w.n_arrived = 0;
                    w.n_deads = 0;
                    if (p.pbrs_on) w.sub_p = w.subgoals_here(p.pbrs_set);  // ... with the positions the world still has
                }
                bool dup = false;
                for (int o = 0; o < A; ++o) {
                    const int oi = (int)w.gshfl((uint32_t)si, o), oj = (int)w.gshfl((uint32_t)sj, o);
                    if (o != gl && oi == si && oj == sj) dup = true;
                }
                const bool any_dup = w.gballot(dup && gl < A) != 0;
                const bool any_oob = w.gballot(gl < A && (si < 0 || sj < 0 || si >= p.H || sj >= p.W)) != 0;
                if (real) {
                    if (any_dup) err = ERR_STATE_DUPLICATE;          // :529-534
                    else if (any_oob) err = ERR_STATE_OUT_OF_WORLD;  // :536-540
                }
                const bool go = real && err == ERR_OK;
                const uint32_t cur_pos = w.pos;  // current_state = self.get_state() (:541)
                const uint64_t cur_g = w.collected();
                const uint32_t cur_a = w.alive;
                const uint32_t target = go ? (((uint32_t)si << 8) | (uint32_t)sj) : w.pos;
                const uint32_t r1 = w.set_state_apply(go, target, sg, sa, ev, n_gem, n_exit, n_died);
                if (go) err = r1;
                // self.set_state(&current_state).unwrap() (:563): the previous state is re-derived, events dropped
                const bool restore = go && r1 == ERR_STATE_NOT_WALKABLE;
                if (__any_sync(kFull, restore)) {
                    uint32_t e2, a2, b2, c2;
                    (void)w.set_state_apply(restore, cur_pos, cur_g, cur_a, e2, a2, b2, c2);
                }
                if (restore) ev = 0;
                // compute_reward(events); done = compute_done() (env.py:215-216)
                w.account(go && err == ERR_OK && p.lle_semantics, n_exit, n_died);
                if (p.pbrs_on && go && err == ERR_OK && p.lle_semantics) w.sub_p |= w.subgoals_here(p.pbrs_set);  // compute_potential()
            }

            if (touch) {
                for (int r = gl; r < p.R; r += Wd) {
                    float v = 0.0f;
                    if (paid) {
                        if (p.R == 1) v = __fadd_rn(w.reward_component(0, 1, n_gem, n_exit, n_died), (float)shaped);  // np.float32 += python float
                        else if (r < 4) v = w.reward_component(r, 4, n_gem, n_exit, n_died);
                        else v = (float)shaped;  // fifth component of MultiObjective + PBRS (np.concat, :153)
                    }
                    p.reward[env * p.R + r] = v;
                    if (p.reward2 && real) p.reward2[env * p.R + r] = v;  // the host's own buffer: N worlds, no padding
                    if (p.ep_return) episode_stat_reward(p.ep_return + env * p.R + r, p.last_return + env * p.R + r, v, paid, w.done != 0, MODE == MODE_RESET);
                }
                if (gl == 0) {
                    p.done[env] = (uint8_t)w.done;
                    if (p.done2 && real) p.done2[env] = (uint8_t)w.done;
                    p.err[env] = (uint8_t)err;
                    if (p.ep_length) episode_stat_length(p.ep_length + env, p.last_length + env, paid, w.done != 0, MODE == MODE_RESET);
                }
                if (p.info) {  // Step.info (env.py:174-188): World::n_gems_collected (top-level gems only, world.rs:265-275), n_arrived, Agent.has_arrived
                    uint8_t* io = p.info + env * (2 + A);
                    if (gl == 0) {
                        io[0] = (uint8_t)__popcll(w.collected() & w.m.gem_toplevel);
                        io[1] = (uint8_t)w.n_arrived;
                    }
                    if (gl < A) io[2 + gl] = (uint8_t)((w.arrived >> gl) & 1u);
                }
                if (gl < A) {
                    p.events[env * A + gl] = (uint8_t)ev;
                    p.actions[env * A + gl] = (int8_t)act;
                }
            }
            // auto-reset: the transition above is reported; observation / state / availability below are those
            // of the freshly reset world (SURVEY §8d "Auto-reset")
            const bool do_reset = MODE == MODE_STEP && p.auto_reset && w.done && err == ERR_OK;
            if (__any_sync(kFull, do_reset)) {
                w.reset(do_reset, p.pbrs_set, (uint32_t)(p.env_id_base + (uint64_t)env), (uint32_t)t_now, p.reset_epoch, p.seed, !FAST);
                if constexpr (!FAST)
                    if (p.randomize) recolour(do_reset);
            }

            // compute_available_actions (world.rs:343-363) closes reset (:431), step (:473) and a successful set_state
            // (:595, also reached by the restore at :563); a set_state that fails with InvalidWorldState returns before it,
            // leaving the cache stale, and so do we.
            const bool refresh = MODE != MODE_SET_STATE || err == ERR_OK || err == ERR_STATE_NOT_WALKABLE;
            uint32_t mask = w.available();
            if (refresh) w.store_avail(mask);
            else mask = w.cached_avail();
            if (!p.walkable) mask = w.available_no_walk(mask);  // LLE-level mask (env.py:153-163), output only
            // LaserSubgoal.compute runs when the observation is built (env.py:218-223): after a step or a reset, not
            // after set_state
            if (p.JE && MODE != MODE_SET_STATE) w.sub_e |= w.subgoals_here(p.extras_set);
            w.pack();
            __syncwarp();
            {   // record back to HBM and the small per-step vectors
                uint32_t* out = p.records + env * stride;
                for (int k = gl; k < stride; k += Wd) __stcg(out + k, rec[k]);
                // PyWorldState::as_array (pyworld_state.rs:79-101): [i0,j0,...,gems...,alive...]
                float* st = p.state + env * p.S;
                if (gl < A) {
                    st[2 * gl] = (float)(w.pos >> 8);
                    st[2 * gl + 1] = (float)(w.pos & 0xFFu);
                    st[2 * A + p.G + gl] = ((w.alive >> gl) & 1u) ? 1.0f : 0.0f;
                    uint8_t* av = p.avail + (env * A + gl) * 5;  // LLE.available_actions (env.py:146-163): u8[A,5]
#pragma unroll
                    for (int k = 0; k < 5; ++k) av[k] = (uint8_t)((mask >> k) & 1u);
                }
                if (p.state_obs) {  // StateGenerator.observe (observations.py:155-158): the state row, positions / [H, W] if normalised
                    float* ob = p.obs + env * p.S;
                    if (gl < A) {
                        const float fi = (float)(w.pos >> 8), fj = (float)(w.pos & 0xFFu);
                        // float32 / int64 -> float64 division, stored back into the float32 array
                        ob[2 * gl] = p.state_obs == 2 ? (float)((double)fi / (double)p.H) : fi;
                        ob[2 * gl + 1] = p.state_obs == 2 ? (float)((double)fj / (double)p.W) : fj;
                        ob[2 * A + p.G + gl] = ((w.alive >> gl) & 1u) ? 1.0f : 0.0f;
                    }
                    if (p.G) {
                        const uint64_t coll = w.collected();
                        for (int g = gl; g < p.G; g += Wd) ob[2 * A + g] = ((coll >> g) & 1ull) ? 1.0f : 0.0f;
                    }
                }
                if (p.JE && gl < A) {
                    float* ex = p.extras + (env * A + gl) * p.JE;
                    for (int j = 0; j < p.JE; ++j) ex[j] = ((w.sub_e >> p.extras_beam[j]) & 1ull) ? 1.0f : 0.0f;
                }
                if (p.G) {
                    const uint64_t coll = w.collected();
                    for (int g = gl; g < p.G; g += Wd) st[2 * A + g] = ((coll >> g) & 1ull) ? 1.0f : 0.0f;
                }
            }
        }
        __syncwarp();
        if (!p.write_obs) {
            if (MODE == MODE_STEP && lane == 0) ticket_done<PARTS>(p, ticket, my_seq);
            continue;
        }

        // ================================================================== observations of the group
        if constexpr (FAST) {
            const int agent_base = lane * p.HW;
            const bool multi = p.map_of_env != nullptr;
            const int n_tiles = p.group / p.E;
            for (int tix = 0; tix < n_tiles; ++tix) {
                // the bulk store that last read the tile must have finished reading it
                if (lane == 0) bulk_wait_read<0>();
                __syncwarp();
                if (tile_fresh) {
                    cp_async_wait_all();  // the static planes prefetched at kernel start
                    tile_fresh = false;
                    __syncwarp();
                }
                // Tiles that hold several (tiny) worlds: patch all sub-tiles at once, 32/E lanes per world, when they share
                // one map and already hold its static plane (always, after the first tile, for single-map batches and for
                // batches laid out map by map).  Otherwise fall through to the world-by-world path below.
                bool parallel = false;
                if (p.E > 1) {
                    const int Pr = 32 / p.E, s = lane / Pr, e = lane - s * Pr;
                    const int g = tix * p.E + s;
                    const int mid = multi ? map_ids[g] : 0;
                    const int mid0 = __shfl_sync(kFull, mid, 0);
                    parallel = __all_sync(kFull, mid == mid0);
                    if (parallel) {
                        if (mid0 != render_map) {
                            rm.bind(p.blobs[mid0]);
                            render_map = mid0;
                            pc.load(rm, L, lane);
                        }
                        if (__any_sync(kFull, tags[s] != mid0)) {  // another map: every sub-tile starts from its static plane
                            for (int t = 0; t < p.E; ++t) tile_rebuild_async(tiles + (size_t)t * p.obs_stride, rm, 0, (int)p.obs_stride, lane);
                            cp_async_wait_all();
                            __syncwarp();
                            if (lane < p.E) tags[lane] = mid0;
                            fresh_bits |= p.E >= 32 ? ~0u : ((1u << p.E) - 1u);
                            __syncwarp();
                        }
                        const uint32_t* cur = recs + (size_t)g * stride;
                        const uint32_t* old = applied + (size_t)s * stride;
                        OT* sub = tiles + (size_t)s * p.obs_stride;
                        if (!((fresh_bits >> s) & 1u)) {  // un-patch what the previous occupant had lit and this one has not
                            for (int k = e; k < rm.n_patch; k += Pr) {
                                const LlePatch pe = rm.patches[k];
                                if (rec_lit(old, L, pe) && !rec_lit(cur, L, pe)) sub[pe.idx] = (OT)pe.stat;
                            }
                            for (int a = e; a < A; a += Pr) {
                                const uint32_t op = rec_pos(old, a);
                                sub[a * p.HW + (int)(op >> 8) * p.W + (int)(op & 0xFFu)] = (OT)0;
                            }
                        }
                        fresh_bits &= ~(p.E >= 32 ? ~0u : ((1u << p.E) - 1u));
                        __syncwarp();
                        for (int k = e; k < rm.n_patch; k += Pr) {  // every lit entry is rewritten (aliasing entries, see below)
                            const LlePatch pe = rm.patches[k];
                            if (rec_lit(cur, L, pe)) sub[pe.idx] = (OT)1;
                        }
                        for (int a = e; a < A; a += Pr) {
                            const uint32_t np = rec_pos(cur, a);
                            sub[a * p.HW + (int)(np >> 8) * p.W + (int)(np & 0xFFu)] = (OT)1;
                        }
                        // the tile now shows worlds [tix*E, tix*E + E) of the group: their records are contiguous
                        for (int k = lane; k < p.E * stride; k += 32) applied[k] = recs[(size_t)tix * p.E * stride + k];
                    }
                }
                for (int s = 0; s < (parallel ? 0 : p.E); ++s) {
                    const int g = tix * p.E + s;
                    const uint32_t* cur = recs + (size_t)g * stride;
                    OT* sub = tiles + (size_t)s * p.obs_stride;
                    uint32_t* old = applied + (size_t)s * stride;
                    int mid = 0;
                    if (multi) {
                        mid = map_ids[g];
                        if (mid != render_map) {
                            rm.bind(p.blobs[mid]);
                            render_map = mid;
                            pc.load(rm, L, lane);
                        }
                    }
                    // what this world lights: laser cells whose beam bit is on, uncollected gems (observations.py:256-263)
                    const bool now0 = pc.valid0 && pc.lit0(cur), now1 = pc.valid1 && pc.lit1(cur);
                    if (tags[s] != mid) {
                        tile_rebuild_async(sub, rm, 0, (int)p.obs_stride, lane);  // another map: start from its static plane
                        cp_async_wait_all();
                        if (lane == 0) tags[s] = mid;
                    } else if (!((fresh_bits >> s) & 1u)) {
                        // un-patch what the previous occupant had lit and this one has not
                        if (lane < A) {
                            const uint32_t op = rec_pos(old, lane);
                            sub[agent_base + (int)(op >> 8) * p.W + (int)(op & 0xFFu)] = (OT)0;  // agent planes have no static content
                        }
                        if (pc.valid0 && !now0 && pc.lit0(old)) sub[pc.idx0] = pc.stat0;
                        if (pc.valid1 && !now1 && pc.lit1(old)) sub[pc.idx1] = pc.stat1;
                    }
                    fresh_bits &= ~(1u << s);
                    __syncwarp();
                    // patch.  Every lit entry is rewritten so that entries aliasing one cell (crossing beams of one colour,
                    // colours >= n_agents) stay correct whatever was un-patched above; then the agents (observations.py:264-265).
                    if (now0) sub[pc.idx0] = (OT)1;
                    if (now1) sub[pc.idx1] = (OT)1;
                    if (lane < A) {
                        const uint32_t np = rec_pos(cur, lane);
                        sub[agent_base + (int)(np >> 8) * p.W + (int)(np & 0xFFu)] = (OT)1;
                    }
                    if (lane < stride) old[lane] = cur[lane];
                }
                fence_proxy_async_smem();  // generic-proxy writes above -> visible to the async proxy
                __syncwarp();
                if (lane == 0) {
                    // evict-first: the rows stream through L2 to HBM (491 MB per level-6 step of 65,536 worlds, four times the L2)
                    // and should not push out the records, flags and small outputs the next step reads and rewrites
                    bulk_store_hint(obs_rows<OT>(p) + (env0 + (int64_t)tix * p.E) * p.obs_stride, tiles,
                                    (uint32_t)(p.E * p.obs_stride) * (uint32_t)sizeof(OT), l2_evict_first_policy());
                    bulk_commit();
                    if (p.timeline) {
                        t_last = globaltimer_ns();
                        if (!t_first) t_first = t_last;
                    }
                    if (MODE == MODE_STEP && owed && tix == 0) {
                        bulk_wait<1>();  // every store but the one just issued has completed: the previous ticket is done
                        ticket_done<PARTS>(p, owed_ticket, owed_seq);
                    }
                }
            }
            owed = true; owed_ticket = ticket; owed_seq = my_seq;
            continue;
        } else {
        if constexpr (sizeof(OT) == 4) if (p.obs_kind == LLE_OBS_PARTIAL) {
            // PartialGenerator.observe (observations.py:331-350): per agent a (2A+3, size, size) window centred on it; channels
            // agents, WALL, lasers, GEM, EXIT.  One lane per (agent, window cell): it looks the map cell up once and
            // writes the few non-zero channels into a zero-filled tile, which leaves with one bulk store per E worlds.
            const int sz = p.obs_param, s2 = sz * sz, ctr = sz >> 1, Cp = 2 * A + 3;
            const float inv_s2 = 1.0f / (float)s2, inv_sz = 1.0f / (float)sz;
            const int n_tiles = p.group / p.E, tile_len = p.E * (int)p.obs_stride;
            for (int tix = 0; tix < n_tiles; ++tix) {
                OT* tile = tiles + (size_t)buf * p.tile_floats;
                if (lane == 0) {
                    if (p.n_buf == 2) bulk_wait_read<1>();
                    else bulk_wait_read<0>();
                }
                __syncwarp();
                for (int f = lane * 4; f < tile_len; f += 128) *reinterpret_cast<float4*>(tile + f) = make_float4(0.f, 0.f, 0.f, 0.f);
                __syncwarp();
                for (int s = 0; s < p.E; ++s) {
                    const int g = tix * p.E + s;
                    const int mid = map_ids[g];
                    if (mid != render_map) {
                        rm.bind(p.blobs[mid]);
                        render_map = mid;
                    }
                    const uint32_t* cur = recs + (size_t)g * stride;
                    OT* sub = tile + (size_t)s * p.obs_stride;
                    if constexpr (BY_FEATURE) {
                        // Sparse maps (the host selects this kernel when every map has at most 2 s^2 features): one lane per
                        // (agent, feature) — the map's walls, exits, sources, gems and laser tiles — instead of one per
                        // (agent, window cell): uniform, branch-light tasks.  A 7x7 window of level 6 has 196 cell tasks of
                        // ~100 instructions each; its 300 feature tasks take ~20 each (173 -> 142 us/step).
                        const int F = rm.n_patch;
                        const float inv_f = 1.0f / (float)max(F, 1);
                        for (int t = lane; t < A * F; t += 32) {
                            const int a = (int)(((float)t + 0.5f) * inv_f), f = t - a * F;
                            const LlePatch pe = rm.patches[f];
                            const uint32_t pa = rec_pos(cur, a);
                            const int di = (int)((pe.idx >> 8) & 255u) - (int)(pa >> 8) + ctr;
                            const int dj = (int)(pe.idx & 255u) - (int)(pa & 0xFFu) + ctr;
                            if (di < 0 || dj < 0 || di >= sz || dj >= sz) continue;
                            if (pe.src != LLE_FEATURE_STATIC && !rec_lit(cur, L, pe)) continue;
                            sub[(a * Cp + (int)(pe.idx >> 16)) * s2 + di * sz + dj] = (float)pe.stat;
                        }
                    }
                    for (int q = lane; q < (BY_FEATURE ? 0 : A * s2); q += 32) {
                        // (agent, row, column) of the window cell; the float products are exact for these small integers
                        const int a = (int)(((float)q + 0.5f) * inv_s2), r = q - a * s2;
                        const int wi = (int)(((float)r + 0.5f) * inv_sz), wj = r - wi * sz;
                        const uint32_t pa = rec_pos(cur, a);
                        const int i = (int)(pa >> 8) + wi - ctr, j = (int)(pa & 0xFFu) + wj - ctr;
                        if (i < 0 || j < 0 || i >= p.H || j >= p.W) continue;  // outside the map: all layers stay 0 (:325-329)
                        const int c = i * p.W + j;
                        const uint32_t info = rm.cellinfo[c];
                        if (!(info & (7u | (1u << 24)))) continue;  // plain floor, no beam: nothing but agents (below)
                        OT* o = sub + a * Cp * s2 + r;
                        const uint32_t kind = info & 7u;
                        if (kind == LLE_T_WALL) {
                            // WALL = n_agents; wall_pos holds the walls and the v1 sources (parser_v1.rs:22-25), but not
                            // the sources of a TOML [[lasers]] table
                            if (info & (1u << 25)) o[A * s2] = 1.0f;
                            if (info & 128u) {
                                const int ch = A + 1 + (int)((info >> 16) & 255u);  // LASER_0 + source.agent_id, fill -1 (:348-350)
                                if (ch < Cp) o[ch * s2] = -1.0f;
                            }
                        } else if (kind == LLE_T_EXIT) {
                            o[(2 * A + 2) * s2] = 1.0f;
                        } else if (kind == LLE_T_GEM) {
                            const uint32_t gi = (info >> 8) & 63u;
                            if (!((cur[L.w_gems + (gi >> 5)] >> (gi & 31u)) & 1u)) o[(2 * A + 1) * s2] = 1.0f;
                        }
                        if (info & (1u << 24)) {
                            const LleCellBeams cb = rm.cellbeams[c];
#pragma unroll
                            for (int n = 0; n < 4; ++n) {  // lit lasers listed by World::lasers (:352-360)
                                const uint32_t e = cb.e[n];
                                if (e == LLE_NO_BEAM) break;
                                const int k = be_k(e);
                                if (be_listed(e) && ((cur[L.w_on + be_b(e) * L.on_words + (k >> 5)] >> (k & 31)) & 1u)) {
                                    const int ch = A + 1 + be_colour(e);
                                    if (ch < Cp) o[ch * s2] = 1.0f;
                                }
                            }
                        }
                    }
                    // agent layers (:335-336): agent a2 as seen from agent a, for the A*A ordered pairs
                    for (int t = lane; t < A * A; t += 32) {
                        const int a = t / A, a2 = t - a * A;
                        const uint32_t pa = rec_pos(cur, a), pb = rec_pos(cur, a2);
                        const int di = (int)(pb >> 8) - (int)(pa >> 8) + ctr, dj = (int)(pb & 0xFFu) - (int)(pa & 0xFFu) + ctr;
                        if (di >= 0 && dj >= 0 && di < sz && dj < sz) sub[(a * Cp + a2) * s2 + di * sz + dj] = 1.0f;
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    bulk_store(p.obs + (env0 + (int64_t)tix * p.E) * p.obs_stride, tile, (uint32_t)tile_len * 4u);
                    bulk_commit();
                    if (MODE == MODE_STEP && owed && tix == 0) {
                        bulk_wait<1>();
                        ticket_done<PARTS>(p, owed_ticket, owed_seq);
                    }
                }
                buf = (buf + 1 == p.n_buf) ? 0 : buf + 1;
            }
            owed = true; owed_ticket = ticket; owed_seq = my_seq;
            __syncwarp();
            continue;
        }
        const int tiles_per_group = p.n_chunks > 1 ? p.group : p.group / p.E;
        const bool whole = p.n_chunks == 1;  // a tile holds whole worlds: every patch index is in range
        for (int chunk = 0; chunk < p.n_chunks; ++chunk) {
            const int lo = chunk * p.chunk_floats;  // float range [lo, hi) of one world's block
            const int hi = min(lo + p.chunk_floats, (int)p.obs_stride);
            for (int tix = 0; tix < tiles_per_group; ++tix) {
                OT* tile = tiles + (size_t)buf * p.tile_floats;
                // the bulk store that last read this buffer must have finished reading it
                if (lane == 0) {
                    if (p.n_buf == 2) bulk_wait_read<1>();
                    else bulk_wait_read<0>();
                }
                __syncwarp();
                const int n_sub = whole ? p.E : 1;
                for (int s = 0; s < n_sub; ++s) {
                    const int g = whole ? tix * p.E + s : tix;
                    const int mid = map_ids[g];
                    if (mid != render_map) {
                        rm.bind(p.blobs[mid]);
                        render_map = mid;
                        pc.load(rm, L, lane);
                    }
                    OT* sub_tile = tile + (size_t)s * p.obs_stride;
                    uint32_t* old = applied + ((size_t)buf * p.E + s) * stride;
                    const uint32_t* cur = recs + (size_t)g * stride;
                    const int slot_id = buf * p.E + s;
                    const bool same = tags[slot_id] == mid && tags[p.n_buf * p.E + buf] == chunk;
                    // Patch entries of this tile.  Whole worlds: the first 64 live in registers (pc), the rest is scanned.
                    // Chunks: the entries are sorted by float index and the map gives each chunk's range, so a chunk only
                    // visits its own (a 64x64 map has hundreds of entries and dozens of chunks).
                    const int k_begin = whole ? 64 : (int)__ldg(rm.chunk_tbl + chunk);
                    const int k_end = whole ? rm.n_patch : (int)__ldg(rm.chunk_tbl + chunk + 1);
                    // what this world lights: laser cells whose beam bit is on, uncollected gems (observations.py:256-263)
                    const bool v0 = whole && pc.valid0, v1 = whole && pc.valid1;
                    const bool now0 = v0 && pc.lit0(cur), now1 = v1 && pc.lit1(cur);
                    const bool in0 = whole, in1 = whole;
                    if (!same) {
                        tile_rebuild_async(sub_tile, rm, lo, hi, lane);
                        cp_async_wait_all();
                    } else if (fresh[slot_id]) {
                        cp_async_wait_all();  // the prefetch issued at kernel start
                    } else {
                        // un-patch what the previous occupant had lit and the new one has not
                        for (int k = lane; k < rm.n_ap; k += 32) {
                            const LleAgentPlane ap = rm.agent_planes[k];
                            const uint32_t op = rec_pos(old, (int)ap.agent);
                            const int idx = (int)ap.base + (int)(op >> 8) * p.W + (int)(op & 0xFFu);
                            if (whole || (idx >= lo && idx < hi)) sub_tile[idx - lo] = (OT)0;  // agent planes have no static content
                        }
                        if (v0 && in0 && pc.lit0(old) && !now0) sub_tile[pc.idx0 - lo] = pc.stat0;
                        if (v1 && in1 && pc.lit1(old) && !now1) sub_tile[pc.idx1 - lo] = pc.stat1;
                        for (int k = k_begin + lane; k < k_end; k += 32) {
                            const LlePatch pe = rm.patches[k];
                            if (rec_lit(old, L, pe) && !rec_lit(cur, L, pe)) sub_tile[pe.idx - lo] = (OT)pe.stat;
                        }
                    }
                    __syncwarp();
                    // patch.  Every lit entry is rewritten so that entries aliasing one cell (crossing beams of one colour,
                    // colours >= n_agents) stay correct whatever was un-patched above; then the agents (observations.py:264-265).
                    if (now0 && in0) sub_tile[pc.idx0 - lo] = (OT)1;
                    if (now1 && in1) sub_tile[pc.idx1 - lo] = (OT)1;
                    for (int k = k_begin + lane; k < k_end; k += 32) {
                        const LlePatch pe = rm.patches[k];
                        if (rec_lit(cur, L, pe)) sub_tile[pe.idx - lo] = (OT)1;
                    }
                    for (int k = lane; k < rm.n_ap; k += 32) {
                        const LleAgentPlane ap = rm.agent_planes[k];
                        const uint32_t np = rec_pos(cur, (int)ap.agent);
                        const int idx = (int)ap.base + (int)(np >> 8) * p.W + (int)(np & 0xFFu);
                        if (whole || (idx >= lo && idx < hi)) sub_tile[idx - lo] = (OT)1;
                    }
                    for (int k = lane; k < stride; k += 32) old[k] = cur[k];
                    if (lane == 0) { tags[slot_id] = mid; fresh[slot_id] = 0; }
                }
                if (lane == 0) tags[p.n_buf * p.E + buf] = chunk;
                fence_proxy_async_smem();  // generic-proxy writes above -> visible to the async proxy
                __syncwarp();
                if (lane == 0) {
                    const int64_t first_env = env0 + (whole ? tix * p.E : tix);
                    OT* dst = obs_rows<OT>(p) + first_env * p.obs_stride + lo;
                    const uint32_t bytes = (uint32_t)((whole ? p.E * (int)p.obs_stride : (hi - lo)) * (int)sizeof(OT));
                    bulk_store(dst, tile, bytes);
                    bulk_commit();
                    if (p.timeline) {
                        t_last = globaltimer_ns();
                        if (!t_first) t_first = t_last;
                    }
                    if (MODE == MODE_STEP && owed && chunk == 0 && tix == 0) {
                        bulk_wait<1>();  // every store but the one just issued has completed: the previous ticket is done
                        ticket_done<PARTS>(p, owed_ticket, owed_seq);
                    }
                }
                buf = (buf + 1 == p.n_buf) ? 0 : buf + 1;
            }
        }
        owed = true; owed_ticket = ticket; owed_seq = my_seq;
        }  // !FAST
        __syncwarp();
    }
    if (lane == 0) {
        bulk_wait_all();
        if (MODE == MODE_STEP && owed) ticket_done<PARTS>(p, owed_ticket, owed_seq);
        launch_epilogue(p, MODE == MODE_STEP);
        if (p.timeline) {
            p.timeline[warp_global * 4 + 1] = t_first;
            p.timeline[warp_global * 4 + 2] = t_last;
            p.timeline[warp_global * 4 + 3] = globaltimer_ns();
        }
    }
}

// LaserBeam::enable / disable (laser.rs:69-77) for one source of one map, in every world that uses the map: the whole
// beam turns on (turn_on(0), whoever stands in it) or off.
__global__ void lle_set_beam_kernel(uint32_t* records, LleStateLayout L, int64_t N_pad, const int32_t* map_of_env, int map_index,
                                    int beam, uint64_t mask) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= N_pad) return;
    if (map_of_env && map_of_env[env] != map_index) return;
    uint32_t* w = records + env * L.stride + L.w_on + beam * L.on_words;
    w[0] = (uint32_t)mask;
    if (L.on_words == 2) w[1] = (uint32_t)(mask >> 32);
}

// Gem::collect (gem.rs:17-19) through PyGem.collect (pygem.rs:51-65): gem `gem` of one map becomes collected in every world
// that uses the map; nothing else changes (no event, no reward, slots untouched).
__global__ void lle_collect_gem_kernel(uint32_t* records, LleStateLayout L, int64_t N_pad, const int32_t* map_of_env, int map_index, int gem) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= N_pad) return;
    if (map_of_env && map_of_env[env] != map_index) return;
    records[env * L.stride + L.w_gems + (gem >> 5)] |= 1u << (gem & 31);
}

// The engine record of every world unpacked into plain arrays (EXPORT) or rebuilt from them (IMPORT): what the reference's world
// holds beyond `WorldState` — tile slots, beam bits (world.rs:507-513 drops them), arrival flags, the reward strategy's counters,
// the availability cache and the LaserSubgoal / PBRS flags — so that a batch can be checkpointed and resumed bit-exactly.
struct RawState {  // device pointers, any may be null (lle_raw_state of include/lle_b200.h)
    int16_t* pos;
    uint8_t *alive, *arrived, *slot;
    uint64_t* beam_on;
    uint64_t* collected;
    uint8_t* counters;
    uint8_t* avail_cache;
    uint64_t *sub_extras, *sub_pbrs;
};
template <bool IMPORT>
__global__ void lle_raw_state_kernel(uint32_t* records, LleStateLayout L, int64_t N, int A, int NBmax, RawState r) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= N) return;
    uint32_t* rec = records + env * L.stride;
    if constexpr (IMPORT) {
        uint32_t al = 0, ar = 0, sl = 0;
        for (int a = 0; a < A; ++a) {
            if (r.pos) {
                const uint32_t pp = ((uint32_t)(uint16_t)r.pos[(env * A + a) * 2] << 8) | ((uint32_t)(uint16_t)r.pos[(env * A + a) * 2 + 1] & 0xFFu);
                uint32_t w = rec[a >> 1];
                w = (a & 1) ? ((w & 0xFFFFu) | (pp << 16)) : ((w & 0xFFFF0000u) | pp);
                rec[a >> 1] = w;
            }
            if (r.alive && r.alive[env * A + a]) al |= 1u << a;
            if (r.arrived && r.arrived[env * A + a]) ar |= 1u << a;
            if (r.slot && r.slot[env * A + a]) sl |= 1u << a;
            if (r.avail_cache) reinterpret_cast<uint8_t*>(rec + L.w_avail)[a] = r.avail_cache[env * A + a];
            if (L.sub_words && r.sub_extras && L.w_subp > L.w_sube) {
                rec[L.w_sube + a * L.sub_words] = (uint32_t)r.sub_extras[env * A + a];
                if (L.sub_words == 2) rec[L.w_sube + a * 2 + 1] = (uint32_t)(r.sub_extras[env * A + a] >> 32);
            }
            if (L.sub_words && r.sub_pbrs && L.n_words > L.w_subp) {
                rec[L.w_subp + a * L.sub_words] = (uint32_t)r.sub_pbrs[env * A + a];
                if (L.sub_words == 2) rec[L.w_subp + a * 2 + 1] = (uint32_t)(r.sub_pbrs[env * A + a] >> 32);
            }
        }
        const uint32_t na = r.counters ? r.counters[env * 3] : 0u, nd = r.counters ? r.counters[env * 3 + 1] : 0u, dn = r.counters ? (r.counters[env * 3 + 2] & 1u) : 0u;
        if (!L.wide_flags) {
            rec[L.w_flags] = (al & 0xFFu) | ((ar & 0xFFu) << 8) | ((sl & 0xFFu) << 16) | ((na & 0xFu) << 24) | ((nd > 7u ? 7u : nd) << 28) | (dn << 31);
        } else {
            rec[L.w_flags] = al; rec[L.w_flags + 1] = ar; rec[L.w_flags + 2] = sl;
            rec[L.w_flags + 3] = (na & 0xFFu) | ((nd > 255u ? 255u : nd) << 8) | (dn << 16);
        }
        if (r.collected) {
            if (L.gem_words >= 1) rec[L.w_gems] = (uint32_t)r.collected[env];
            if (L.gem_words == 2) rec[L.w_gems + 1] = (uint32_t)(r.collected[env] >> 32);
        }
        if (r.beam_on)
            for (int b = 0; b < NBmax; ++b) {
                rec[L.w_on + b * L.on_words] = (uint32_t)r.beam_on[env * NBmax + b];
                if (L.on_words == 2) rec[L.w_on + b * 2 + 1] = (uint32_t)(r.beam_on[env * NBmax + b] >> 32);
            }
        return;
    }
    uint32_t al, ar, sl, na, nd, dn;
    if (!L.wide_flags) {
        const uint32_t f = rec[L.w_flags];
        al = f & 0xFF; ar = (f >> 8) & 0xFF; sl = (f >> 16) & 0xFF; na = (f >> 24) & 0xF; nd = (f >> 28) & 7; dn = f >> 31;
    } else {
        al = rec[L.w_flags]; ar = rec[L.w_flags + 1]; sl = rec[L.w_flags + 2];
        const uint32_t mm = rec[L.w_flags + 3];
        na = mm & 0xFF; nd = (mm >> 8) & 0xFF; dn = (mm >> 16) & 1;
    }
    for (int a = 0; a < A; ++a) {
        const uint32_t pp = rec_pos(rec, a);
        if (r.pos) { r.pos[(env * A + a) * 2] = (int16_t)(pp >> 8); r.pos[(env * A + a) * 2 + 1] = (int16_t)(pp & 0xFF); }
        if (r.alive) r.alive[env * A + a] = (al >> a) & 1;
        if (r.arrived) r.arrived[env * A + a] = (ar >> a) & 1;
        if (r.slot) r.slot[env * A + a] = (sl >> a) & 1;
        if (r.avail_cache) r.avail_cache[env * A + a] = reinterpret_cast<const uint8_t*>(rec + L.w_avail)[a];
        if (r.sub_extras) {
            uint64_t v = 0;
            if (L.sub_words && L.w_subp > L.w_sube) {
                v = rec[L.w_sube + a * L.sub_words];
                if (L.sub_words == 2) v |= (uint64_t)rec[L.w_sube + a * 2 + 1] << 32;
            }
            r.sub_extras[env * A + a] = v;
        }
        if (r.sub_pbrs) {
            uint64_t v = 0;
            if (L.sub_words && L.n_words > L.w_subp) {
                v = rec[L.w_subp + a * L.sub_words];
                if (L.sub_words == 2) v |= (uint64_t)rec[L.w_subp + a * 2 + 1] << 32;
            }
            r.sub_pbrs[env * A + a] = v;
        }
    }
    if (r.collected) {
        uint64_t c = 0;
        if (L.gem_words >= 1) c = rec[L.w_gems];
        if (L.gem_words == 2) c |= (uint64_t)rec[L.w_gems + 1] << 32;
        r.collected[env] = c;
    }
    if (r.beam_on) {
        for (int b = 0; b < NBmax; ++b) {
            uint64_t v = rec[L.w_on + b * L.on_words];
            if (L.on_words == 2) v |= (uint64_t)rec[L.w_on + b * 2 + 1] << 32;
            r.beam_on[env * NBmax + b] = v;
        }
    }
    if (r.counters) { r.counters[env * 3] = (uint8_t)na; r.counters[env * 3 + 1] = (uint8_t)nd; r.counters[env * 3 + 2] = (uint8_t)dn; }
}

}  // namespace lle
