// lle_b200 — the step kernel for TINY maps (sm_100a): one THREAD per world.
//
// The general kernel (world_kernel.cuh) gives a world to a group of lanes, one lane per agent, and talks between the
// agents of a world with group ballots and shuffles.  That is the right shape when the observation dominates (level 6:
// 7.5 KB per world), but on a 5x5 map (BASELINE configs[2]: 800 B per world, 2 agents) the step is bound by instruction
// issue: 136 warp-instructions per world, of which the group machinery, the per-lane predicates and the 32/E-lanes-per-world
// tile patching are most (profiles/ncu_cfg3_r01_summary.csv).  Here a lane owns a whole world:
//   * the agents of a world are walked by a compile-time loop (A_ <= 4) in the reference's own order — leave, pre_enter,
//     enter, repeated while somebody died (world.rs:454-505) — with positions, flags and events in registers and the beam /
//     gem masks in a lane-private column of shared memory (dynamic index by beam): no ballots, no shuffles, no predicated
//     phases, and 32 worlds advance per warp pass instead of 32 / Wd;
//   * a 5x5 layered block is 200 floats of which about 16 are not zero (a dozen static cells, the lit laser cells, the
//     uncollected gems, the agents), and a warp meets another map with nearly every ticket of a heterogeneous batch, so there
//     is nothing worth keeping in a tile between tickets.  E worlds at a time, the warp zero-fills a shared-memory tile, ALL
//     lanes (32 / E per world) apply the worlds' render lists — the non-zero static floats, then the dynamic cells, staged in
//     shared memory ahead of time — and the agents' one-hots, and the tile leaves with one TMA bulk store.  What was tried on
//     the way (2^20 worlds, us per step; profiles/cfg3_history_r02.md): un-patching tiles 300, 16-byte copies of the static
//     planes 275, TMA bulk loads of the static planes on mbarriers 284, one lane per world in the tile 277, no tile at all
//     (zero-fill and 4-byte list stores straight to HBM: 40 % fewer instructions, but 19 M tiny L2 write requests) 262,
//     this one 232;
//   * every lane follows its own map (blob pointer per lane), so heterogeneous batches need no uniformity checks.
// Everything around it is the general kernel's protocol, unchanged: tickets of 32 worlds handed out by an atomic counter,
// per-ticket epoch flags for the dataflow ordering between overlapped launches and rollout steps, the record layout
// (static_map.h), Philox action sampling, auto-reset, the host-pipeline flags.  Reset / set_state / refresh launches of the
// same vec run on the general kernel, and so do the steps of a parts loop (lle_vec_parts_*).  Results are bit-identical by construction of the tests (tests/test_gpu_parity.py,
// tests/test_gpu_fullsize.py run both).
#pragma once
#include "tiny_core.cuh"
#include "world_kernel.cuh"

namespace lle {

#ifndef LLE_TINY_LIST2
#define LLE_TINY_LIST2 1
#endif
#ifndef LLE_TINY_MIN_CTAS
#define LLE_TINY_MIN_CTAS 7
#endif

// word k of the record of lane `lane` in the warp's [stride][32] column block
struct SmemColumn {
    uint32_t* base;
    int pitch;
    __device__ __forceinline__ uint32_t& operator()(int word) const { return base[word * pitch]; }
};

// `n` bytes (compile-time) from registers to global memory with the widest stores the alignment of `n` allows
template <int N>
__device__ __forceinline__ void store_bytes(uint8_t* dst, const uint32_t (&b)[N]) {
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int k = 0; k < N; k += 4)
            *reinterpret_cast<uint32_t*>(dst + k) = b[k] | (b[k + 1] << 8) | (b[k + 2] << 16) | (b[k + 3] << 24);
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int k = 0; k < N; k += 2) *reinterpret_cast<uint16_t*>(dst + k) = (uint16_t)(b[k] | (b[k + 1] << 8));
    } else {
#pragma unroll
        for (int k = 0; k < N; ++k) dst[k] = (uint8_t)b[k];
    }
}

// PARTIAL: the observation is PartialGenerator's (A windows of size x size per world, tiny_core.cuh partial_cell_task) instead of
// the layered block; its own instantiation, so that the layered kernel keeps its 72 registers / 7 CTAs per SM.
// OT: the observation's element type, float or int8_t (lle_vec_options.obs_dtype; PARTIAL is float only).  An int8 tile is
// zero-filled and drawn in bytes and leaves with a bulk store of a quarter of the size.
template <int A_, bool PARTIAL = false, typename OT = float>
__global__ void __launch_bounds__(kThreads, PARTIAL ? 4 : LLE_TINY_MIN_CTAS) lle_tiny_step_kernel(const KParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int stride = p.L.stride, w_flags = p.L.w_flags, w_avail = p.L.w_avail, w_gems = p.L.w_gems, w_on = p.L.w_on;
    const bool has_gems = p.L.gem_words != 0;
    const int W = p.W, ostr = (int)p.obs_stride;
    uint8_t* wbase = smem_raw + (size_t)warp * p.warp_smem_bytes;
    uint32_t* srec = reinterpret_cast<uint32_t*>(wbase);                             // [stride][32]: word k of lane l at k*32+l
    uint32_t* snext = srec + stride * 32;                                            // [32][stride]: the NEXT ticket's records, prefetched
    const LlePatch** slptr = reinterpret_cast<const LlePatch**>(snext + stride * 32); // [32]: the render list of lane l's map (PARTIAL: its cellinfo)
    uint32_t* smeta = reinterpret_cast<uint32_t*>(slptr + 32);                       // [32]: n_static | n_patch << 16 of lane l's map
    OT* tile = reinterpret_cast<OT*>(smeta + 32 + (PARTIAL ? 64 : 0));               // [E][ostr]: E worlds per bulk store
    const LleCellBeams** sbeams = reinterpret_cast<const LleCellBeams**>(smeta + 32);  // PARTIAL: [32] the beam table of lane l's map
    const int E = p.E;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    launch_wait(p, lane);

    const uint32_t n_pairs = p.n_tickets * (uint32_t)p.n_steps;
    const bool single_step = p.n_steps == 1;
    uint32_t owed_ticket = 0, owed_seq = 0;
    bool owed = false;
    TinyWorld<A_, SmemColumn> w;
    w.rec = SmemColumn{srec + lane, 32};
    w.L = TinyLayout{w_flags, w_avail, w_gems, w_on, stride, has_gems};
    w.W = W;
    int bound_map = -1;

    // The next (step, ticket) pair is taken, its flag looked at and its records and map index requested while this ticket's
    // observation is rendered: the latencies of a ticket's first loads hide behind the previous ticket's stores.
    bool have_next = false, next_ready = false;
    uint32_t next_pair = 0;
    int next_map = 0;
    const uint32_t warp_global = blockIdx.x * kWarps + warp;
    for (;;) {
        uint32_t pair = next_pair;
        if (!have_next) {  // the first pair
            if (lane == 0) pair = take_pair(p, true, warp_global);
            pair = __shfl_sync(kFull, pair, 0);
        }
        if (pair >= n_pairs) break;
        const bool prefetched = have_next && next_ready;
        have_next = false;
        // (step, ticket) of a pair; one step per launch is the common case and needs no division
        const uint32_t ticket = single_step ? pair : pair % p.n_tickets;
        const int step_index = single_step ? 0 : (int)(pair / p.n_tickets);
        const uint32_t my_seq = p.seq + (uint32_t)step_index;
        if (!prefetched) {
            bool flushed = false;
            if (lane == 0 && !ticket_ready(p.flags + ticket, my_seq - 1u)) {
                if (owed) {  // never block while owing a completion
                    bulk_wait_all();
                    ticket_release(p.flags + owed_ticket, owed_seq);
                    flushed = true;
                }
                while (!ticket_ready(p.flags + ticket, my_seq - 1u)) __nanosleep(64);
            }
            if (__shfl_sync(kFull, (int)flushed, 0)) owed = false;
        }
        const int64_t env = (int64_t)ticket * 32 + lane;  // the ticket is 32 consecutive worlds, one per lane
        const uint64_t t_now = p.t + (uint64_t)step_index;
        const bool real = env < p.N;

        // ---- record -> lane-private column of shared memory (through L2: an overlapped launch may just have written it)
        int map_id = next_map;
        if (prefetched) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            for (int q = 0; q < stride / 4; ++q) {
                const uint4 v = *reinterpret_cast<const uint4*>(snext + lane * stride + 4 * q);
                w.rec(4 * q + 0) = v.x; w.rec(4 * q + 1) = v.y; w.rec(4 * q + 2) = v.z; w.rec(4 * q + 3) = v.w;
            }
        } else {
            const uint4* src = reinterpret_cast<const uint4*>(p.records + env * stride);
            for (int q = 0; q < stride / 4; ++q) {
                const uint4 v = __ldcg(src + q);
                w.rec(4 * q + 0) = v.x; w.rec(4 * q + 1) = v.y; w.rec(4 * q + 2) = v.z; w.rec(4 * q + 3) = v.w;
            }
            map_id = p.map_of_env ? __ldcg(p.map_of_env + env) : 0;
        }
        if (map_id != bound_map) {
            w.bind(p.blobs[map_id]);
            bound_map = map_id;
        }
        w.unpack();
        const uint32_t av_cache = w.rec(w_avail);  // World::available_actions cache: one byte per agent (A_ <= 4)
        // ---- actions (world.rs:444-453): supplied, or sampled uniformly among the available ones
        uint32_t act[A_], ev[A_];
        bool bad = false;
        {
            uint32_t r[4] = {0, 0, 0, 0};
            if (!p.actions_in)
                philox4x32_10((uint32_t)(p.env_id_base + (uint64_t)env), (uint32_t)t_now, 0u, (uint32_t)(t_now >> 32), (uint32_t)p.seed,
                              (uint32_t)(p.seed >> 32), r);
#pragma unroll
            for (int a = 0; a < A_; ++a) {
                const uint32_t av = (av_cache >> (8 * a)) & 0xFFu;
                act[a] = 4u;
                if (p.actions_in) {
                    if (real) act[a] = (uint32_t)(uint8_t)p.actions_in[env * A_ + a];  // padding worlds just STAY
                } else {
                    act[a] = pick_action(r[a], av);
                }
                if (act[a] > 4u || !((av >> act[a]) & 1u)) bad = true;
                ev[a] = 0;
            }
        }
        uint32_t err = ERR_OK;
        if (p.lle_semantics && w.done) err = ERR_DONE;  // env.py:166-167
        else if (bad) err = ERR_INVALID_ACTION;          // the world is left untouched
        const bool paid = err == ERR_OK;
        uint32_t n_gem = 0, n_exit = 0, n_died = 0;
        if (paid) w.step(act, ev, n_gem, n_exit, n_died);
        {   // reward / done / err / events / actions of the transition just taken
            float rw[4];
            w.reward(paid, p.R, n_gem, n_exit, n_died, rw);
            if (p.R == 1) {
                p.reward[env] = rw[0];
                if (p.reward2 && real) p.reward2[env] = rw[0];  // the host's own buffer: N worlds, no padding
            } else {
                *reinterpret_cast<float4*>(p.reward + env * 4) = make_float4(rw[0], rw[1], rw[2], rw[3]);
                if (p.reward2 && real) *reinterpret_cast<float4*>(p.reward2 + env * 4) = make_float4(rw[0], rw[1], rw[2], rw[3]);
            }
            p.done[env] = (uint8_t)w.done;
            if (p.done2 && real) p.done2[env] = (uint8_t)w.done;
            p.err[env] = (uint8_t)err;
            if (p.ep_return) {  // lle_vec_options.episode_stats
                for (int k = 0; k < p.R; ++k) episode_stat_reward(p.ep_return + env * p.R + k, p.last_return + env * p.R + k, rw[k], paid, w.done != 0, false);
                episode_stat_length(p.ep_length + env, p.last_length + env, paid, w.done != 0, false);
            }
            if (p.info) {  // Step.info (env.py:174-188)
                uint8_t* io = p.info + env * (2 + A_);
                io[0] = (uint8_t)__popc(has_gems ? (w.rec(w_gems) & (uint32_t)w.hdr->gem_toplevel) : 0u);
                io[1] = (uint8_t)w.n_arrived;
#pragma unroll
                for (int a = 0; a < A_; ++a) io[2 + a] = (uint8_t)((w.arrived >> a) & 1u);
            }
            store_bytes<A_>(p.events + env * A_, ev);
            store_bytes<A_>(reinterpret_cast<uint8_t*>(p.actions) + env * A_, act);
        }
        // auto-reset: the transition above is reported; observation / state / availability are the fresh world's
        if (p.auto_reset && w.done && err == ERR_OK) w.reset();

        // ---- World::compute_available_actions (world.rs:343-363) + LLE.available_actions (env.py:146-163)
        uint32_t cache = 0, avb[5 * A_];
#pragma unroll
        for (int a = 0; a < A_; ++a) {
            uint32_t mask = w.available(a);
            cache |= mask << (8 * a);
            if (!p.walkable) mask = w.available_no_walk(a, mask);  // LLE-level mask, output only
#pragma unroll
            for (int k = 0; k < 5; ++k) avb[5 * a + k] = (mask >> k) & 1u;
        }
        store_bytes<5 * A_>(p.avail + env * (5 * A_), avb);

        // ---- record back (registers -> column -> HBM) and the state vector (pyworld_state.rs:79-101)
        w.pack(cache);
        {
            uint4* dst = reinterpret_cast<uint4*>(p.records + env * stride);
            for (int q = 0; q < stride / 4; ++q) __stcg(dst + q, make_uint4(w.rec(4 * q + 0), w.rec(4 * q + 1), w.rec(4 * q + 2), w.rec(4 * q + 3)));
            float* st = p.state + env * p.S;
#pragma unroll
            for (int a = 0; a < A_; ++a) {
                st[2 * a] = (float)(w.pos[a] >> 8);
                st[2 * a + 1] = (float)(w.pos[a] & 0xFFu);
                st[2 * A_ + p.G + a] = ((w.alive >> a) & 1u) ? 1.0f : 0.0f;
            }
            if (has_gems) {
                const uint32_t coll = w.rec(w_gems);
                for (int g = 0; g < p.G; ++g) st[2 * A_ + g] = ((coll >> g) & 1u) ? 1.0f : 0.0f;
            }
        }
        __syncwarp();

        // ---- layered observation (observations.py:254-266), E worlds per bulk store
        {   // take the next pair now; if its previous step is already complete, start moving its records and map index
            uint32_t np2 = 0;
            int rdy = 0;
            if (lane == 0) {
                np2 = take_pair(p, false, warp_global);
                if (np2 < n_pairs) rdy = ticket_ready(p.flags + (single_step ? np2 : np2 % p.n_tickets), p.seq + (single_step ? 0u : np2 / p.n_tickets) - 1u) ? 1 : 0;
            }
            next_pair = __shfl_sync(kFull, np2, 0);
            next_ready = __shfl_sync(kFull, rdy, 0) != 0;
            have_next = true;
            if (next_ready) {
                const int64_t env2 = (int64_t)(single_step ? next_pair : next_pair % p.n_tickets) * 32 + lane;
                const uint32_t* src = p.records + env2 * stride;
                for (int q = 0; q < stride / 4; ++q) cp_async16(snext + lane * stride + 4 * q, src + 4 * q);
                asm volatile("cp.async.commit_group;" ::: "memory");
                next_map = p.map_of_env ? __ldcg(p.map_of_env + env2) : 0;
            }
        }
        {
            // E worlds per round are built in a zero-filled shared-memory tile by ALL lanes - 32 / E lanes share a world's render
            // list (read from the owner lane's staged copy and record column) - and leave with one TMA bulk store.
            const int lgE = 31 - __clz(E), lgl = 5 - lgE, lpw = 1 << lgl;  // lanes per world
            if constexpr (PARTIAL) {
                slptr[lane] = reinterpret_cast<const LlePatch*>(w.cellinfo);
                sbeams[lane] = w.cellbeams;
            } else {
                smeta[lane] = (uint32_t)w.n_static | ((uint32_t)w.n_patch << 16);
                slptr[lane] = w.list;
            }
            __syncwarp();
            for (int r = 0; r < (32 >> lgE); ++r) {
                // the store that last read the tile has finished reading it.  (A second tile buffer, so that a round is drawn while the
                // previous one is read, was measured on config 3: E = 2 / 4 with two buffers 238 / 207 us against 190 - it costs
                // warps per SM, and even the unused run-time branch for it cost 3 %.)
                if (lane == 0) bulk_wait_read<0>();
                __syncwarp();
                if constexpr (sizeof(OT) == 4)
                    for (int f = lane * 4; f < E * ostr; f += 128) *reinterpret_cast<float4*>(tile + f) = make_float4(0.f, 0.f, 0.f, 0.f);
                else
                    for (int f = lane * 16; f < E * ostr; f += 512) *reinterpret_cast<uint4*>(tile + f) = make_uint4(0u, 0u, 0u, 0u);
                __syncwarp();
                const int ws = (r << lgE) + (lane >> lgl), q = lane & (lpw - 1);  // the world this lane helps to draw, and its share
                OT* sub = tile + (size_t)(lane >> lgl) * ostr;
                auto agent_pos = [&](int a) {
                    const uint32_t wd = srec[(a >> 1) * 32 + ws];
                    return (a & 1) ? (wd >> 16) : (wd & 0xFFFFu);
                };
                if constexpr (PARTIAL) {
                    // one task per (agent, window cell), then one per ordered pair of agents (observations.py:331-350)
                    const int sz = p.obs_param, s2 = sz * sz;
                    const uint32_t* ci = reinterpret_cast<const uint32_t*>(slptr[ws]);
                    const LleCellBeams* cbm = sbeams[ws];
                    const float inv_s2 = 1.0f / (float)s2;
                    for (int t = q; t < A_ * s2; t += lpw) {
                        const int a = (int)(((float)t + 0.5f) * inv_s2);  // exact for these small integers
                        partial_cell_task(sub, A_, a, t - a * s2, sz, agent_pos(a), p.H, W, ci, cbm, w_gems, w_on, [&](int word) { return srec[word * 32 + ws]; });
                    }
                    for (int t = q; t < A_ * A_; t += lpw) partial_agent_task(sub, A_, t / A_, t % A_, sz, agent_pos(t / A_), agent_pos(t % A_));
                } else {
                    const uint32_t meta = smeta[ws];
                    const int ns = (int)(meta & 0xFFFFu), n = ns + (int)(meta >> 16);
                    auto draw = [&](const LlePatch pe, int k) {
                        if (k < ns) {
                            sub[pe.idx] = (OT)pe.stat;  // static layers (observations.py:216-237)
                        } else {
                            const uint32_t wd = srec[(pe.src == 0xFF ? w_gems : w_on + pe.src) * 32 + ws];
                            if ((((wd >> pe.bit) & 1u) != 0) != (pe.src == 0xFF)) sub[pe.idx] = (OT)1;  // lit laser cell / uncollected gem (:256-263)
                        }
                    };
                    const LlePatch* list = slptr[ws];
#if LLE_TINY_LIST2
                    // two entries in flight per lane: the dependent load of an entry was 10.7 % of the stall samples (config 3: 192.9 -> 189.6 us; three in flight: 190.1)
                    for (int k = q; k < n; k += 2 * lpw) {
                        const int k2 = k + lpw;
                        const LlePatch e0 = list[k];
                        const LlePatch e1 = list[k2 < n ? k2 : k];
                        draw(e0, k);
                        if (k2 < n) draw(e1, k2);
                    }
#else
                    for (int k = q; k < n; k += lpw) draw(list[k], k);
#endif
                    for (int a = q; a < A_; a += lpw) {  // the agents' one-hots (:264-265): their planes hold nothing else
                        const uint32_t pp = agent_pos(a);
                        sub[a * p.HW + (int)(pp >> 8) * W + (int)(pp & 0xFFu)] = (OT)1;
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    bulk_store(obs_rows<OT>(p) + ((int64_t)ticket * 32 + ((int64_t)r << lgE)) * ostr, tile, (uint32_t)(E * ostr) * (uint32_t)sizeof(OT));
                    bulk_commit();
                    if (owed && r == 0) {
                        bulk_wait<1>();  // every store but the one just issued has completed: the previous ticket is done
                        ticket_release(p.flags + owed_ticket, owed_seq);
                    }
                }
            }
        }
        owed = true; owed_ticket = ticket; owed_seq = my_seq;
        __syncwarp();
    }
    if (lane == 0) {
        bulk_wait_all();
        if (owed) ticket_release(p.flags + owed_ticket, owed_seq);
        launch_epilogue(p, true);
    }
}

}  // namespace lle
