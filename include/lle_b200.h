/* lle_b200 — C ABI of the B200-native batched `World` step.
 *
 * This is the drop-in boundary for the hot path of yamoling/lle: the functions below are what the
 * reference's FFI would bind to replace its single-world engine calls by a batched device path.
 * Each entry point cites the reference interface it stands in for (paths relative to the reference
 * repository).  Plain pointers and sizes only; no C++/torch types.  A `lle_vec` is externally
 * synchronised (one caller at a time, one stream), like the reference's `Arc<Mutex<World>>`
 * (src/bindings/world/pyworld.rs:69-82).
 *
 * All functions return a status: 0 on success, otherwise one of the LLE_* codes; the message is
 * available from lle_last_error() (thread-local).
 */
#ifndef LLE_B200_H
#define LLE_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define LLE_API __attribute__((visibility("default")))
#else
#define LLE_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes.  1..99 mirror ParseError (src/core/parsing/errors.rs:5-70), 101..110 mirror
 * RuntimeWorldError (src/core/errors.rs:6-45) as mapped to Python exceptions in
 * src/bindings/pyexceptions.rs:43-183. */
enum {
    LLE_OK = 0,
    LLE_PARSE_EMPTY_WORLD = 1,
    LLE_PARSE_NO_AGENTS = 2,
    LLE_PARSE_INVALID_TILE = 3,
    LLE_PARSE_INVALID_FILE_NAME = 4,
    LLE_PARSE_INVALID_LEVEL = 5,
    LLE_PARSE_NOT_ENOUGH_EXITS = 6,
    LLE_PARSE_NOT_ENOUGH_STARTS = 7,
    LLE_PARSE_DUPLICATE_START = 8,
    LLE_PARSE_INCONSISTENT_DIMENSIONS = 9,
    LLE_PARSE_INVALID_LASER_SOURCE_AGENT_ID = 10,
    LLE_PARSE_INVALID_AGENT_ID = 11,
    LLE_PARSE_INVALID_DIRECTION = 12,
    LLE_PARSE_AGENT_WITHOUT_START = 13,
    LLE_PARSE_INCONSISTENT_WORLD_STRING_WIDTH = 14,  /* TOML v2 maps, src/core/parsing/toml/toml_config.rs */
    LLE_PARSE_INCONSISTENT_WORLD_STRING_HEIGHT = 15,
    LLE_PARSE_INCONSISTENT_NUMBER_OF_AGENTS = 16,
    LLE_PARSE_POSITION_OUT_OF_BOUNDS = 17,
    LLE_PARSE_UNKNOWN_TOML_KEY = 18,
    LLE_PARSE_UNSUPPORTED = 20,
    LLE_LIMIT_EXCEEDED = 21,
    LLE_RT_INVALID_ACTION = 101,
    LLE_RT_INVALID_NUMBER_OF_GEMS = 102,
    LLE_RT_INVALID_NUMBER_OF_AGENTS = 103,
    LLE_RT_INVALID_AGENT_POSITION = 104,
    LLE_RT_OUT_OF_WORLD_POSITION = 105,
    LLE_RT_INVALID_NUMBER_OF_ACTIONS = 106,
    LLE_RT_INVALID_WORLD_STATE = 107,
    LLE_RT_DONE = 110,
    LLE_INDEX_ERROR = 201,
    LLE_INVALID_ARGUMENT = 202,
    LLE_CUDA_ERROR = 300,
    LLE_NO_DEVICE = 301
};

/* ---- per-env error byte written to lle_vec_buffers.err by step / set_state */
enum {
    LLE_ENV_OK = 0,
    LLE_ENV_INVALID_ACTION = 1,     /* world.rs:444-453 : the env is left untouched              */
    LLE_ENV_DONE = 2,               /* env.py:166-167   : stepping a done env without auto-reset  */
    LLE_ENV_STATE_DUPLICATE = 3,    /* world.rs:529-534                                           */
    LLE_ENV_STATE_OUT_OF_WORLD = 4, /* world.rs:536-540                                           */
    LLE_ENV_STATE_NOT_WALKABLE = 5, /* world.rs:556-568 : previous state restored                 */
    LLE_ENV_STATE_MISMATCH = 6      /* world.rs:588-594 : env left modified, as in the reference  */
};

typedef struct lle_map lle_map; /* a compiled, immutable map (host object)         */
typedef struct lle_vec lle_vec; /* N independent worlds resident on one CUDA device */

LLE_API const char* lle_last_error(void);
/* Library / build identification, e.g. "lle_b200 0.1 sm_100a". */
LLE_API const char* lle_version(void);

/* ------------------------------------------------------------------------------------------------
 * Maps.  Replaces `World::try_from(&str)` / `parse` (src/core/world.rs:629-643,
 * src/core/parsing/mod.rs:14-21, parser_v1.rs:132-175, world_config.rs:107-250) and
 * `World::get_level` (world.rs:599-608).
 * ---------------------------------------------------------------------------------------------- */
LLE_API int lle_map_parse(const char* text, size_t len, lle_map** out);
LLE_API int lle_map_level(int level, lle_map** out); /* 1..6, embedded like src/core/levels.rs:1-8 */
LLE_API void lle_map_free(lle_map* map);

typedef struct {
    int32_t height, width, n_agents, n_gems, n_sources, n_channels; /* n_channels = 2*n_agents + 4 */
    int32_t n_exits, n_walls, n_voids, n_laser_cells, n_lasers;     /* n_lasers = len(World::lasers()) */
    int32_t obs_invalid;  /* a laser colour indexes past the last channel: the reference's Layered raises IndexError */
    int32_t max_beam_len;
    uint64_t gem_toplevel; /* bit g: gem g is not under a beam (World::n_gems_collected counts only those, world.rs:265-275) */
} lle_map_info;
LLE_API int lle_map_get_info(const lle_map* map, lle_map_info* out);

/* Position lists as (i, j) pairs: World::{walls, void_positions, exits_positions, gems_positions,
 * starts} (world.rs:125-127, 236-238, 289-303) and the laser cells. Returns the count via *n. */
enum { LLE_POS_WALLS = 0, LLE_POS_VOIDS = 1, LLE_POS_EXITS = 2, LLE_POS_GEMS = 3, LLE_POS_STARTS = 4, LLE_POS_LASER_CELLS = 5 };
LLE_API int lle_map_positions(const lle_map* map, int kind, int32_t* out_ij, int32_t cap, int32_t* n);
/* World::possible_starts (world.rs:297-303; `World.random_start_pos`): the start candidates of `agent` after the laser
 * pruning of laser_setup (world_config.rs:225-243), row-major.  One entry for v1 maps; TOML v2 maps may give several, and
 * World::reset then samples distinct starts (see lle_vec_reset). */
LLE_API int lle_map_start_candidates(const lle_map* map, int32_t agent, int32_t* out_ij, int32_t cap, int32_t* n);
/* World::sources() (world.rs:141-149): 7 ints per source: i, j, agent_id, direction(0 N,1 E,2 S,3 W), enabled, laser_id, beam_len */
LLE_API int lle_map_sources(const lle_map* map, int32_t* out, int32_t cap, int32_t* n);
/* World::lasers() (world.rs:159-172): 7 ints per laser tile: i, j, laser_id, agent_id, direction, beam index, offset in beam */
LLE_API int lle_map_lasers(const lle_map* map, int32_t* out, int32_t cap, int32_t* n);
/* The map text the map was compiled from (World::world_string for unmodified maps). */
LLE_API const char* lle_map_text(const lle_map* map);

/* ------------------------------------------------------------------------------------------------
 * Batched worlds.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t device;          /* CUDA ordinal                                                           */
    int32_t reward_dim;      /* 1 = SingleObjective, 4 = MultiObjective (reward_strategy.py:53, :88)  */
    int32_t walkable_lasers; /* LLE(walkable_lasers=...), env.py:84, :146-163                          */
    int32_t auto_reset;      /* reset a done env inside the step that finished it (not in the reference) */
    int32_t lle_semantics;   /* 1: LLE.step rules (done envs refuse to step, env.py:166-167); 0: raw World */
    int32_t write_obs;       /* 0 skips the layered observation (state/avail/reward still written)     */
    uint64_t seed;           /* Philox key: sampled actions, start sampling, laser colours (World::seed) */
    uint64_t env_id_base;    /* global id of env 0 (sharding over GPUs keeps streams independent of the GPU count) */
    /* LaserSubgoal extras (python/lle/env/extras_generators.py:75-101, Builder.add_extras("laser_subgoal")):
     * n_extras = 0 off, -1 all sources, else the first n_extras entries of extras_src (indices in World::sources() order) */
    int32_t n_extras;
    int32_t extras_src[64];
    /* PotentialShapedLLE (python/lle/env/reward_strategy.py:113-181, Builder.pbrs): pbrs = 1 enables it; n_pbrs / pbrs_src
     * select the rewarded sources like above (-1 = all).  With reward_dim 4 the shaped term is a fifth reward component. */
    int32_t pbrs;
    int32_t n_pbrs;
    int32_t pbrs_src[64];
    double pbrs_gamma, pbrs_reward_value;
    /* Observation type (ObservationType.get_observation_generator, python/lle/observations.py:66-97):
     *   LLE_OBS_LAYERED      obs_param = padding_size: "layered", "flattened" (a view), "layered-padded[-1|-2|-3]"  (:196-293)
     *   LLE_OBS_PARTIAL      obs_param = odd square size: "partial3x3" / "partial5x5" / "partial7x7"               (:296-369)
     *   LLE_OBS_PERSPECTIVE  "perspective" (AgentZeroPerspective)                                                 (:372-395)
     *   LLE_OBS_STATE        obs_param 0 "state", 1 "normalized-state"                                            (:141-158) */
    int32_t obs_type, obs_param;
    /* LLE(randomize_lasers=True) (python/lle/env/env.py:198-200, Builder.randomize_lasers): after every LLE-level reset
     * (lle_vec_reset and auto-reset; not the construction reset) each laser source of the env takes a random colour in
     * [0, n_agents).  The reference draws from Python's global `random` (unpinned); the stream here is this library's own:
     * source b takes word (b & 3) of Philox4x32-10(counter = (env_id_base + env, step count, 0x20000000 | b >> 2, number of
     * explicit resets), key = seed), colour = mulhi(word, n_agents).  Needs n_agents ^ n_sources <= 4096 colourings (each is a
     * precompiled map variant), no laser across a start position and source colours < n_agents; excludes lle_vec_set_source
     * and lle_vec_set_exits. */
    int32_t randomize_lasers;
    /* LLE(state_type=...) / Builder.state_type (python/lle/env/builder.py:51-58, env.py:86, :205-206): the observation generator
     * whose first-agent observation is the environment's *state*.  Default LLE_OBS_STATE / 0 (the state vector, lle_vec_buffers.state).
     * Any other type adds a second observation buffer (lle_vec_buffers.state_obs), rendered from the same engine records by a
     * second launch after every step / reset / set_state; step launches then run strictly one after the other. */
    int32_t state_type, state_param;
    /* 1: also keep, per env, Step.info of LLE.step (python/lle/env/env.py:174-188) and episode statistics, written by the step kernel
     * (lle_vec_buffers.info / ep_return / ep_length / last_return / last_length): about 20 more bytes per env-step. */
    int32_t episode_stats;
    /* Element type of `obs` (LLE_DTYPE_*).  Every value of a layered, padded, flattened or perspective observation is -1, 0 or 1,
     * so LLE_DTYPE_I8 stores the same observation in a quarter of the bytes (lle_vec_buffers.obs_i8; `obs` is then NULL).
     * LLE_OBS_PARTIAL and LLE_OBS_STATE are f32 only.  The state_type observation (state_obs) is always f32. */
    int32_t obs_dtype;
} lle_vec_options;
enum { LLE_OBS_LAYERED = 0, LLE_OBS_PARTIAL = 1, LLE_OBS_PERSPECTIVE = 2, LLE_OBS_STATE = 3 };
enum { LLE_DTYPE_F32 = 0, LLE_DTYPE_I8 = 1 };
LLE_API void lle_vec_default_options(lle_vec_options* opts);

/* All maps must share (height, width, n_agents, n_gems).  map_of_env may be NULL (every env uses maps[0]). */
LLE_API int lle_vec_create(const lle_map* const* maps, int32_t n_maps, const int32_t* map_of_env, int64_t n_envs,
                   const lle_vec_options* opts, lle_vec** out);
LLE_API int lle_vec_destroy(lle_vec* vec);

/* Device pointers of the per-step outputs (valid until lle_vec_destroy).  Layouts, C-contiguous:
 *   obs      f32 [N, obs_stride]   one block per env (obs_stride = block length rounded up to 4 floats), by obs_type:
 *            (obs_i8: i8 [N, obs_stride] instead, obs_stride rounded up to 16 bytes, when obs_dtype is LLE_DTYPE_I8)
 *                                    layered      (C,H,W) = LayeredPadded.observe()[0] (observations.py:254-266), C = 2(A+padding)+4;
 *                                                 the reference's (A+padding,C,H,W) np.tile is a stride-0 repeat of it
 *                                    partial      (A, 2A+3, size, size): every agent's own window (:331-350)
 *                                    perspective  (A, C, H, W): every agent's own permuted copy (:381-395)
 *                                    state        (3A+G,), obs_stride = 3A+G; repeated per agent by the reference (:155-158)
 *   state    f32 [N, 3A+G]         PyWorldState::as_array (pyworld_state.rs:79-101)
 *   avail    u8  [N, A, 5]         LLE.available_actions (env.py:146-163), indexed by Action value
 *   reward   f32 [N, reward_dim]   reward_strategy.py:58-75 / :90-109
 *   done     u8  [N]               LLE.compute_done (env.py:253-254) of the transition just taken
 *   events   u8  [N, A]            bits 0-1: event of the first move_agents pass (0 none, 1 AgentExit,
 *                                  2 GemCollected, 3 AgentDied); bits 2-7: pass >= 2 in which the agent died
 *                                  (world.rs:468-472).  Ordered list = sort by (pass, agent).
 *   actions  i8  [N, A]            the joint action applied (sampled or supplied)
 *   err      u8  [N]               LLE_ENV_*
 *   extras   f32 [N, A, extras_dim] LaserSubgoal.compute (extras_generators.py:93-98); NULL when extras are off */
typedef struct {
    int64_t n_envs;
    int32_t n_agents, n_gems, n_channels, height, width, reward_dim, state_dim, n_beams_max;
    int64_t obs_stride; /* elements of the vec's obs_dtype: a multiple of 4 (f32) or of 16 (i8) */
    float* obs;
    float* state;
    uint8_t* avail;
    float* reward;
    uint8_t* done;
    uint8_t* events;
    int8_t* actions;
    uint8_t* err;
    int64_t record_bytes; /* bytes of the per-env engine record kept in HBM (read + written once per step) */
    float* extras;
    int32_t extras_dim;
    int32_t pad;
    int32_t obs_type, obs_param;
    int32_t obs_view_agents;        /* > 0: the agent dimension is a stride-0 repeat of the block (np.tile); 0: materialised */
    int32_t obs_c, obs_h, obs_w;    /* one agent's observation: (obs_c, obs_h, obs_w); state: (obs_c,) */
    int32_t obs_invalid;            /* some map's laser colour indexes past the last channel of this observation type: the
                                       reference raises IndexError when it builds / runs the generator */
    int32_t pad2;
    int32_t* map_index;             /* i32[N] or NULL: index of each env's current map; with randomize_lasers:
                                       map * n_variants + colouring, colouring = sum over sources b of colour_b * n_agents^b */
    int32_t n_variants;             /* colourings per map (1 without randomize_lasers) */
    int32_t pad3;
    /* state_type other than the state vector: one block per env laid out like `obs` for that type (NULL otherwise).  The
     * reference's state is the FIRST agent's observation (observations.py:118-119): the block itself when state_view_agents > 0,
     * else its first (state_c, state_h, state_w) part. */
    float* state_obs;
    int64_t state_obs_stride;
    int32_t state_type, state_param, state_view_agents, state_c, state_h, state_w;
    /* episode_stats (NULL otherwise).  info u8[N, 2 + A] of the transition just taken, before an auto-reset: gems_collected
     * (World::n_gems_collected, world.rs:265-275), n_arrived (exit_rate = n_arrived / A), has-arrived-i; is-alive-i is the tail of
     * `state`.  ep_return f32[N, reward_dim] / ep_length i32[N]: reward summed over, and steps of, the running episode;
     * last_return / last_length: the same of the env's last finished episode (latched by the step that sets done). */
    uint8_t* info;
    float* ep_return;
    int32_t* ep_length;
    float* last_return;
    int32_t* last_length;
    /* obs_dtype LLE_DTYPE_I8: the observation rows (obs is NULL); NULL for an f32 vec */
    int8_t* obs_i8;
    int32_t obs_dtype;
    int32_t pad4;
} lle_vec_buffers;
LLE_API int lle_vec_get_buffers(lle_vec* vec, lle_vec_buffers* out);

/* World::reset / LLE.reset (world.rs:411-432, env.py:191-203) for every env, or for the envs whose byte in
 * `mask_dev` (device, u8[N]) is non-zero.  Rewrites obs/state/avail; clears reward/done/events/err of those envs. */
LLE_API int lle_vec_reset(lle_vec* vec, const uint8_t* mask_dev, void* cuda_stream);
/* Maps with several start candidates per agent (TOML v2): every reset — explicit or automatic — samples distinct start
 * positions like sample_different (src/utils/mod.rs:39-86).  The reference draws from rand::StdRng, whose stream is not
 * pinned by any test or lockfile; this library defines its own: for attempt n = 0..15, agent a draws word (a & 3) of
 * Philox4x32-10(counter = (env_id_base + env, step count, 0x40000000 | n << 8 | a >> 2, number of explicit resets so far),
 * key = seed) and probes its row-major sorted candidates cyclically from index mulhi(word, count); agents are served by
 * increasing number of candidates (stable) and take the first candidate no earlier agent took; an agent with no free
 * candidate fails the attempt; after 16 failed attempts a fixed assignment (bipartite matching) is used. */

/* Re-exports observation / state / availability (and extras) of every env from its current engine state without resetting
 * any (after lle_vec_set_source / lle_vec_set_exits, when the change should show before the next step). */
LLE_API int lle_vec_refresh(lle_vec* vec, void* cuda_stream);

/* World::step + LLE.step (world.rs:435-475, env.py:165-189) for every env in one kernel launch.
 * actions_dev: device i8[N, A] of Action values, or NULL to sample uniformly among the available
 * actions with Philox4x32-10 (key = seed, counter = (env_id_base+env, step, agent/4)). */
LLE_API int lle_vec_step(lle_vec* vec, const int8_t* actions_dev, void* cuda_stream);

/* `n_steps` consecutive lockstep steps with device-sampled actions in ONE launch.  Bit-identical to calling
 * lle_vec_step(vec, NULL, stream) n_steps times: every step writes all of its outputs (the buffers end up holding
 * the last step's), but each warp keeps ownership of its worlds across steps, so there is no launch gap and no
 * ramp-up / drain between steps. */
LLE_API int lle_vec_rollout(lle_vec* vec, int32_t n_steps, void* cuda_stream);

/* Same step, host-facing: copies `actions_host` (i8[N,A], pinned for async behaviour; NULL = device sampling)
 * to the device, steps, and copies reward (f32[N,reward_dim]) and done (u8[N]) back, then synchronises the
 * stream.  The observation stays resident in HBM (zero-copy DLPack hand-off to the policy). */
LLE_API int lle_vec_step_host(lle_vec* vec, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* cuda_stream);

/* Copies `bytes` bytes, starting at byte `offset`, of one of the per-step buffers of lle_vec_get_buffers to host memory after
 * waiting for the work queued on cuda_stream - for hosts without a CUDA runtime of their own (the reference's Rust crate), e.g.
 * to look at an observation or to record the actions the device sampled.  The same role as lle_gen_fetch. */
enum { LLE_BUF_OBS = 0, LLE_BUF_STATE = 1, LLE_BUF_AVAIL = 2, LLE_BUF_REWARD = 3, LLE_BUF_DONE = 4, LLE_BUF_EVENTS = 5, LLE_BUF_ACTIONS = 6,
       LLE_BUF_ERR = 7, LLE_BUF_EXTRAS = 8, LLE_BUF_STATE_OBS = 9, LLE_BUF_INFO = 10 };
LLE_API int lle_vec_fetch(lle_vec* vec, int which, size_t offset, size_t bytes, void* host_dst, void* cuda_stream);

/* Page-locked (pinned) host memory for the host-facing calls below.  lle_vec_pipeline_submit REQUIRES its action / reward / done
 * buffers to be pinned (memory from here, cudaHostAlloc, cudaHostRegister or torch's pin_memory): the step kernel waits on the
 * device for the action copy and writes reward / done straight into the host buffers.  A host without a CUDA runtime of its own
 * (the reference's Rust crate) allocates them here. */
LLE_API int lle_host_alloc(size_t bytes, void** out);
LLE_API int lle_host_free(void* ptr);

/* Pipelined host stepping: the same step as lle_vec_step_host without the per-step stream synchronisation.
 * lle_vec_pipeline_submit enqueues (1) the copy of `actions_host` (pinned i8[N,A]; NULL = device sampling) on a copy
 * stream and (2) the fused step on the vec's own compute stream, which waits for the actions inside the kernel and writes
 * reward / done (pinned f32[N,reward_dim] / u8[N]) straight into the host buffers, followed by a completion word in pinned
 * memory; it returns at once.  lle_vec_pipeline_wait polls that word: it blocks until the OLDEST submitted step's results are
 * in its host buffers.  Up to 8 steps may be outstanding; with two or more, the copies of one step overlap the kernels of its
 * neighbours and consecutive step kernels stay back to back (programmatic dependent launch), so an OPEN host-driven loop runs
 * at the device rate.  A CLOSED loop (the actions of step t+1 depend on the results of step t) uses lle_vec_parts_* below.
 * The first submit after the pipeline was empty is ordered after the work already in `after_stream` (pass LLE_STREAM_NONE when
 * nothing the step depends on is pending on any stream: saves two driver calls per step of a closed loop); no other call
 * on the vec is allowed until the pipeline has been drained.  Device buffers (lle_vec_get_buffers) are updated as usual. */
#define LLE_STREAM_NONE ((void*)(intptr_t)-1)
LLE_API int lle_vec_pipeline_submit(lle_vec* vec, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* after_stream);
LLE_API int lle_vec_pipeline_wait(lle_vec* vec, int32_t* outstanding);

/* ---- Closed loop over PARTS of one batch (the EnvPool pattern without sub-batch launches).
 * A host policy that needs step t's results before it can choose step t+1's actions leaves the device idle for a round trip
 * per step (lle_vec_step_host), or steps sub-batches as separate vecs and pays a launch ramp and tail per sub-batch.  Here
 * the batch stays ONE vec and every step ONE launch over all of it; the dependency is enforced per part (n_parts contiguous
 * env ranges, multiples of the kernel's ticket size: lle_vec_parts_range) on the device:
 *   lle_vec_parts_begin   opens the loop on three pinned buffers (lle_host_alloc): actions i8[N,A], which the step kernel reads in
 *                         place, reward f32[N,reward_dim] and done u8[N], which it writes in place (either may be NULL).
 *   lle_vec_parts_launch  enqueues one step of the whole batch and returns.  Its tickets of part k start once the host has
 *                         released the part's actions for that step (lle_vec_parts_feed), so it may be - and should be: keep two
 *                         in flight - launched before the previous step has finished; at most four may be in flight.
 *   lle_vec_parts_feed    the host has written the actions of `part` for its next step into the actions buffer: release them
 *                         (one stream memory operation, no copy).  Only after the part's previous step was waited for.
 *   lle_vec_parts_wait    blocks until the oldest fed, un-waited step of `part` has put the part's reward / done into the host
 *                         buffers (the kernel publishes a per-part completion word in pinned memory, which this call polls).
 *   lle_vec_parts_end     closes the loop; every launched step must have been fed and waited for on every part (a launched step
 *                         waits for its actions ON THE DEVICE).  lle_vec_parts_abort releases whatever is still waited for
 *                         (those steps then run on whatever the actions buffer holds), drains and closes: for error paths;
 *                         lle_vec_destroy calls it.
 * A launched step that is never fed keeps spinning on the device and blocks every device-wide synchronisation of the process:
 * always end or abort the loop (the Python wrapper does so when the loop object is dropped or an exception leaves its block).
 * For the same reason keep ONE parts loop per device going at a time from a host thread: the waiting CTAs of one loop's launch can
 * fill the SMs, and if the host then blocks in lle_vec_parts_wait on another vec whose kernel cannot become resident, neither moves.
 * (And a parts loop cannot run under a profiler that serialises kernel launches, e.g. ncu: the launch call would
 * only return once the step has its actions, which the same thread releases after the call.)
 * Per step and part the host pays one poll and one driver call; the device runs full-width step kernels back to back, the parts
 * of consecutive steps overlapping (B200, level 6 x 65,536, 8 parts, compiled host: 84 us per step against 80 us for device-side
 * stepping and 108 us for eight sub-batch vecs).  Results (every buffer of lle_vec_get_buffers) are bit-identical to lle_vec_step
 * with the same actions.  No other call on the vec is allowed while the loop is open.  Replaces: a loop of LLE.step
 * (python/lle/env/env.py:165-189) over a vector of envs whose policy runs on the host between steps.  `after_stream`: as for
 * lle_vec_pipeline_submit. */
LLE_API int lle_vec_parts_begin(lle_vec* vec, int32_t n_parts, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* after_stream);
LLE_API int lle_vec_parts_count(lle_vec* vec, int32_t* n_parts);  /* the number of parts actually formed: <= the number asked for (1..1024), at least one ticket (8-32 envs) each */
LLE_API int lle_vec_parts_range(lle_vec* vec, int32_t part, int64_t* first_env, int64_t* n_envs);
LLE_API int lle_vec_parts_launch(lle_vec* vec);
LLE_API int lle_vec_parts_feed(lle_vec* vec, int32_t part);
LLE_API int lle_vec_parts_wait(lle_vec* vec, int32_t part);
LLE_API int lle_vec_parts_end(lle_vec* vec);
LLE_API int lle_vec_parts_abort(lle_vec* vec);

/* Laser-source mutators for every env that uses map `map_index` (index into the maps given to lle_vec_create):
 * LaserBeam::set_agent_id / enable / disable (src/core/tiles/laser.rs:69-84, exposed as PyLaserSource.agent_id / set_colour /
 * enable / disable, src/bindings/tiles/pylaser_source.rs:55-142).  agent_id < 0 keeps the colour, enabled < 0 keeps the
 * switch.  Disabling turns the whole beam off, enabling turns the whole beam on (turn_on(0): whoever stands in it), and
 * both survive World::reset (laser.rs:168-171).  The colour is NOT checked against n_agents here (the engine does not,
 * world_config.rs:137-145; the Python setter does).  Observation / state / availability buffers keep showing the last
 * step until the next step or reset (lle_vec_refresh re-exports every env without resetting any).
 * Synchronises `cuda_stream`.  lle_vec_get_sources: current (agent_id, enabled) pairs of the map's sources. */
LLE_API int lle_vec_set_source(lle_vec* vec, int32_t map_index, int32_t source_index, int32_t agent_id, int32_t enabled, void* cuda_stream);
LLE_API int lle_vec_get_sources(lle_vec* vec, int32_t map_index, int32_t* out_pairs, int32_t cap, int32_t* n);

/* Gem::collect (src/core/tiles/gem.rs:17-19) as reached through PyGem.collect (src/bindings/tiles/pygem.rs:51-65): gem
 * `gem_index` (World::gems order) of map `map_index` becomes collected in every env of that map; nothing else changes (no
 * event, no reward).  LLE_INVALID_ARGUMENT when the gem sits under a laser tile (a Tile::Laser there, "not a gem").  Call
 * lle_vec_refresh to re-export observation / state. */
LLE_API int lle_vec_collect_gem(lle_vec* vec, int32_t map_index, int32_t gem_index, void* cuda_stream);

/* World::set_exit_positions (src/core/world.rs:195-234; the `World.exit_pos` setter, pyworld.rs:202-210) for every env that
 * uses map `map_index`: the current exits become floor tiles and the (i, j) pairs of `exits_ij` become the exits.  Agents keep
 * their position, alive and arrived flags.  Fewer exits than agents -> LLE_PARSE_NOT_ENOUGH_EXITS.  A new exit must be a
 * floor, start or former exit cell crossed by at most one beam (the reference panics or corrupts its grid otherwise).
 * Synchronises `cuda_stream`; buffers show the change from the next step / reset on. */
LLE_API int lle_vec_set_exits(lle_vec* vec, int32_t map_index, const int32_t* exits_ij, int32_t n_exits, void* cuda_stream);

/* World::set_state / LLE.set_state (world.rs:515-597, env.py:208-216) for every env.
 *   pos_dev i32[N,A,2], gems_dev u8[N,G], alive_dev u8[N,A] (device).  Per-env failures are reported in err. */
LLE_API int lle_vec_set_state(lle_vec* vec, const int32_t* pos_dev, const uint8_t* gems_dev, const uint8_t* alive_dev, void* cuda_stream);

/* Raw engine state (the part of the reference's world that WorldState does not carry), unpacked on the
 * device into caller-provided device arrays; any pointer may be NULL.
 *   pos i16[N,A,2]; alive/arrived/slot u8[N,A] (Agent.dead/arrived, tile slot, agent.rs:6-10, tile.rs:86-99);
 *   beam_on u64[N,n_beams_max] (bit k = LaserBeam.beam[k], laser.rs:16); collected u64[N]; counters u8[N,3] = n_arrived, n_deads, done */
LLE_API int lle_vec_export_raw(lle_vec* vec, int16_t* pos, uint8_t* alive, uint8_t* arrived, uint8_t* slot, uint64_t* beam_on,
                       uint64_t* collected, uint8_t* counters, void* cuda_stream);

/* The whole engine record, for checkpoints: lle_vec_export_raw plus the World::available_actions cache (world.rs:37, one 5-bit
 * mask per agent, bit = Action value) and the LaserSubgoal / PotentialShapedLLE flags (bit b = source b), and its inverse.
 * A batch re-created with the same maps and options, given lle_vec_import_raw_state(exported arrays), the step count
 * (lle_vec_set_step_count), the reset count (lle_vec_set_reset_count) and - with randomize_lasers - the map_index buffer,
 * continues bit-identically (the reference's WorldState alone cannot: it drops beam bits, slots and arrivals, world.rs:507-513).
 * Export: any pointer may be NULL.  Import: every array of a feature the vec uses is required; observation / state /
 * availability buffers are re-exported from the imported records (lle_vec_refresh).  Device pointers. */
typedef struct {
    int16_t* pos;              /* i16[N,A,2] */
    uint8_t* alive;            /* u8[N,A] */
    uint8_t* arrived;          /* u8[N,A] */
    uint8_t* slot;             /* u8[N,A] */
    uint64_t* beam_on;         /* u64[N,n_beams_max] */
    uint64_t* collected;       /* u64[N] */
    uint8_t* counters;         /* u8[N,3] n_arrived, n_deads (saturating), done */
    uint8_t* avail_cache;      /* u8[N,A] */
    uint64_t* subgoals_extras; /* u64[N,A] */
    uint64_t* subgoals_pbrs;   /* u64[N,A] */
} lle_raw_state;
LLE_API int lle_vec_export_raw_state(lle_vec* vec, const lle_raw_state* dst, void* cuda_stream);
LLE_API int lle_vec_import_raw_state(lle_vec* vec, const lle_raw_state* src, void* cuda_stream);
/* Number of explicit resets so far: a word of the start-sampling / laser-recolouring Philox counters (see lle_vec_reset). */
LLE_API int lle_vec_get_reset_count(lle_vec* vec, uint32_t* out);
LLE_API int lle_vec_set_reset_count(lle_vec* vec, uint32_t value);

/* World::seed (world.rs:92-96): the Philox key of the action sampler and of the start sampler. */
LLE_API int lle_vec_set_seed(lle_vec* vec, uint64_t seed);
/* Step counter used as the Philox counter word (incremented by every lle_vec_step). */
LLE_API int lle_vec_get_step_count(lle_vec* vec, uint64_t* out);
LLE_API int lle_vec_set_step_count(lle_vec* vec, uint64_t value);

/* Number of kernels this library launched since the vec was created (bench.py's `gpu_launches`). */
LLE_API int lle_vec_launch_count(lle_vec* vec, uint64_t* out);

/* Average device time (ms, CUDA events on the launching stream) of the step kernels launched between
 * lle_vec_timing_begin and lle_vec_timing_end; *launches receives how many were timed. */
LLE_API int lle_vec_timing_begin(lle_vec* vec, void* cuda_stream);
LLE_API int lle_vec_timing_end(lle_vec* vec, void* cuda_stream, float* total_ms, uint64_t* launches);

/* Development aid (only when the vec was created with LLE_B200_TIMELINE=1 in the environment): per warp of the last
 * launch, 4 globaltimer readings in ns: kernel start, first observation store issued, last store issued, warp end. */
LLE_API int lle_vec_debug_timeline(lle_vec* vec, uint64_t* out_host, int64_t cap_warps, int64_t* n_warps);

/* =====================================================================================================================
 * Layout generator (SURVEY 8f rank 4): `lle.generate(...)` / `WorldGenerator` of python/lle/generator/generator.py, one
 * *attempt* per device thread.
 *
 * An attempt is `WorldGenerator._try_generate(seed)` with constraint=None (generator.py:243-254): seed a
 * `random.Random`, place agents -> exits -> lasers -> walls -> gems (generator.py:188-228, placements.py, geometry.py),
 * check the beam geometry (candidates.py:27-41).  The device code re-implements CPython's `random.Random` (MT19937 seeded
 * with an int, `_randbelow_with_getrandbits`, `sample`, `shuffle`, `choice`, `randint`, `choices`; CPython 3.12), so the
 * layout of seed s is the reference's layout for that seed, bit for bit (tests/golden/generator_vectors.json).
 * Batches correspond to the reference's parallel path `_generate_n_multi` (generator.py:296-314), whose attempts are
 * seeded one by one with `rng.randrange(sys.maxsize)`: lle_gen_attempt_seeds reproduces that seed list.
 *
 * Not the reference's: (1) `cluster_shape` is an option (placements.py:44-60 draws it from Python's global, unseeded
 * generator in each of its three callers; here one shape serves all three); (2) the `labels` byte is a breadth-first
 * reachability heuristic of this library - LLE_GEN_WALKABLE: the agents can be matched to distinct exits they reach
 * through non-wall, non-source cells; LLE_GEN_INDEPENDENT: the same when agent a also avoids every cell lit (at reset,
 * nobody blocking) by a beam of another colour; LLE_GEN_NEEDS_BLOCKER: walkable but not independent.  It is NOT the
 * SAT-based `Cooperative()` / `Independent()` predicates of world_filter.py (out of scope).
 * Limits: height, width <= 32; n_agents <= 32.
 * ===================================================================================================================== */
typedef struct lle_gen lle_gen;

enum { LLE_GEN_STARTS_RANDOM = 0, LLE_GEN_STARTS_EDGE = 1, LLE_GEN_STARTS_CLUSTERED = 2 };
enum { LLE_GEN_EXITS_RANDOM = 0, LLE_GEN_EXITS_EDGE = 1, LLE_GEN_EXITS_CLUSTER = 2, LLE_GEN_EXITS_OPPOSITE = 3 };
enum { LLE_GEN_LASERS_FREE = 0, LLE_GEN_LASERS_CROSS_AGENT = 1, LLE_GEN_LASERS_CROSS_CLUSTER = 2 };
enum { LLE_GEN_SPAN_ANY = 0, LLE_GEN_SPAN_ACROSS = -1 };           /* or an explicit minimum length >= 2 */
enum { LLE_GEN_WALLS_AUTO = -1 };                                   /* (width * height) / 10, generator.py:165 */
enum { LLE_GEN_WALKABLE = 1, LLE_GEN_INDEPENDENT = 2, LLE_GEN_NEEDS_BLOCKER = 4 };
/* cell codes of the generated grids */
enum { LLE_CELL_FLOOR = 0, LLE_CELL_WALL = 1, LLE_CELL_EXIT = 2, LLE_CELL_GEM = 3, LLE_CELL_START = 16 /* + agent */,
       LLE_CELL_SOURCE = 64 /* + 4 * colour + direction (0 N, 1 S, 2 E, 3 W) */ };

/* The keyword arguments of WorldGenerator.__init__ (generator.py:97-114). */
typedef struct {
    int32_t width, height, n_agents;
    int32_t starts, exits;
    int32_t n_lasers, n_gems;
    int32_t laser_placement, laser_span;
    int32_t n_walls, walls_shapes;                   /* walls_style: 0 "individual", 1 "shapes" */
    int32_t n_rooms_rows, n_rooms_cols, door_size;   /* rooms mode when n_rooms_rows > 0 (generator.py:156-161) */
    int32_t cluster_h, cluster_w;                    /* clustered starts / exits only */
} lle_gen_options;
LLE_API void lle_gen_default_options(lle_gen_options* opts);

/* Validates like WorldGenerator.__init__ (generator.py:116-181; LLE_INVALID_ARGUMENT carries its message) and allocates
 * device buffers for `capacity` attempts per run. */
LLE_API int lle_gen_create(const lle_gen_options* opts, int32_t device, int64_t capacity, lle_gen** out);
LLE_API int lle_gen_destroy(lle_gen* gen);

/* generator.py:296-301: out[i] = the i-th `rng.randrange(sys.maxsize)` after `rng.seed(seed)` (host, MT19937). */
LLE_API int lle_gen_attempt_seeds(uint64_t seed, int64_t n, uint64_t* out);

/* Runs n <= capacity independent chains on the device, one per thread.  Chain i seeds its generator with seeds_dev[i] (or
 * first_seed + i when seeds_dev is NULL) and makes up to max_attempts attempts from that one stream, stopping at the first
 * layout whose label byte contains every bit of `require` (0: any layout): max_attempts = 1 is
 * `WorldGenerator._try_generate(seed)`, max_attempts = m is `WorldGenerator.generate(m, seed)` (generator.py:268-284), both
 * with the label test in the place of the reference's constraint (`_accept_world` draws no random number). */
LLE_API int lle_gen_run(lle_gen* gen, const uint64_t* seeds_dev, uint64_t first_seed, int64_t n, int32_t max_attempts, uint32_t require,
                        void* cuda_stream);

typedef struct {
    int64_t capacity, n;       /* n: chains of the last run */
    int32_t height, width;
    uint8_t* cells;            /* u8[capacity, height*width] cell codes (all floor when the chain found nothing) */
    uint8_t* status;           /* u8[capacity] 1 = layout, 0 = none (LayoutRetry / rejected in every attempt) */
    uint8_t* labels;           /* u8[capacity] LLE_GEN_* bits (0 when status is 0) */
    int32_t* tries;            /* i32[capacity] attempts the chain used */
} lle_gen_buffers;
LLE_API int lle_gen_get_buffers(lle_gen* gen, lle_gen_buffers* out);

/* Copies chains [first, first + n) of the last run into host buffers (any of them may be NULL) after waiting for the work
 * queued on cuda_stream: cells u8[n, height*width], status u8[n], labels u8[n], tries i32[n].  For hosts without a CUDA
 * runtime of their own (the same role as lle_vec_step_host). */
LLE_API int lle_gen_fetch(lle_gen* gen, int64_t first, int64_t n, uint8_t* cells_host, uint8_t* status_host, uint8_t* labels_host,
                          int32_t* tries_host, void* cuda_stream);

/* `CandidateLayout.is_geometry_valid` (python/lle/generator/candidates.py:27-41) of a cell grid (host): every source has an
 * in-bounds first beam cell and a beam of >= 2 cells before a wall or another source, and no exit lies on a beam. */
LLE_API int lle_gen_geometry_valid(const uint8_t* cells_host, int32_t height, int32_t width, int32_t* valid);

/* The v1 map text of a cell grid (host; world_builder.py:83-88: tokens joined by ' ', rows by '\n'). Returns the length
 * needed (without the terminator) in *len; writes at most cap bytes including the terminator. */
LLE_API int lle_gen_cells_to_text(const uint8_t* cells_host, int32_t height, int32_t width, char* out, size_t cap, size_t* len);

#ifdef __cplusplus
}
#endif
#endif /* LLE_B200_H */
