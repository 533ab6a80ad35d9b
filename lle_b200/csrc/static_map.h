// Static (per-map) tables and the dynamic per-env record shared by the host map compiler and the
// sm_100a kernels.  Everything here is plain-old-data so it can be memcpy'd to HBM verbatim.
//
// Reference concepts (paths relative to the reference repository):
//   base tile plane   <- WorldConfig::make_grid            src/core/parsing/world_config.rs:176-199
//   beams             <- WorldConfig::laser_setup          src/core/parsing/world_config.rs:203-250
//   LaserBeam state   <- `beam: RefCell<Vec<bool>>`        src/core/tiles/laser.rs:15-21   (here: one u64 mask)
//   layered channels  <- LayeredPadded.__init__/_setup     python/lle/observations.py:199-237
#pragma once
#include <stdint.h>

#include "../../include/lle_b200.h"

#define LLE_MAX_AGENTS 32  // alive/arrived/slot are u32 masks
#define LLE_MAX_BEAMS 64   // per map
#define LLE_MAX_GEMS 64    // one u64 collected mask
#define LLE_MAX_BEAM_LEN 64

// base tile kinds (low 3 bits of a tile word; gem index in bits 8..15)
enum : uint16_t { LLE_T_FLOOR = 0, LLE_T_WALL = 1, LLE_T_GEM = 2, LLE_T_EXIT = 3, LLE_T_VOID = 4 };

// One laser source and its beam.  Cell k of the beam is (first_i + k*di, first_j + k*dj), k < len.
struct LleBeam {
    uint64_t vis;      // bit k set <=> this beam's laser tile at cell k is listed by World::lasers()
                       //   (only the two outermost lasers of a nested cell are, world.rs:159-172)
    uint16_t first_i, first_j;
    int8_t di, dj;
    uint8_t len;       // 0..64 (0: the source faces a wall or the border)
    uint8_t colour;    // agent id that blocks the beam; may be >= n_agents (world_config.rs:137-145)
    uint8_t enabled;   // LaserBeam::is_enabled
    uint8_t src_i, src_j;
    uint8_t pad[5];
};
static_assert(sizeof(LleBeam) == 24, "LleBeam layout");

// One dynamic cell of the layered observation other than the agents' own cells: a laser tile
// (1.0 while its beam bit is on) or a gem (1.0 until collected).  `idx` is the float index inside
// one env's (C,H,W) block; `stat` is what the static plane holds there (restored when the bit is off).
#define LLE_FEATURE_STATIC 0xFD  // LlePatch.src of a partial-observation feature that does not depend on state
struct LlePatch {
    uint32_t idx;
    uint8_t src;   // beam index, or 0xFF for a gem
    uint8_t bit;   // offset k in the beam, or gem index
    int8_t stat;   // -1, 0, 1
    uint8_t pad;
};
static_assert(sizeof(LlePatch) == 8, "LlePatch layout");

// Observation kinds: LLE_OBS_* of include/lle_b200.h (ObservationType.get_observation_generator, observations.py:66-97)

// Where agent `agent`'s one-hot cell goes in an env's observation block: float index base + i*W + j.
// Layered: A entries (agent a -> plane a).  Perspective: A*A entries (copy n draws agent a in plane perm_n(a)).
struct LleAgentPlane {
    uint32_t base;
    uint32_t agent;
};

// Per-cell lookup tables used by the step kernel (one load each instead of a scan over all beams):
//   cellinfo[cell]  : bits 0-2 base tile kind | bits 3-6 walkable-neighbour mask indexed by Action value
//                     (N, S, E, W: in bounds and neither Wall nor LaserSource, tile.rs:63-73) | bit 7: the cell is a
//                     laser source | bits 8-15 gem index | bits 16-23 colour of the source (bit 7 set) | bit 24: a beam crosses the cell
//                     | bit 25: the cell is in World::walls() (every wall; sources too, except TOML [[lasers]] outside `walls`)
//   cellbeams[cell] : the (at most four: one per direction of travel) beams crossing the cell, inner first.
//                     entry = b (0-5) | k<<6 (6-11) | colour<<12 (12-19) | len<<20 (20-26) | enabled<<27 | listed<<28
//                     (listed: the laser tile is one of the two reported by World::lasers(), world.rs:159-172);
//                     0xFFFFFFFF = no entry.
#define LLE_NO_BEAM 0xFFFFFFFFu
// Observation blocks larger than a shared-memory tile are streamed in chunks of this many floats (12 KB).  The map
// blob carries, per chunk, the first patch entry (sorted by float index) that falls into it.
#define LLE_CHUNK_FLOATS 3072
#ifdef __cplusplus
// Chunks are balanced: a block of n floats is cut into ceil(n / 3072) chunks of (nearly) equal length, so the last bulk
// store of a block is about as large as the others (perspective level 6: 3 x 9,984 B instead of 2 x 12 KB + 5 KB).  The
// length is a multiple of 32 floats: chunk boundaries stay on 128-byte lines (3,036-float chunks on a 64x64 map, whose
// boundaries split a line between two bulk stores, measured 6 % slower than 3,072).
// Only done when the last 3,072-float chunk would be less than half full (on a 64x64 map, 26 x 12 KB + 8 KB, equal
// chunks of 3,040 floats were 1 % slower).
// An int8 block is cut by the same byte budget: chunks of up to 12,288 elements on 128-byte lines.
static inline int lle_chunk_elems(int64_t block, int elem_bytes) {
    const int64_t max_len = LLE_CHUNK_FLOATS * 4 / elem_bytes, line = 128 / elem_bytes;
    const int64_t rest = block % max_len;
    if (rest == 0 || rest >= max_len / 2) return (int)max_len;
    const int64_t n = (block + max_len - 1) / max_len;
    const int64_t len = (block + n - 1) / n;
    return (int)((len + line - 1) / line * line);
}
static inline int lle_chunk_floats(int64_t block_floats) { return lle_chunk_elems(block_floats, 4); }
#endif
struct LleCellBeams {
    uint32_t e[4];
};

// Per-map header; all *_off are byte offsets from the start of the map blob (16-byte aligned).
struct LleMapHeader {
    int32_t H, W, A, G, NB, C;
    int32_t n_patch;
    int32_t obs_floats;       // C*H*W (elements, whatever the element type)
    uint32_t tiles_off;       // uint16_t[H*W]
    uint32_t cellinfo_off;    // uint32_t[H*W]
    uint32_t cellbeams_off;   // LleCellBeams[H*W]
    uint32_t beams_off;       // LleBeam[NB]
    uint32_t patch_off;       // LlePatch[n_patch]
    uint32_t static_off;      // float[C*H*W], or int8_t[C*H*W rounded up to 16] for an int8 observation (obs_dtype)
    uint32_t blob_bytes;
    uint32_t obs_invalid;     // some LASER_0+colour >= C: the reference raises IndexError (observations.py:235)
    uint64_t gem_toplevel;    // bit g set <=> gem g is NOT wrapped by a laser (world.rs:265-275, :550-554)
    int32_t obs_kind, obs_param;   // LLE_OBS_* and its parameter
    int32_t view_agents;           // layered / state: agent copies of the stride-0 view (A + padding); else 0 (materialised)
    int32_t obs_c, obs_h, obs_w;   // shape of ONE agent's observation (state: obs_c = length, obs_h = obs_w = 0)
    int32_t n_ap;                  // entries of the agent-plane table
    uint32_t ap_off;               // LleAgentPlane[n_ap]
    uint32_t chunk_tbl_off;        // uint32_t[n_chunks + 1]: patch index range of every chunk of lle_chunk_elems(padded block) elements
    int32_t n_static;              // layered observations: non-zero floats of the static plane, listed at static_list_off
    int32_t random_starts;         // some agent has several start candidates: World::reset samples (world.rs:421)
    uint32_t cand_index_off;       // uint32_t[2*A]: first index and count of each agent's candidates in cand_pos
    uint32_t cand_pos_off;         // uint16_t[]: packed candidate positions, sorted like AgentConfig::compute_start_positions
    uint32_t static_list_off;      // LlePatch[n_static + n_patch]: the static floats (idx, stat = value), then a copy of the patch table
    uint8_t start_order[LLE_MAX_AGENTS];  // agents by increasing number of candidates (stable), the order sample_different assigns them
    uint16_t start[LLE_MAX_AGENTS];   // packed position (i<<8 | j); with random starts: the first candidate
    uint16_t gem_pos[LLE_MAX_GEMS];   // packed position, gems_positions order (parser_v1.rs:149)
    int32_t obs_dtype;                // LLE_DTYPE_*: element type of the static plane and of the observation rows
    int32_t pad_dtype;
};

// ---- dynamic per-env record: `stride` 32-bit words per environment, stored contiguously (array of
// records): a warp owns one world at a time and moves its record with one coalesced transaction.
//   [0, w_flags)        packed positions (i<<8 | j), two per word
//   [w_flags, w_gems)   A <= 8: alive | arrived<<8 | slot<<16 | n_arrived<<24 (4 bits) | n_deads<<28 (3 bits, saturating)
//                       | done<<31 ; else four words: alive, arrived, slot, n_arrived | n_deads<<8 | done<<16
//   [w_avail, w_gems)   World::available_actions cache (world.rs:37): one byte per agent, bit = Action value
//   [w_gems, w_on)      collected mask (0, 1 or 2 words)
//   [w_on, w_sube)      beam on-masks (LaserBeam.beam, laser.rs:16): 1 word per beam when every beam of the
//                       batch is <= 32 cells, else 2
//   [w_sube, w_subp)    LaserSubgoal flags (extras_generators.py:91): per agent, one bit per source (sub_words words)
//   [w_subp, n_words)   PotentialShapedLLE._agents_pos_reached (reward_strategy.py:140), same shape
struct LleStateLayout {
    int32_t n_words, w_flags, w_avail, w_gems, w_on;
    int32_t gem_words, on_words;  // words of the gem mask (0/1/2), words per beam (1/2)
    int32_t wide_flags;           // A > 8
    int32_t stride;               // n_words rounded up to 4 words (16 bytes)
    int32_t w_sube, w_subp, sub_words;  // sub_words: words per agent of a subgoal mask (0 when the feature is off)
    int32_t pad;
};

#ifdef __cplusplus
static inline LleStateLayout lle_state_layout(int A, int G, int NB, int max_beam_len, int extras = 0, int pbrs = 0) {
    LleStateLayout L;
    L.wide_flags = A > 8;
    L.w_flags = (A + 1) / 2;
    L.w_avail = L.w_flags + (L.wide_flags ? 4 : 1);
    L.w_gems = L.w_avail + (A + 3) / 4;
    L.gem_words = G == 0 ? 0 : (G <= 32 ? 1 : 2);
    L.w_on = L.w_gems + L.gem_words;
    L.on_words = max_beam_len <= 32 ? 1 : 2;
    L.sub_words = (extras || pbrs) ? (NB <= 32 ? 1 : 2) : 0;
    L.w_sube = L.w_on + NB * L.on_words;
    L.w_subp = L.w_sube + (extras ? A * L.sub_words : 0);
    L.n_words = L.w_subp + (pbrs ? A * L.sub_words : 0);
    L.stride = (L.n_words + 3) / 4 * 4;
    L.pad = 0;
    return L;
}
#endif
