// Host map compiler: v1 map text -> immutable device tables (static_map.h).
//
// It restates, table-first, what the reference does when it builds a `World` from a string:
//   grammar                    src/core/parsing/parser_v1.rs:132-175, laser_config.rs:19-35
//   validation                 src/core/parsing/world_config.rs:124-170
//   tile plane                 src/core/parsing/world_config.rs:176-199 (Floor, then gems, exits, voids, walls)
//   beams + start pruning      src/core/parsing/world_config.rs:203-250
//   layered static planes      python/lle/observations.py:216-237
//   lasers listing (outer two) src/core/world.rs:159-172
// Instead of wrapping tiles in nested `Laser` objects it records, per source, the beam's first cell,
// direction and length, and per map a "patch table" of the observation cells that depend on state.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/lle_b200.h"
#include "static_map.h"

namespace lle {

// status codes: the LLE_* enum of include/lle_b200.h

struct MapError : std::runtime_error {
    int status;
    MapError(int s, const std::string& msg) : std::runtime_error(msg), status(s) {}
};

struct Cell {
    int i, j;
    bool operator==(const Cell& o) const { return i == o.i && j == o.j; }
};

struct SourceInfo {
    Cell pos;
    int colour, direction /* 0 N, 1 E, 2 S, 3 W */, laser_id, len;
    bool enabled;
};

struct LaserTileInfo {  // one entry of World::lasers() (outer two per cell), in row-major cell order
    Cell pos;
    int laser_id, colour, direction, beam, offset;
};

// What both map grammars produce before the world is built (WorldConfig, src/core/parsing/world_config.rs:12-22)
struct RawSource {
    Cell pos;
    int colour, direction /* 0 N, 1 E, 2 S, 3 W */, laser_id;
};
struct RawConfig {
    int H = 0, W = 0;
    std::vector<Cell> gems, voids, exits, walls;
    std::vector<std::vector<Cell>> starts;  // candidate start positions per agent
    std::vector<RawSource> sources;
};
RawConfig parse_v1_config(const std::string& text);
// TOML v2 (src/core/parsing/toml/*.rs).  Returns false when the text is not a v2 document (ParseError::NotV2: the caller
// falls back to v1, parsing/mod.rs:14-21); throws MapError for v2 documents that are invalid.
bool parse_toml_config(const std::string& text, RawConfig& out);

struct CompiledMap {
    std::string text;
    int H = 0, W = 0, A = 0, G = 0, NB = 0, C = 0;
    std::vector<Cell> walls, voids, exits, gems, starts, laser_cells;
    std::vector<std::vector<Cell>> start_candidates;  // World.random_start_positions (after the laser pruning)
    std::vector<SourceInfo> sources;
    std::vector<LaserTileInfo> lasers;
    int max_beam_len = 0;
    std::vector<uint8_t> blob;  // LleMapHeader + tables, ready for HBM
    const LleMapHeader& header() const { return *reinterpret_cast<const LleMapHeader*>(blob.data()); }
};

// Which observation the device tables are laid out for (static_map.h: LLE_OBS_*)
struct ObsSpec {
    int kind = LLE_OBS_LAYERED;
    int param = 0;
    int dtype = LLE_DTYPE_F32;  // element type of the static plane (LLE_DTYPE_I8: int8_t, for layered / perspective only)
    bool operator==(const ObsSpec& o) const { return kind == o.kind && param == o.param && dtype == o.dtype; }
};

// State of a laser source after the world was built: LaserBeam::{set_agent_id, enable, disable} (src/core/tiles/laser.rs:69-84).
// The start pruning of laser_setup (world_config.rs:225-243) is a build-time step and keeps using the colours of the text.
struct SourceState {
    int colour;
    bool enabled;
};

// `exits`: World::set_exit_positions (src/core/world.rs:195-234) applied after the build — the exits of the text become
// floor tiles and these cells (plain floor, start or former exit cells crossed by at most one beam) become the exits.
CompiledMap compile_map(const std::string& text, const ObsSpec& spec = ObsSpec(), const std::vector<SourceState>* sources = nullptr,
                        const std::vector<Cell>* exits = nullptr);

}  // namespace lle
