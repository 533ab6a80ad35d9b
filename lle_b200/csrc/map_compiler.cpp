#include "map_compiler.hpp"

#include <algorithm>
#include <cctype>
#include <cstring>
#include <functional>
#include <sstream>

namespace lle {
namespace {

struct Token {
    char kind;  // '.', 'G', '@', 'X', 'V', 'S', 'L'
    int id;     // agent id for S / L
    int dir;    // 0 N, 1 E, 2 S, 3 W for L
};

// Rust's `str::parse::<usize>()`: ASCII digits with an optional leading '+'
bool parse_usize(const std::string& s, int& out) {
    size_t k = (!s.empty() && s[0] == '+') ? 1 : 0;
    if (k >= s.size()) return false;
    long v = 0;
    for (; k < s.size(); ++k) {
        if (s[k] < '0' || s[k] > '9') return false;
        v = v * 10 + (s[k] - '0');
        if (v > 1000000) return false;
    }
    out = (int)v;
    return true;
}

const int DI[4] = {-1, 0, 1, 0};  // N E S W (direction.rs:20-27)
const int DJ[4] = {0, 1, 0, -1};

size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

}  // namespace

// ---- v1 grammar (parser_v1.rs:132-175): lines, trimmed, blank lines skipped, whitespace-separated tokens
RawConfig parse_v1_config(const std::string& text) {
    RawConfig rc;
    std::vector<std::vector<Token>> rows;
    {
        std::istringstream lines(text);
        std::string line;
        int width = -1;
        std::vector<Cell> first_start;
        while (std::getline(lines, line)) {
            std::istringstream toks(line);
            std::string t;
            std::vector<Token> row;
            while (toks >> t) {
                Token tok{(char)std::toupper((unsigned char)t[0]), -1, -1};
                switch (tok.kind) {
                    case '.': case 'G': case '@': case 'X': case 'V': break;
                    case 'S': {
                        if (!parse_usize(t.substr(1), tok.id))
                            throw MapError(LLE_PARSE_INVALID_AGENT_ID, "InvalidAgentId { given_agent_id: \"" + t.substr(1) + "\" }");
                        // a second start for the same agent is an error at the token (parser_v1.rs:27-44)
                        if ((int)first_start.size() <= tok.id) first_start.resize(tok.id + 1, Cell{-1, -1});
                        Cell here{(int)rows.size(), (int)row.size()};
                        if (first_start[tok.id].i >= 0)
                            throw MapError(LLE_PARSE_DUPLICATE_START,
                                           "DuplicateStartTile { agent_id: " + std::to_string(tok.id) + ", start1: (" +
                                               std::to_string(first_start[tok.id].i) + ", " + std::to_string(first_start[tok.id].j) +
                                               "), start2: (" + std::to_string(here.i) + ", " + std::to_string(here.j) + ") }");
                        first_start[tok.id] = here;
                        break;
                    }
                    case 'L': {
                        switch (std::tolower((unsigned char)t.back())) {
                            case 'n': tok.dir = 0; break;
                            case 'e': tok.dir = 1; break;
                            case 's': tok.dir = 2; break;
                            case 'w': tok.dir = 3; break;
                            default:  // the reference unwraps the direction and panics (laser_config.rs:20)
                                throw MapError(LLE_PARSE_INVALID_DIRECTION, "InvalidDirection { given: \"" + t + "\" }");
                        }
                        std::string id = t.size() >= 2 ? t.substr(1, t.size() - 2) : std::string();
                        if (!parse_usize(id, tok.id))
                            throw MapError(LLE_PARSE_INVALID_AGENT_ID, "InvalidAgentId { given_agent_id: \"" + id + "\" }");
                        break;
                    }
                    default:
                        throw MapError(LLE_PARSE_INVALID_TILE, "InvalidTile { tile_str: \"" + t + "\", line: " +
                                                                  std::to_string(rows.size()) + ", col: " + std::to_string(row.size()) + " }");
                }
                row.push_back(tok);
            }
            if (row.empty()) continue;
            if (width < 0) width = (int)row.size();
            if ((int)row.size() != width)
                throw MapError(LLE_PARSE_INCONSISTENT_DIMENSIONS,
                               "InconsistentDimensions { expected_n_cols: " + std::to_string(width) + ", actual_n_cols: " +
                                   std::to_string(row.size()) + ", row: " + std::to_string(rows.size()) + " }");
            rows.push_back(std::move(row));
        }
    }
    if (rows.empty()) throw MapError(LLE_PARSE_EMPTY_WORLD, "EmptyWorld");
    rc.H = (int)rows.size();
    rc.W = (int)rows[0].size();
    // ---- row-major collection (parser_v1.rs:147-161)
    for (int i = 0; i < rc.H; ++i) {
        for (int j = 0; j < rc.W; ++j) {
            const Token& t = rows[i][j];
            Cell c{i, j};
            switch (t.kind) {
                case 'G': rc.gems.push_back(c); break;
                case '@': rc.walls.push_back(c); break;
                case 'X': rc.exits.push_back(c); break;
                case 'V': rc.voids.push_back(c); break;
                case 'S':
                    if ((int)rc.starts.size() <= t.id) rc.starts.resize(t.id + 1);
                    rc.starts[t.id].push_back(c);
                    break;
                case 'L':
                    rc.sources.push_back(RawSource{c, t.id, t.dir, (int)rc.sources.size()});
                    rc.walls.push_back(c);  // a source is also a wall (parser_v1.rs:22-25)
                    break;
                default: break;
            }
        }
    }
    return rc;
}

// parsing::parse (src/core/parsing/mod.rs:14-21): TOML (v2) first, the v1 grammar when the text is not a v2 document
RawConfig parse_config(const std::string& text) {
    RawConfig rc;
    if (parse_toml_config(text, rc)) return rc;
    return parse_v1_config(text);
}

CompiledMap compile_map(const std::string& text, const ObsSpec& spec, const std::vector<SourceState>* source_state,
                        const std::vector<Cell>* new_exits) {
    if (spec.kind < LLE_OBS_LAYERED || spec.kind > LLE_OBS_STATE) throw MapError(LLE_INVALID_ARGUMENT, "unknown observation kind");
    if (spec.kind == LLE_OBS_LAYERED && (spec.param < 0 || spec.param > 64)) throw MapError(LLE_INVALID_ARGUMENT, "padding_size out of range");
    if (spec.kind == LLE_OBS_PARTIAL && (spec.param < 1 || spec.param % 2 != 1 || spec.param > 31))
        throw MapError(LLE_INVALID_ARGUMENT, "Can only use odd numbers for the square size");  // observations.py:299
    CompiledMap cm;
    cm.text = text;
    const RawConfig rc = parse_config(text);
    const int H = rc.H, W = rc.W;
    cm.gems = rc.gems; cm.walls = rc.walls; cm.exits = rc.exits; cm.voids = rc.voids;
    std::vector<std::vector<Cell>> starts = rc.starts;  // candidate starts per agent (exactly one in v1)
    for (const auto& s : rc.sources) cm.sources.push_back(SourceInfo{s.pos, s.colour, s.direction, s.laser_id, 0, true});
    for (const auto* lst : {&cm.gems, &cm.walls, &cm.exits, &cm.voids})
        for (const auto& c : *lst)
            if (c.i < 0 || c.j < 0 || c.i >= H || c.j >= W) throw MapError(LLE_PARSE_POSITION_OUT_OF_BOUNDS, "PositionOutOfBounds");
    // ---- pre_validate (world_config.rs:124-148)
    const int A = (int)starts.size();
    if (A == 0) throw MapError(LLE_PARSE_NO_AGENTS, "NoAgents");
    if ((int)cm.exits.size() < A)
        throw MapError(LLE_PARSE_NOT_ENOUGH_EXITS, "NotEnoughExitTiles { n_starts: " + std::to_string(A) +
                                                       ", n_exits: " + std::to_string(cm.exits.size()) + " }");

    // a [[lasers]] position is not bounds-checked by the reference's parser: it indexes its grid with it after pre_validate and
    // panics (world_config.rs:247); here the document is refused at the same point
    for (const auto& s : cm.sources)
        if (s.pos.i < 0 || s.pos.j < 0 || s.pos.i >= H || s.pos.j >= W) throw MapError(LLE_PARSE_POSITION_OUT_OF_BOUNDS, "PositionOutOfBounds");

    if (new_exits) {  // World::set_exit_positions (world.rs:195-234)
        if ((int)new_exits->size() < A)
            throw MapError(LLE_PARSE_NOT_ENOUGH_EXITS, "NotEnoughExitTiles { n_starts: " + std::to_string(A) +
                                                           ", n_exits: " + std::to_string(new_exits->size()) + " }");
        for (const auto& c : *new_exits) {
            if (c.i < 0 || c.j < 0 || c.i >= H || c.j >= W) throw MapError(LLE_INDEX_ERROR, "exit position out of the world");
            auto in = [&](const std::vector<Cell>& lst) { return std::find(lst.begin(), lst.end(), c) != lst.end(); };
            bool is_source = false;
            for (const auto& src : cm.sources) is_source = is_source || src.pos == c;
            if (in(cm.gems) || in(cm.voids) || in(cm.walls) || is_source)  // the reference panics: "Tile is not a floor"
                throw MapError(LLE_INVALID_ARGUMENT, "an exit can only be placed on a floor tile");
        }
        cm.exits = *new_exits;
    }
    // ---- base tile plane (world_config.rs:176-199)
    std::vector<uint16_t> tiles((size_t)H * W, LLE_T_FLOOR);
    for (size_t g = 0; g < cm.gems.size(); ++g) tiles[cm.gems[g].i * W + cm.gems[g].j] = (uint16_t)(LLE_T_GEM | (g << 8));
    for (auto& c : cm.exits) tiles[c.i * W + c.j] = LLE_T_EXIT;
    for (auto& c : cm.voids) tiles[c.i * W + c.j] = LLE_T_VOID;
    for (auto& c : cm.walls) tiles[c.i * W + c.j] = LLE_T_WALL;
    // two [[lasers]] entries on one cell: the reference writes the second source tile over the first (world_config.rs:247) and
    // lists the surviving source twice, with the first beam's laser tiles orphaned
    for (size_t a = 0; a < cm.sources.size(); ++a)
        for (size_t b = a + 1; b < cm.sources.size(); ++b)
            if (cm.sources[a].pos == cm.sources[b].pos) throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: two laser sources on one cell");
    // ---- beams and start pruning (world_config.rs:203-250), sources in list order.  A beam walks while the tile is
    // walkable: it stops at walls and at the sources placed before it (the source tile is written after its beam, :247).
    std::vector<std::vector<std::pair<int, int>>> cell_beams((size_t)H * W);  // (beam index, offset), inner first
    std::vector<char> placed((size_t)H * W, 0);
    for (int b = 0; b < (int)cm.sources.size(); ++b) {
        auto& s = cm.sources[b];
        int i = s.pos.i + DI[s.direction], j = s.pos.j + DJ[s.direction];
        std::vector<Cell> cells;
        while (i >= 0 && j >= 0 && i < H && j < W && (tiles[i * W + j] & 7u) != LLE_T_WALL && !placed[i * W + j]) {
            cells.push_back(Cell{i, j});
            i += DI[s.direction];
            j += DJ[s.direction];
        }
        for (int later = b + 1; later < (int)cm.sources.size(); ++later)
            if (std::find(cells.begin(), cells.end(), cm.sources[later].pos) != cells.end())
                // only possible with TOML [[lasers]] outside the wall list: the reference lets the earlier beam run through the
                // cell and then overwrites its laser tile with the source, leaving `lasers_positions` inconsistent
                throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: a laser source sits on the beam of an earlier source");
        s.len = (int)cells.size();
        bool shielded = false;  // `is_blocked`: from the owner's single start on, the beam is cut at reset
        for (int k = 0; k < s.len; ++k) {
            const Cell c = cells[k];
            if (s.colour < A && starts[s.colour].size() == 1 && starts[s.colour][0] == c) shielded = true;
            if (!shielded)
                for (int a = 0; a < A; ++a)
                    if (a != s.colour) starts[a].erase(std::remove(starts[a].begin(), starts[a].end(), c), starts[a].end());
            cell_beams[c.i * W + c.j].push_back({b, k});
        }
        placed[s.pos.i * W + s.pos.j] = 1;
    }
    for (const auto& s : cm.sources) tiles[s.pos.i * W + s.pos.j] = LLE_T_WALL;  // Tile::LaserSource is not walkable (tile.rs:63-73)
    // A gem position overwritten by an exit, a void, a wall or a laser source (only possible in TOML documents): the reference keeps the
    // position in `gems_positions`, so World::gems / get_state reach `unreachable!()` (world.rs:129-139) - the world is unusable
    for (auto& c : cm.gems)
        if ((tiles[c.i * W + c.j] & 7u) != LLE_T_GEM)
            throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: a gem position is also an exit, void, wall or laser source cell (World::gems panics there in the reference)");
    if (new_exits)
        for (const auto& c : *new_exits)
            if (cell_beams[c.i * W + c.j].size() > 1)  // the reference's set_tile would drop the inner beam's tile there
                throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: an exit cannot be placed where two beams cross");
    // A start candidate on a laser source (only possible with TOML [[lasers]]): World::reset panics in the reference as soon as
    // that candidate is drawn ("The agent should be able to pre-enter", world.rs:424-427) - refused here
    for (int a = 0; a < A; ++a)
        for (const auto& c : starts[a])
            for (const auto& src : cm.sources)
                if (c == src.pos) throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: a start position coincides with a laser source");
    // ---- post_validate (world_config.rs:150-170)
    for (int a = 0; a < A; ++a)
        if (starts[a].empty())
            throw MapError(LLE_PARSE_AGENT_WITHOUT_START, "AgentWithoutStart { agent_id: " + std::to_string(a) + " }");
    bool random_starts = false;
    for (int a = 0; a < A; ++a) {
        random_starts = random_starts || starts[a].size() != 1;
        cm.starts.push_back(starts[a][0]);
    }
    cm.start_candidates = starts;
    if (!random_starts)  // every agent has one start: two agents sharing it make sample_different panic (utils/mod.rs:80-84)
        for (int a = 0; a < A; ++a)
            for (int b = a + 1; b < A; ++b)
                if (starts[a][0] == starts[b][0]) throw MapError(LLE_PARSE_NOT_ENOUGH_STARTS, "Could not assign positions to agents");
    // sample_different (src/utils/mod.rs:39-86) visits the agents by increasing number of candidates (stable sort)
    std::vector<int> order(A);
    for (int a = 0; a < A; ++a) order[a] = a;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return starts[x].size() < starts[y].size(); });
    if (random_starts) {
        // a complete assignment of distinct starts must exist (the reference panics at the first reset otherwise): augmenting paths
        std::vector<int> owner((size_t)H * W, -1);
        std::function<bool(int, std::vector<char>&)> place = [&](int a, std::vector<char>& seen) {
            for (const auto& c : starts[a]) {
                const int cell = c.i * W + c.j;
                if (seen[cell]) continue;
                seen[cell] = 1;
                if (owner[cell] < 0 || place(owner[cell], seen)) { owner[cell] = a; return true; }
            }
            return false;
        };
        for (int a = 0; a < A; ++a) {
            std::vector<char> seen((size_t)H * W, 0);
            if (!place(a, seen)) throw MapError(LLE_PARSE_NOT_ENOUGH_STARTS, "Could not assign positions to agents");
        }
        for (int cell = 0; cell < H * W; ++cell)  // the device's last resort when its sampling attempts all dead-end
            if (owner[cell] >= 0) cm.starts[owner[cell]] = Cell{cell / W, cell % W};
    }
    // duplicated gem positions make World::gems() report one tile twice; the device format indexes gems by cell
    for (size_t g = 0; g < cm.gems.size(); ++g)
        for (size_t g2 = g + 1; g2 < cm.gems.size(); ++g2)
            if (cm.gems[g] == cm.gems[g2]) throw MapError(LLE_PARSE_UNSUPPORTED, "Unsupported: a gem position is listed twice");

    // ---- device-format limits
    const int G = (int)cm.gems.size(), NB = (int)cm.sources.size();
    if (A > LLE_MAX_AGENTS || G > LLE_MAX_GEMS || NB > LLE_MAX_BEAMS || H > 256 || W > 256)
        throw MapError(LLE_LIMIT_EXCEEDED, "map exceeds the device format (agents<=32, gems<=64, sources<=64, H,W<=256)");
    for (auto& s : cm.sources) {
        if (s.len > LLE_MAX_BEAM_LEN) throw MapError(LLE_LIMIT_EXCEEDED, "beam longer than 64 cells");
        if (s.colour > 254) throw MapError(LLE_LIMIT_EXCEEDED, "laser colour above 254");
        cm.max_beam_len = std::max(cm.max_beam_len, s.len);
    }
    cm.H = H; cm.W = W; cm.A = A; cm.G = G; cm.NB = NB;
    if (source_state) {  // mutated after construction: colours and enabled flags as they are now
        if ((int)source_state->size() != NB) throw MapError(LLE_INVALID_ARGUMENT, "source state does not match the map");
        for (int b = 0; b < NB; ++b) {
            if ((*source_state)[b].colour < 0 || (*source_state)[b].colour > 254) throw MapError(LLE_LIMIT_EXCEEDED, "laser colour out of range");
            cm.sources[b].colour = (*source_state)[b].colour;
            cm.sources[b].enabled = (*source_state)[b].enabled;
        }
    }
    // channel layout (observations.py:199-211): the agent count of the layout includes the padding budget
    const int Ap = A + (spec.kind == LLE_OBS_LAYERED ? spec.param : 0);
    const int C = 2 * Ap + 4;
    cm.C = C;
    const int LASER_0 = Ap, WALL = 2 * Ap, VOID = WALL + 1, GEM = WALL + 2, EXIT = WALL + 3, HW = H * W;

    // ---- lasers listing: the outermost laser of a cell and the one directly under it (world.rs:159-172)
    std::vector<uint64_t> vis(NB, 0);
    for (int c = 0; c < HW; ++c) {
        auto& lst = cell_beams[c];
        if (lst.empty()) continue;
        cm.laser_cells.push_back(Cell{c / W, c % W});
        for (int n = 0; n < 2 && n < (int)lst.size(); ++n) {
            auto [b, k] = lst[lst.size() - 1 - n];  // later source wraps earlier ones (world_config.rs:233-245)
            vis[b] |= 1ull << k;
            cm.lasers.push_back(LaserTileInfo{Cell{c / W, c % W}, b, cm.sources[b].colour, cm.sources[b].direction, b, k});
        }
    }

    // ---- layered static plane (observations.py:216-237): wall, void, exit, then sources = -1
    std::vector<float> stat((size_t)C * HW, 0.0f);
    bool obs_invalid = false;
    for (auto& c : cm.walls) stat[(size_t)WALL * HW + c.i * W + c.j] = 1.0f;
    for (auto& c : cm.voids) stat[(size_t)VOID * HW + c.i * W + c.j] = 1.0f;
    for (auto& c : cm.exits) stat[(size_t)EXIT * HW + c.i * W + c.j] = 1.0f;
    for (auto& s : cm.sources) {
        int ch = LASER_0 + s.colour;
        if (ch >= C) { obs_invalid = true; continue; }  // numpy IndexError in the reference
        stat[(size_t)ch * HW + s.pos.i * W + s.pos.j] = -1.0f;
    }
    // ---- dynamic cells (observations.py:256-263)
    std::vector<LlePatch> patch;
    for (auto& l : cm.lasers) {
        int ch = LASER_0 + l.colour;
        if (ch >= C) { obs_invalid = true; continue; }
        uint32_t idx = (uint32_t)(ch * HW + l.pos.i * W + l.pos.j);
        patch.push_back(LlePatch{idx, (uint8_t)l.beam, (uint8_t)l.offset, (int8_t)stat[idx], 0});
    }
    for (int g = 0; g < G; ++g) {
        uint32_t idx = (uint32_t)(GEM * HW + cm.gems[g].i * W + cm.gems[g].j);
        patch.push_back(LlePatch{idx, 0xFF, (uint8_t)g, (int8_t)stat[idx], 0});
    }
    std::vector<LleAgentPlane> planes;
    for (int a = 0; a < A; ++a) planes.push_back(LleAgentPlane{(uint32_t)(a * HW), (uint32_t)a});
    int obs_floats = C * HW, view_agents = Ap, obs_c = C, obs_h = H, obs_w = W;
    if (spec.kind == LLE_OBS_PERSPECTIVE) {
        // AgentZeroPerspective (observations.py:381-395): copy n of the layered block with the agent planes 0 <-> n and
        // the laser planes 0 <-> n exchanged.  The block of one env is the A copies back to back, so the static plane,
        // the patch table and the agent-plane table are replicated per copy with the permuted channel.
        auto perm = [&](int n, int ch) {  // destination channel of source channel `ch` in copy n
            if (ch == 0) return n;
            if (ch == n) return 0;
            if (ch == LASER_0) return LASER_0 + n;
            if (ch == LASER_0 + n) return LASER_0;
            return ch;
        };
        std::vector<float> all((size_t)A * C * HW, 0.0f);
        std::vector<LlePatch> all_patch;
        planes.clear();
        for (int n = 0; n < A; ++n) {
            for (int ch = 0; ch < C; ++ch)
                std::memcpy(&all[((size_t)n * C + perm(n, ch)) * HW], &stat[(size_t)ch * HW], (size_t)HW * sizeof(float));
            for (const auto& pe : patch) {
                LlePatch q = pe;
                q.idx = (uint32_t)(((size_t)n * C + perm(n, (int)(pe.idx / HW))) * HW + pe.idx % HW);
                all_patch.push_back(q);
            }
            for (int a = 0; a < A; ++a) planes.push_back(LleAgentPlane{(uint32_t)(((size_t)n * C + perm(n, a)) * HW), (uint32_t)a});
        }
        stat.swap(all);
        patch.swap(all_patch);
        obs_floats = A * C * HW;
        view_agents = 0;
    } else if (spec.kind == LLE_OBS_PARTIAL) {
        // PartialGenerator (observations.py:296-369): rendered cell by cell on the device; nothing static
        const int Cp = 2 * A + 3;
        for (auto& s : cm.sources)
            if (A + 1 + s.colour >= Cp) obs_invalid = true;  // obs[a, LASER_0 + agent_id]: numpy IndexError
        stat.assign(4, 0.0f);
        // For the feature-driven renderer (sparse maps): every cell content the generator encodes, as a patch entry with
        // idx = packed position | channel << 16, stat = the value, src = LLE_FEATURE_STATIC / 0xFF (gem) / beam index.
        // All writes commute: equal values or distinct (channel, cell) targets.
        patch.clear();
        auto feature = [&](const Cell& c, int channel, int value, int src, int bit) {
            if (channel < Cp)
                patch.push_back(LlePatch{(uint32_t)((c.i << 8) | c.j) | ((uint32_t)channel << 16), (uint8_t)src, (uint8_t)bit, (int8_t)value, 0});
        };
        for (const auto& c : cm.walls) feature(c, A, 1, LLE_FEATURE_STATIC, 0);                       // WALL = n_agents
        for (const auto& c : cm.exits) feature(c, 2 * A + 2, 1, LLE_FEATURE_STATIC, 0);               // EXIT
        for (const auto& sinfo : cm.sources) feature(sinfo.pos, A + 1 + sinfo.colour, -1, LLE_FEATURE_STATIC, 0);
        for (int g = 0; g < G; ++g) feature(cm.gems[g], 2 * A + 1, 1, 0xFF, g);                        // GEM, while not collected
        for (const auto& l : cm.lasers) feature(l.pos, A + 1 + l.colour, 1, l.beam, l.offset);       // listed laser tiles, while on
        planes.clear();
        obs_floats = A * Cp * spec.param * spec.param;
        view_agents = 0;
        obs_c = Cp; obs_h = obs_w = spec.param;
    } else if (spec.kind == LLE_OBS_STATE) {
        stat.assign(4, 0.0f);
        patch.clear();
        planes.clear();
        obs_invalid = false;
        obs_floats = 3 * A + G;
        view_agents = A;
        obs_c = obs_floats; obs_h = obs_w = 0;
    }
    std::stable_sort(patch.begin(), patch.end(), [](const LlePatch& x, const LlePatch& y) { return x.idx < y.idx; });
    // The render list of the tiny-map kernel: the non-zero floats of the static plane (src = LLE_FEATURE_STATIC, stat = the
    // value), then a copy of the dynamic entries above.  A tiny tile is zero-filled and this list is applied to it.
    std::vector<LlePatch> static_list;
    int n_static = 0;
    if (spec.kind == LLE_OBS_LAYERED) {
        for (size_t k = 0; k < stat.size(); ++k)
            if (stat[k] != 0.0f) static_list.push_back(LlePatch{(uint32_t)k, LLE_FEATURE_STATIC, 0, (int8_t)stat[k], 0});
        n_static = (int)static_list.size();
        static_list.insert(static_list.end(), patch.begin(), patch.end());
    }

    // ---- blob
    LleMapHeader h;
    std::memset(&h, 0, sizeof h);
    h.H = H; h.W = W; h.A = A; h.G = G; h.NB = NB; h.C = C;
    h.n_patch = (int)patch.size();
    h.obs_floats = obs_floats;
    h.obs_invalid = obs_invalid;
    h.obs_kind = spec.kind; h.obs_param = spec.param; h.view_agents = view_agents;
    h.obs_c = obs_c; h.obs_h = obs_h; h.obs_w = obs_w;
    h.n_ap = (int)planes.size();
    size_t off = align16(sizeof(LleMapHeader));
    h.tiles_off = (uint32_t)off;   off = align16(off + tiles.size() * sizeof(uint16_t));
    h.cellinfo_off = (uint32_t)off;  off = align16(off + (size_t)HW * sizeof(uint32_t));
    h.cellbeams_off = (uint32_t)off; off = align16(off + (size_t)HW * sizeof(LleCellBeams));
    h.beams_off = (uint32_t)off;   off = align16(off + (size_t)std::max(NB, 1) * sizeof(LleBeam));
    h.patch_off = (uint32_t)off;   off = align16(off + std::max<size_t>(patch.size(), 1) * sizeof(LlePatch));
    // An int8 observation (obs_dtype) takes its static plane as bytes, zero-padded to the row stride (a multiple of 16): every
    // 16-byte piece of a row is then one asynchronous copy from the plane.
    const bool i8 = spec.dtype == LLE_DTYPE_I8;
    std::vector<int8_t> stat_i8;
    if (i8) {
        stat_i8.assign(((size_t)obs_floats + 15) / 16 * 16, 0);
        for (size_t k = 0; k < stat.size() && k < stat_i8.size(); ++k) stat_i8[k] = (int8_t)stat[k];
    }
    h.obs_dtype = spec.dtype;
    h.static_off = (uint32_t)off;  off = align16(off + (i8 ? stat_i8.size() : stat.size() * sizeof(float)));
    h.ap_off = (uint32_t)off;      off = align16(off + std::max<size_t>(planes.size(), 1) * sizeof(LleAgentPlane));
    h.n_static = n_static;
    h.static_list_off = (uint32_t)off; off = align16(off + std::max<size_t>(static_list.size(), 1) * sizeof(LlePatch));
    // start candidates (World.random_start_positions): per agent (first index, count), then the packed positions
    std::vector<uint32_t> cand_index;
    std::vector<uint16_t> cand_pos;
    for (int a = 0; a < A; ++a) {
        cand_index.push_back((uint32_t)cand_pos.size());
        cand_index.push_back((uint32_t)starts[a].size());
        for (const auto& c : starts[a]) cand_pos.push_back((uint16_t)((c.i << 8) | c.j));
    }
    h.random_starts = random_starts ? 1 : 0;
    h.cand_index_off = (uint32_t)off; off = align16(off + cand_index.size() * sizeof(uint32_t));
    h.cand_pos_off = (uint32_t)off;   off = align16(off + std::max<size_t>(cand_pos.size(), 1) * sizeof(uint16_t));
    for (int a = 0; a < A; ++a) h.start_order[a] = (uint8_t)order[a];
    std::vector<uint32_t> chunk_tbl;  // patches are sorted by idx: chunk c owns entries [tbl[c], tbl[c+1])
    {
        // the vec pads a block to 16 bytes (obs_stride): 4 floats or 16 int8 elements
        const int per16 = i8 ? 16 : 4;
        const int64_t block = ((int64_t)obs_floats + per16 - 1) / per16 * per16;
        const int chunk = lle_chunk_elems(block, i8 ? 1 : 4);
        const int n_chunks = (int)((block + chunk - 1) / chunk);
        size_t k = 0;
        for (int c = 0; c <= n_chunks; ++c) {
            while (k < patch.size() && patch[k].idx < (uint32_t)c * (uint32_t)chunk) ++k;
            chunk_tbl.push_back((uint32_t)k);
        }
    }
    h.chunk_tbl_off = (uint32_t)off; off = align16(off + chunk_tbl.size() * sizeof(uint32_t));
    h.blob_bytes = (uint32_t)off;
    h.gem_toplevel = 0;
    for (int g = 0; g < G; ++g) {
        h.gem_pos[g] = (uint16_t)((cm.gems[g].i << 8) | cm.gems[g].j);
        if (cell_beams[cm.gems[g].i * W + cm.gems[g].j].empty()) h.gem_toplevel |= 1ull << g;
    }
    for (int a = 0; a < A; ++a) h.start[a] = (uint16_t)((cm.starts[a].i << 8) | cm.starts[a].j);

    cm.blob.assign(off, 0);
    std::memcpy(cm.blob.data(), &h, sizeof h);
    std::memcpy(cm.blob.data() + h.tiles_off, tiles.data(), tiles.size() * sizeof(uint16_t));
    for (int b = 0; b < NB; ++b) {
        const auto& s = cm.sources[b];
        LleBeam bm;
        std::memset(&bm, 0, sizeof bm);
        bm.vis = vis[b];
        bm.first_i = (uint16_t)(s.pos.i + DI[s.direction]);
        bm.first_j = (uint16_t)(s.pos.j + DJ[s.direction]);
        bm.di = (int8_t)DI[s.direction];
        bm.dj = (int8_t)DJ[s.direction];
        bm.len = (uint8_t)s.len;
        bm.colour = (uint8_t)s.colour;
        bm.enabled = s.enabled ? 1 : 0;
        bm.src_i = (uint8_t)s.pos.i;
        bm.src_j = (uint8_t)s.pos.j;
        std::memcpy(cm.blob.data() + h.beams_off + b * sizeof(LleBeam), &bm, sizeof bm);
    }
    // per-cell lookup tables
    {
        std::vector<uint32_t> info((size_t)HW, 0);
        std::vector<LleCellBeams> cb((size_t)HW);
        const int adi[4] = {-1, 1, 0, 0}, adj[4] = {0, 0, 1, -1};  // Action deltas N, S, E, W (action.rs:18-26)
        for (int i = 0; i < H; ++i) {
            for (int j = 0; j < W; ++j) {
                const int c = i * W + j;
                uint32_t nbr = 0;
                for (int act = 0; act < 4; ++act) {
                    int ti = i + adi[act], tj = j + adj[act];
                    if (ti >= 0 && tj >= 0 && ti < H && tj < W && (tiles[ti * W + tj] & 7u) != LLE_T_WALL) nbr |= 1u << act;
                }
                info[c] = (tiles[c] & 7u) | (nbr << 3) | ((uint32_t)(tiles[c] >> 8) << 8);
                for (const auto& src : cm.sources)
                    if (src.pos.i == i && src.pos.j == j) info[c] |= (1u << 7) | ((uint32_t)src.colour << 16);
                for (int n = 0; n < 4; ++n) cb[c].e[n] = LLE_NO_BEAM;
                if (std::find(cm.walls.begin(), cm.walls.end(), Cell{i, j}) != cm.walls.end()) info[c] |= 1u << 25;
                const auto& lst = cell_beams[c];
                if (!lst.empty()) info[c] |= 1u << 24;
                if (lst.size() > 4) throw MapError(LLE_LIMIT_EXCEEDED, "more than four beams cross one cell");
                for (size_t n = 0; n < lst.size(); ++n) {
                    const int b = lst[n].first, k = lst[n].second;
                    const auto& src = cm.sources[b];
                    const uint32_t listed = (vis[b] >> k) & 1ull;
                    cb[c].e[n] = (uint32_t)b | ((uint32_t)k << 6) | ((uint32_t)src.colour << 12) | ((uint32_t)src.len << 20) |
                                 ((src.enabled ? 1u : 0u) << 27) | (listed << 28);
                }
            }
        }
        std::memcpy(cm.blob.data() + h.cellinfo_off, info.data(), info.size() * sizeof(uint32_t));
        std::memcpy(cm.blob.data() + h.cellbeams_off, cb.data(), cb.size() * sizeof(LleCellBeams));
    }
    if (!patch.empty()) std::memcpy(cm.blob.data() + h.patch_off, patch.data(), patch.size() * sizeof(LlePatch));
    if (!static_list.empty()) std::memcpy(cm.blob.data() + h.static_list_off, static_list.data(), static_list.size() * sizeof(LlePatch));
    if (i8) std::memcpy(cm.blob.data() + h.static_off, stat_i8.data(), stat_i8.size());
    else std::memcpy(cm.blob.data() + h.static_off, stat.data(), stat.size() * sizeof(float));
    std::memcpy(cm.blob.data() + h.chunk_tbl_off, chunk_tbl.data(), chunk_tbl.size() * sizeof(uint32_t));
    std::memcpy(cm.blob.data() + h.cand_index_off, cand_index.data(), cand_index.size() * sizeof(uint32_t));
    if (!cand_pos.empty()) std::memcpy(cm.blob.data() + h.cand_pos_off, cand_pos.data(), cand_pos.size() * sizeof(uint16_t));
    if (!planes.empty()) std::memcpy(cm.blob.data() + h.ap_off, planes.data(), planes.size() * sizeof(LleAgentPlane));
    return cm;
}

}  // namespace lle
