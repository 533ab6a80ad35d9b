// TEST INFRASTRUCTURE: a host (g++) build of the expert core (lle_b200/csrc/expert_core.cuh is __host__ __device__) — the same
// limits check (plan_prepare), the same per-state step and key (PlanWorld over TinyWorld) and the same forward enumeration and
// backward levels as the device build in expert.cu, one item after the other — so that `-m "not gpu"` tests can compare it with
// an independent computation over the oracle, and GPU tests can compare the device tables with it byte for byte.  The maps are
// compiled by the product's own host map compiler.  The product never loads this file.
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../lle_b200/csrc/map_compiler.hpp"
#include "../../lle_b200/csrc/expert_core.cuh"

namespace {
std::vector<uint32_t> g_table;  // the words of the last expert_host_build
lle::PlanSpec g_spec;
}  // namespace

extern "C" {

// Builds the table of one map.  *n_keys receives K, *n_states the size of the reached set.  Returns 0 or an LLE_* status with
// the message in err.
int expert_host_build(const char* text, int all_gems, int64_t* n_keys, int64_t* n_states, char* err, int errlen) {
    auto fail = [&](int code, const std::string& why) {
        if (err && errlen > 0) {
            std::strncpy(err, why.c_str(), (size_t)errlen - 1);
            err[errlen - 1] = 0;
        }
        return code;
    };
    lle::CompiledMap cm;
    try {
        cm = lle::compile_map(text);
    } catch (const lle::MapError& e) {
        return fail(e.status, e.what());
    }
    const char* why = "";
    const int rc = lle::plan_prepare(cm.blob.data(), all_gems != 0, g_spec, &why);
    if (rc != LLE_OK) return fail(rc, why);
    switch (g_spec.A) {
        case 1: *n_states = lle::expert_map_host<1>(cm.blob.data(), g_spec, g_table); break;
        case 2: *n_states = lle::expert_map_host<2>(cm.blob.data(), g_spec, g_table); break;
        case 3: *n_states = lle::expert_map_host<3>(cm.blob.data(), g_spec, g_table); break;
        default: *n_states = lle::expert_map_host<4>(cm.blob.data(), g_spec, g_table); break;
    }
    *n_keys = g_spec.K;
    return 0;
}

// The last build's table in the API's form (lle_vec_expert_table): dist i32[K], joint i16[K]; and the map's cell index table
// (u16[H*W], 0xFFFF off the standable cells) with its number of standable cells.
void expert_host_fetch(int32_t* dist, int16_t* joint, uint16_t* cell_index, int32_t* n_cells) {
    lle::expert_decode(g_table.data(), (int64_t)g_table.size(), dist, joint);
    if (cell_index) std::memcpy(cell_index, g_spec.cell_index.data(), g_spec.cell_index.size() * 2);
    if (n_cells) *n_cells = g_spec.n_cells;
}

}  // extern "C"
