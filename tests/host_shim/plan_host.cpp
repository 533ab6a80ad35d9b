// TEST INFRASTRUCTURE: a host (g++) build of the planning core (lle_b200/csrc/plan_core.cuh is __host__ __device__) — the
// same limits check (plan_prepare), the same per-state step and key (PlanWorld over TinyWorld) and the same search rules as
// lle_plan_kernel, one claim after the other — so that `-m "not gpu"` tests can compare it with an independent search over
// the oracle, and GPU tests can compare the device planner with it byte for byte.  The maps are compiled by the product's own
// host map compiler.  The product never loads this file.
#include <cstdint>
#include <cstring>
#include <string>

#include "../../lle_b200/csrc/map_compiler.hpp"
#include "../../lle_b200/csrc/plan_core.cuh"

extern "C" {

// length i32[n], n_states i64[n], actions i8[n][max_steps][4] (filled with -1 here).  Returns 0 or an LLE_* status with the
// message in err.
int plan_host(const char** texts, int n, int max_steps, int all_gems, int32_t* length, int64_t* n_states, int8_t* actions, char* err,
              int errlen) {
    auto fail = [&](int code, const std::string& why) {
        if (err && errlen > 0) {
            std::strncpy(err, why.c_str(), (size_t)errlen - 1);
            err[errlen - 1] = 0;
        }
        return code;
    };
    if (max_steps < 1 || max_steps > LLE_PLAN_MAX_STEPS) return fail(LLE_INVALID_ARGUMENT, "max_steps must be in [1, 1024]");
    std::memset(actions, 0xFF, (size_t)n * (size_t)max_steps * 4);
    for (int m = 0; m < n; ++m) {
        lle::CompiledMap cm;
        try {
            cm = lle::compile_map(texts[m]);
        } catch (const lle::MapError& e) {
            return fail(e.status, "map " + std::to_string(m) + ": " + e.what());
        }
        lle::PlanSpec s;
        const char* why = "";
        const int rc = lle::plan_prepare(cm.blob.data(), all_gems != 0, s, &why);
        if (rc != LLE_OK) return fail(rc, "map " + std::to_string(m) + ": " + why);
        int8_t* act = actions + (size_t)m * (size_t)max_steps * 4;
        lle::PlanResult r;
        switch (s.A) {
            case 1: r = lle::plan_map_host<1>(cm.blob.data(), s, max_steps, act); break;
            case 2: r = lle::plan_map_host<2>(cm.blob.data(), s, max_steps, act); break;
            case 3: r = lle::plan_map_host<3>(cm.blob.data(), s, max_steps, act); break;
            default: r = lle::plan_map_host<4>(cm.blob.data(), s, max_steps, act); break;
        }
        length[m] = r.length;
        n_states[m] = r.n_states;
    }
    return 0;
}

}  // extern "C"
