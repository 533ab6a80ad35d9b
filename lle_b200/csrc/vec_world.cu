// lle_b200 — host side of the C ABI (include/lle_b200.h): map handles, device buffers, launch
// configuration and the kernel launches.  The kernel itself lives in world_kernel.cuh.
#include <cuda.h>  // types of the stream memory operations only; the entry points are resolved at run time
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/lle_b200.h"
#include "levels_embedded.inc"
#include "map_compiler.hpp"
#include "world_kernel.cuh"
#include "tiny_kernel.cuh"

namespace lle {

// ---------------------------------------------------------------------------------------- host side
thread_local std::string g_error;
int fail(int code, const std::string& msg) { g_error = msg; return code; }

#define LLE_CUDA(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t _e = (expr);                                                                           \
        if (_e != cudaSuccess)                                                                             \
            return fail(_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver ? LLE_NO_DEVICE : LLE_CUDA_ERROR, \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                               \
    } while (0)

using KernelFn = void (*)(KParams);  // every instantiation of lle_world_kernel and lle_tiny_step_kernel

}  // namespace lle

using namespace lle;

struct lle_map {
    CompiledMap cm;
};

struct lle_vec {
    lle_vec_options opts;
    // LLE(state_type=...): a second vec over the SAME engine records (and map indices), created for the state's observation
    // type; it never steps, it only re-exports (lle_vec_refresh) after every launch of this one
    lle_vec* shadow = nullptr;
    bool borrows_records = false;  // this vec is somebody's shadow: records / map indices belong to the owner
    int device = 0;
    int64_t N = 0, N_pad = 0;
    int A = 0, G = 0, NBmax = 0, C = 0, H = 0, W = 0, S = 0, R = 1, max_beam_len = 0;
    LleStateLayout L;
    // device memory
    std::vector<CompiledMap> own_maps;  // maps recompiled for a non-default observation type
    // laser sources can be recoloured / switched after creation (lle_vec_set_source): what is needed to recompile a map
    std::vector<std::string> map_texts;
    std::vector<std::vector<SourceState>> src_state;
    std::vector<int> map_patches, map_obs_invalid;
    std::vector<uint64_t> map_gem_toplevel;  // per map: gems that are top-level Gem tiles (not wrapped by a laser tile)
    std::vector<std::vector<Cell>> map_exits;  // World::set_exit_positions overrides (empty: the exits of the text)
    std::vector<char> map_exits_set;
    std::vector<uint8_t*> retired_blobs;
    // LLE(randomize_lasers=True): every map is compiled once per colouring (variant index = sum colour_b * A^b)
    bool randomize = false, creating = false;
    int n_variants = 1;
    std::vector<CompiledMap> variant_maps;  // [n_maps * n_variants]
    bool render = true;
    LleMapHeader hdr0;  // header of the first map (observation shape)
    int obs_invalid = 0;
    std::vector<uint8_t*> d_blobs;
    const uint8_t** d_blob_table = nullptr;
    int32_t* d_map_of_env = nullptr;
    uint32_t* d_records = nullptr;
    float* d_obs = nullptr;
    int8_t* d_obs_i8 = nullptr;  // obs_dtype LLE_DTYPE_I8: the observation rows (d_obs stays null)
    bool i8 = false;             // the observation is rendered in int8 (the kernels' OT = int8_t)
    float* d_state = nullptr;
    uint8_t* d_avail = nullptr;
    float* d_reward = nullptr;
    uint8_t* d_done = nullptr;
    uint8_t* d_events = nullptr;
    int8_t* d_actions = nullptr;
    uint8_t* d_err = nullptr;
    uint32_t* d_sched = nullptr;        // kSchedSlots x {next pair, warps finished}
    uint32_t* d_flags = nullptr;        // [n_tickets] last completed step sequence number per ticket
    uint32_t reset_epoch = 0;           // explicit resets so far (start-sampling counter word, random starts)
    uint32_t seq = 0;                   // sequence number of the last step launched
    uint32_t launch_index = 0;          // rotates the scheduler slots
    bool last_was_step = false;         // the previous launch on this vec was a step (may be overlapped via PDL)
    int8_t* d_actions_stage = nullptr;  // for step_host
    uint64_t* d_timeline = nullptr;     // development aid (LLE_B200_TIMELINE=1)
    float* d_extras = nullptr;          // [N_pad][A][JE]
    uint8_t* d_info = nullptr;          // episode_stats: Step.info bytes and the episode accumulators
    float *d_ep_return = nullptr, *d_last_return = nullptr;
    int32_t *d_ep_length = nullptr, *d_last_length = nullptr;
    int JE = 0;
    uint64_t extras_set = 0, pbrs_set = 0;
    int8_t extras_beam[64] = {0};
    int64_t obs_stride = 0;
    // launch configuration
    bool fast = false, pdl = true;
    int feature_limit = 0;
    bool by_feature = false;  // partial observations rendered feature by feature (kernel KIND 2): every map has <= 2 s^2 features
    // tiny maps: step launches run the thread-per-world kernel (tiny_kernel.cuh) with its own tiling and grid
    bool tiny = false, tiny_partial = false;
    int tiny_E = 8, tiny_warp_smem = 0, tiny_grid = 0;
    size_t tiny_smem = 0;
    // the instantiations this vec launches (select_kernels): step, step of a parts loop, reset, set_state, tiny step (or null)
    KernelFn k_step = nullptr, k_step_parts = nullptr, k_reset = nullptr, k_set_state = nullptr, k_tiny = nullptr;
    uint32_t* h_retired_seq = nullptr;  // pinned, device-mapped: [0] sequence number of the last step launch that retired,
                                        // [32] number of launches of this vec (any mode) whose last warp has left
    uint32_t* d_retired_count = nullptr;  // device counter behind [32]
    MapDev map0;                        // the tables of map 0 as device pointers (kernel parameter of single-map batches)
    bool has_map0 = false;
    bool narrow_next = false;  // the next step launch finds its predecessor still running: use the narrow grid
    int grid = 0, grid_step = 0, grid_idle = 0, Wd = 32, group = 4, E = 1, n_chunks = 1, chunk_floats = 0, tile_floats = 0, n_buf = 1, warp_smem = 0;
    size_t smem = 0;
    uint64_t t = 0, launches = 0;
    // timing
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint64_t timing_launches0 = 0;
    // pipelined host stepping (lle_vec_pipeline_submit / _wait): three streams, a ring of staging slots
    static constexpr int kPipeSlots = 8;
    bool pipe_ready = false;
    cudaStream_t s_in = nullptr, s_main = nullptr, last_stream = nullptr;
    cudaEvent_t ev_user = nullptr;
    int8_t* d_stage[kPipeSlots] = {};
    uint32_t* d_pipe_flags = nullptr;  // [0] actions of submit n have landed (written by the copy stream)
    uint32_t* h_out_flags = nullptr;   // pinned + mapped, one word per ring slot: submit n has retired and its results are in host memory
    uint32_t* d_out_flags = nullptr;   // the same words as the device sees them
    uint64_t pipe_submitted = 0, pipe_completed = 0;
    // closed loop over parts of the batch (lle_vec_parts_*)
    int parts_n = 0;                    // > 0: a parts loop is open
    uint32_t parts_tpp = 0;             // tickets per part
    uint64_t parts_launched = 0;        // whole-batch steps enqueued in this loop
    std::vector<uint64_t> parts_fed, parts_read;  // per part: steps whose actions were released / whose results were waited for
    uint32_t* d_part_in = nullptr;      // device: [parts][32] steps fed (written by stream memory ops on s_in)
    uint32_t* h_part_out = nullptr;     // pinned + mapped: [parts][32] steps whose reward / done are in host memory
    uint32_t* d_part_out = nullptr;     // the same words as the device sees them
    uint32_t* d_part_count = nullptr;   // device: [parts] tickets of the part completed in the running step
    int parts_cap = 0;
    const int8_t* parts_actions_dev = nullptr;  // device views of the caller's pinned buffers
    float* parts_reward = nullptr;
    uint8_t* parts_done = nullptr;
    const void* pinned_seen[32] = {};  // host pointers already checked to be page-locked ...
    void* pinned_dev[32] = {};         // ... and the address the device reaches them at
    unsigned pinned_next = 0;
};

namespace {

// Scheduler slots rotate over the launches of a vec.  Any number of (small) launches can be resident at once through
// programmatic dependent launch, so a slot carries a generation word and a launch waits on the device until the launch that
// used its slot before has re-armed it (world_kernel.cuh: sched_slot_armed).  One 128-byte line per slot.
constexpr int kSchedSlots = 8;
constexpr int kSchedSlotWords = 32;

// The kernels a vec launches: the one place that names an instantiation of lle_world_kernel or lle_tiny_step_kernel.
// KIND 1 (FAST) for the common layered shape, KIND 2 (the feature-driven renderer) for partial observations of sparse maps, KIND 0
// for everything else; a parts loop has its own step instantiations.  Partial observations are float only: no int8 KIND 2 or
// PARTIAL tiny kernel.  The thread-per-world step kernel (tiny_kernel.cuh) has one instantiation per agent count.
void select_kernels(lle_vec* v) {
    auto world = [v](KernelFn step, KernelFn step_parts, KernelFn reset, KernelFn set_state) {
        v->k_step = step;
        v->k_step_parts = step_parts;
        v->k_reset = reset;
        v->k_set_state = set_state;
    };
    if (v->i8 && v->fast)
        world(lle_world_kernel<MODE_STEP, 1, false, int8_t>, lle_world_kernel<MODE_STEP, 1, true, int8_t>,
              lle_world_kernel<MODE_RESET, 1, false, int8_t>, lle_world_kernel<MODE_SET_STATE, 1, false, int8_t>);
    else if (v->i8)
        world(lle_world_kernel<MODE_STEP, 0, false, int8_t>, lle_world_kernel<MODE_STEP, 0, true, int8_t>,
              lle_world_kernel<MODE_RESET, 0, false, int8_t>, lle_world_kernel<MODE_SET_STATE, 0, false, int8_t>);
    else if (v->fast)
        world(lle_world_kernel<MODE_STEP, 1>, lle_world_kernel<MODE_STEP, 1, true>, lle_world_kernel<MODE_RESET, 1>,
              lle_world_kernel<MODE_SET_STATE, 1>);
    else if (v->by_feature)
        world(lle_world_kernel<MODE_STEP, 2>, lle_world_kernel<MODE_STEP, 2, true>, lle_world_kernel<MODE_RESET, 2>,
              lle_world_kernel<MODE_SET_STATE, 2>);
    else
        world(lle_world_kernel<MODE_STEP, 0>, lle_world_kernel<MODE_STEP, 0, true>, lle_world_kernel<MODE_RESET, 0>,
              lle_world_kernel<MODE_SET_STATE, 0>);
    static const KernelFn tiny[3][4] = {  // [float / float PARTIAL / int8][A - 1]
        {lle_tiny_step_kernel<1>, lle_tiny_step_kernel<2>, lle_tiny_step_kernel<3>, lle_tiny_step_kernel<4>},
        {lle_tiny_step_kernel<1, true>, lle_tiny_step_kernel<2, true>, lle_tiny_step_kernel<3, true>, lle_tiny_step_kernel<4, true>},
        {lle_tiny_step_kernel<1, false, int8_t>, lle_tiny_step_kernel<2, false, int8_t>, lle_tiny_step_kernel<3, false, int8_t>,
         lle_tiny_step_kernel<4, false, int8_t>},
    };
    v->k_tiny = v->tiny ? tiny[v->i8 ? 2 : v->tiny_partial ? 1 : 0][std::min(v->A, 4) - 1] : nullptr;
}

cudaError_t launch_mode(lle_vec* v, KParams& p, cudaStream_t s) {
    const bool step = p.mode == MODE_STEP;
    // Programmatic stream serialization: the kernel calls griddepcontrol.wait before it touches anything a
    // previous launch wrote, so its prologue may overlap the tail of the launch before it.
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof cfg);
    // A single step that may overlap its predecessor runs on a narrow grid (grid_step CTAs), so that several consecutive
    // step launches are resident at once and form a software pipeline over the epoch flags: while step t drains, steps
    // t+1.. already stream their first tickets.  Rollouts, resets and set_state use the full-width grid.
    const bool overlaps = v->pdl && step && v->last_was_step && v->last_stream == s;
    // (A parts loop takes the full grid too: its launches wait for the host part by part, and a wide grid keeps enough unblocked
    // warps resident.  Level 6 x 65,536, 8 parts, us per step with 2 / 3 / 5 CTAs per SM: 96.9 / 87.8 / 84.5.)
    // A single step that finds the device idle takes four CTAs per SM of the five, which leaves room for the first CTAs of the
    // launch that follows it (the driver's 20-step window after a sync, idle launch at 5 / 4 / 3 / 2 CTAs per SM: 79.8 / 78.7 /
    // 78.8 / 78.9 us per step).
    const int grid = (step && p.n_steps == 1 && !p.part_in) ? ((overlaps && v->narrow_next) ? v->grid_step : v->grid_idle) : v->grid;
    v->narrow_next = false;
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    p.n_warps_total = (uint32_t)(grid * kWarps);
    cfg.dynamicSmemBytes = v->smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    // only a step that directly follows a step may overlap it: the epoch flags order them ticket by ticket
    attr[0].val.programmaticStreamSerializationAllowed = overlaps ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    KernelFn kern = step ? (p.part_in ? v->k_step_parts : v->k_step) : p.mode == MODE_RESET ? v->k_reset : v->k_set_state;
    if (step && v->tiny && !p.part_in) {  // thread-per-world kernel: same tickets, flags and records, its own tile layout (not in a parts loop)
        kern = v->k_tiny;
        cfg.gridDim = dim3((unsigned)v->tiny_grid);
        cfg.dynamicSmemBytes = v->tiny_smem;
        p.n_warps_total = (uint32_t)(v->tiny_grid * kWarps);
        p.E = v->tiny_E;
        p.tile_floats = (int32_t)(v->tiny_E * v->obs_stride);
        p.warp_smem_bytes = v->tiny_warp_smem;
    }
    return cudaLaunchKernelEx(&cfg, kern, p);
}
// Host bookkeeping (launch index, sequence number, "the last launch was a step") advances only when the launch was accepted.
cudaError_t launch(lle_vec* v, KParams& p, cudaStream_t s) {
    p.sched = v->d_sched + kSchedSlotWords * (v->launch_index % kSchedSlots);
    p.sched_gen = v->launch_index / kSchedSlots;
    // every launch issued so far has retired (a closed loop, synchronous stepping): the slot is certainly re-armed
    p.sched_check = *(volatile uint32_t*)(v->h_retired_seq + 32) != v->launch_index ? 1u : 0u;
    p.retired_launch = v->h_retired_seq + 32;
    p.retired_count = v->d_retired_count;
    p.map0 = v->map0;
    p.has_map0 = v->has_map0 ? 1 : 0;
    p.flags = v->d_flags;
    cudaError_t e;
    switch (p.mode) {
        case MODE_STEP:
            p.seq = v->seq + 1;  // sequence number of the first step of this launch
            p.retired_seq = v->h_retired_seq;
            // Narrow-grid software pipelining: a step that finds its predecessor still in flight runs on a grid of
            // `grid_step` CTAs (two per SM for large observations), so that two or three consecutive launches are resident at once
            // and the next step's prologue and first tickets overlap this step's tail.  A step that finds the device idle
            // (synchronous stepping, a policy between two steps) takes the full-width grid: alone, a narrow launch cannot
            // saturate HBM.  Measured on B200, level 6 x 65,536, us/step in windows of 20 / 2,000 launches after a sync, CTAs per
            // SM 1 / 2 / 3 / 5: 81.6 / 79.4 / 80.6 / 83.6 and 75.6 / 76.3 / 78.6 / 82.3 (profiles/grid_sweep_r02.jsonl).
            v->narrow_next = (int32_t)(v->seq - *(volatile uint32_t*)v->h_retired_seq) >= 1;
            e = launch_mode(v, p, s);
            if (e != cudaSuccess) return e;
            v->launch_index++;
            v->seq += (uint32_t)p.n_steps;
            v->last_was_step = true;
            v->last_stream = s;
            return e;
        default: e = launch_mode(v, p, s); break;
    }
    if (e != cudaSuccess) return e;
    v->launch_index++;
    v->last_was_step = false;
    v->last_stream = s;
    return e;
}

// Stream memory operations of the driver API, resolved through the runtime so that the library carries no link-time
// dependency on libcuda (it must load on a machine without a driver for the build / ABI checks).
typedef CUresult (*StreamValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
StreamValue32Fn g_write_value32 = nullptr, g_wait_value32 = nullptr;
cudaError_t resolve_memops() {
    if (g_write_value32 && g_wait_value32) return cudaSuccess;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuStreamWriteValue32", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess) return e;
    if (q != cudaDriverEntryPointSuccess || !fn) return cudaErrorNotSupported;
    g_write_value32 = (StreamValue32Fn)fn;
    e = cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess) return e;
    if (q != cudaDriverEntryPointSuccess || !fn) return cudaErrorNotSupported;
    g_wait_value32 = (StreamValue32Fn)fn;
    return cudaSuccess;
}

// The dynamic shared-memory limit is an attribute of the FUNCTION, shared by every vec of the process: it is raised to the
// device's opt-in maximum (227 KB on B200) once, never to one vec's own size — a second vec with a smaller tile would otherwise
// lower it under the first one's launches.
int g_smem_optin = 0;
cudaError_t smem_optin(int device, int* out) {
    if (!g_smem_optin) {
        cudaError_t e = cudaDeviceGetAttribute(&g_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (e != cudaSuccess) return e;
    }
    *out = g_smem_optin;
    return cudaSuccess;
}

// Raises the kernel's dynamic shared-memory limit to the opt-in maximum and lowers *blocks (< 0: not set yet) to the CTAs per SM
// it reaches with `smem` bytes each
cudaError_t configure_kernel(KernelFn kern, size_t smem, int* blocks) {
    int dev = 0, optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = smem_optin(dev, &optin);
    if (e == cudaSuccess && smem > (size_t)optin) return cudaErrorInvalidValue;
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e != cudaSuccess) return e;
    int b = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, kThreads, smem);
    if (e == cudaSuccess && (*blocks < 0 || b < *blocks)) *blocks = b;
    return e;
}

int env_int(const char* name, int fallback) {
    const char* v = std::getenv(name);
    return v && *v ? std::atoi(v) : fallback;
}

// MapDev::bind on the host: the device addresses of a map's tables from the device address of its blob and a host copy of its header
MapDev host_bind(const uint8_t* dblob, const LleMapHeader& h) {
    MapDev m;
    m.blob = dblob;
    m.hdr = reinterpret_cast<const LleMapHeader*>(dblob);
    m.cellinfo = reinterpret_cast<const uint32_t*>(dblob + h.cellinfo_off);
    m.cellbeams = reinterpret_cast<const LleCellBeams*>(dblob + h.cellbeams_off);
    m.beams = reinterpret_cast<const LleBeam*>(dblob + h.beams_off);
    m.patches = reinterpret_cast<const LlePatch*>(dblob + h.patch_off);
    m.stat = reinterpret_cast<const float*>(dblob + h.static_off);
    m.agent_planes = reinterpret_cast<const LleAgentPlane*>(dblob + h.ap_off);
    m.n_ap = h.n_ap;
    m.chunk_tbl = reinterpret_cast<const uint32_t*>(dblob + h.chunk_tbl_off);
    m.n_patch = h.n_patch;
    m.NB = h.NB;
    m.obs_floats = h.obs_floats;
    m.gem_toplevel = h.gem_toplevel;
    return m;
}

KParams base_params(lle_vec* v) {
    KParams p;
    std::memset(&p, 0, sizeof p);
    p.blobs = v->d_blob_table;
    p.map_of_env = v->d_map_of_env;
    p.records = v->d_records;
    p.L = v->L;
    p.N = v->N;
    p.N_pad = v->N_pad;
    p.A = v->A; p.G = v->G; p.NBmax = v->NBmax; p.C = v->C; p.H = v->H; p.W = v->W; p.S = v->S; p.R = v->R;
    p.HW = v->H * v->W;
    p.obs = v->d_obs; p.obs_i8 = v->d_obs_i8; p.obs_stride = v->obs_stride;
    p.state = v->d_state; p.avail = v->d_avail; p.reward = v->d_reward; p.done = v->d_done;
    p.events = v->d_events; p.actions = v->d_actions; p.err = v->d_err;
    p.seed = v->opts.seed; p.env_id_base = v->opts.env_id_base; p.t = v->t;
    p.auto_reset = v->opts.auto_reset; p.lle_semantics = v->opts.lle_semantics;
    p.walkable = v->opts.walkable_lasers; p.write_obs = v->render ? 1 : 0;
    p.obs_kind = v->opts.obs_type; p.obs_param = v->opts.obs_param;
    p.state_obs = (v->opts.write_obs && v->opts.obs_type == LLE_OBS_STATE) ? (v->opts.obs_param ? 2 : 1) : 0;
    p.Wd = v->Wd; p.group = v->group; p.E = v->E; p.n_chunks = v->n_chunks; p.chunk_floats = v->chunk_floats; p.tile_floats = v->tile_floats;
    p.n_buf = v->n_buf;
    p.warp_smem_bytes = v->warp_smem;
    p.n_tickets = (uint32_t)(v->N_pad / v->group);
    p.n_warps_total = (uint32_t)(v->grid * kWarps);
    p.n_steps = 1;
    p.extras = v->d_extras; p.JE = v->JE; p.pbrs_on = v->opts.pbrs ? 1 : 0;
    p.extras_set = v->extras_set; p.pbrs_set = v->pbrs_set;
    p.pbrs_gamma = v->opts.pbrs_gamma; p.pbrs_value = v->opts.pbrs_reward_value;
    std::memcpy(p.extras_beam, v->extras_beam, sizeof p.extras_beam);
    p.timeline = v->d_timeline;
    p.info = v->d_info; p.ep_return = v->d_ep_return; p.ep_length = v->d_ep_length; p.last_return = v->d_last_return; p.last_length = v->d_last_length;
    p.reset_epoch = v->reset_epoch;
    p.randomize = (v->randomize && !v->creating) ? 1 : 0;  // the construction reset is World::new's, not LLE.reset (env.py:191-203)
    p.n_variants = v->n_variants;
    return p;
}

// The device-side address of page-locked host memory (cudaHostAlloc / cudaHostRegister / lle_host_alloc / torch pin_memory), or
// nullptr when `ptr` is not page-locked.  The answers for the last few pointers are remembered: a host loop passes the same
// ring of buffers over and over.
void* device_view(lle_vec* v, const void* ptr) {
    for (int k = 0; k < 32; ++k)
        if (v->pinned_seen[k] == ptr) return v->pinned_dev[k];
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (attr.type != cudaMemoryTypeHost || !attr.devicePointer) return nullptr;
    const unsigned k = v->pinned_next++ % 32;
    v->pinned_seen[k] = ptr;
    v->pinned_dev[k] = attr.devicePointer;
    return attr.devicePointer;
}

template <class T>
cudaError_t dalloc(T** ptr, size_t count) {
    cudaError_t e = cudaMalloc((void**)ptr, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) e = cudaMemset(*ptr, 0, std::max<size_t>(count, 1) * sizeof(T));
    return e;
}

int pow2_floor(int x) { int p = 1; while (p * 2 <= x) p *= 2; return p; }

}  // namespace

namespace {
template <bool IMPORT>
int raw_state_launch(lle_vec* v, const RawState& r, void* stream) {
    LLE_CUDA(cudaSetDevice(v->device));
    const int threads = 128;
    const int blocks = (int)((v->N + threads - 1) / threads);
    lle_raw_state_kernel<IMPORT><<<blocks, threads, 0, (cudaStream_t)stream>>>(v->d_records, v->L, v->N, v->A, v->NBmax, r);
    LLE_CUDA(cudaGetLastError());
    v->launches++;
    return LLE_OK;
}
RawState raw_of(const lle_raw_state* s, int n_beams) {
    RawState r;
    r.pos = s->pos; r.alive = s->alive; r.arrived = s->arrived; r.slot = s->slot; r.beam_on = n_beams ? s->beam_on : nullptr;
    r.collected = s->collected; r.counters = s->counters; r.avail_cache = s->avail_cache;
    r.sub_extras = s->subgoals_extras; r.sub_pbrs = s->subgoals_pbrs;
    return r;
}
}  // namespace

extern "C" {

const char* lle_last_error(void) { return g_error.c_str(); }
const char* lle_version(void) { return "lle_b200 0.1 (sm_100a)"; }

int lle_map_parse(const char* text, size_t len, lle_map** out) {
    if (!text || !out) return fail(LLE_INVALID_ARGUMENT, "null argument");
    try {
        auto m = std::make_unique<lle_map>();
        m->cm = compile_map(std::string(text, len));
        *out = m.release();
        return LLE_OK;
    } catch (const MapError& e) {
        return fail(e.status, e.what());
    } catch (const std::exception& e) {
        return fail(LLE_INVALID_ARGUMENT, e.what());
    }
}

int lle_map_level(int level, lle_map** out) {
    if (level < 1 || level > 6)  // world.rs:599-606
        return fail(LLE_PARSE_INVALID_LEVEL, "InvalidLevel { asked: " + std::to_string(level) + ", min: 1, max: 6 }");
    const char* text = kEmbeddedLevels[level - 1];
    return lle_map_parse(text, std::strlen(text), out);
}

void lle_map_free(lle_map* map) { delete map; }

int lle_map_get_info(const lle_map* map, lle_map_info* out) {
    if (!map || !out) return fail(LLE_INVALID_ARGUMENT, "null argument");
    const CompiledMap& c = map->cm;
    std::memset(out, 0, sizeof *out);
    out->height = c.H; out->width = c.W; out->n_agents = c.A; out->n_gems = c.G; out->n_sources = c.NB; out->n_channels = c.C;
    out->n_exits = (int)c.exits.size(); out->n_walls = (int)c.walls.size(); out->n_voids = (int)c.voids.size();
    out->n_laser_cells = (int)c.laser_cells.size(); out->n_lasers = (int)c.lasers.size();
    out->obs_invalid = (int)c.header().obs_invalid;
    out->max_beam_len = c.max_beam_len;
    out->gem_toplevel = c.header().gem_toplevel;
    return LLE_OK;
}

int lle_map_positions(const lle_map* map, int kind, int32_t* out_ij, int32_t cap, int32_t* n) {
    if (!map || !n) return fail(LLE_INVALID_ARGUMENT, "null argument");
    const CompiledMap& c = map->cm;
    const std::vector<Cell>* v;
    switch (kind) {
        case LLE_POS_WALLS: v = &c.walls; break;
        case LLE_POS_VOIDS: v = &c.voids; break;
        case LLE_POS_EXITS: v = &c.exits; break;
        case LLE_POS_GEMS: v = &c.gems; break;
        case LLE_POS_STARTS: v = &c.starts; break;
        case LLE_POS_LASER_CELLS: v = &c.laser_cells; break;
        default: return fail(LLE_INVALID_ARGUMENT, "unknown position kind");
    }
    *n = (int32_t)v->size();
    for (int k = 0; k < (int)v->size() && k < cap && out_ij; ++k) {
        out_ij[2 * k] = (*v)[k].i;
        out_ij[2 * k + 1] = (*v)[k].j;
    }
    return LLE_OK;
}

int lle_map_start_candidates(const lle_map* map, int32_t agent, int32_t* out_ij, int32_t cap, int32_t* n) {
    if (!map || !n || agent < 0 || agent >= map->cm.A) return fail(LLE_INVALID_ARGUMENT, "bad argument");
    const auto& v = map->cm.start_candidates[(size_t)agent];
    *n = (int32_t)v.size();
    for (int k = 0; k < (int)v.size() && k < cap && out_ij; ++k) {
        out_ij[2 * k] = v[k].i;
        out_ij[2 * k + 1] = v[k].j;
    }
    return LLE_OK;
}

int lle_map_sources(const lle_map* map, int32_t* out, int32_t cap, int32_t* n) {
    if (!map || !n) return fail(LLE_INVALID_ARGUMENT, "null argument");
    const auto& s = map->cm.sources;
    *n = (int32_t)s.size();
    for (int k = 0; k < (int)s.size() && k < cap && out; ++k) {
        int32_t* o = out + 7 * k;
        o[0] = s[k].pos.i; o[1] = s[k].pos.j; o[2] = s[k].colour; o[3] = s[k].direction; o[4] = s[k].enabled; o[5] = s[k].laser_id; o[6] = s[k].len;
    }
    return LLE_OK;
}

int lle_map_lasers(const lle_map* map, int32_t* out, int32_t cap, int32_t* n) {
    if (!map || !n) return fail(LLE_INVALID_ARGUMENT, "null argument");
    const auto& l = map->cm.lasers;
    *n = (int32_t)l.size();
    for (int k = 0; k < (int)l.size() && k < cap && out; ++k) {
        int32_t* o = out + 7 * k;
        o[0] = l[k].pos.i; o[1] = l[k].pos.j; o[2] = l[k].laser_id; o[3] = l[k].colour; o[4] = l[k].direction; o[5] = l[k].beam; o[6] = l[k].offset;
    }
    return LLE_OK;
}

const char* lle_map_text(const lle_map* map) { return map ? map->cm.text.c_str() : ""; }

void lle_vec_default_options(lle_vec_options* o) {
    std::memset(o, 0, sizeof *o);
    o->device = 0; o->reward_dim = 1; o->walkable_lasers = 1; o->auto_reset = 1; o->lle_semantics = 1; o->write_obs = 1;
    o->seed = 0; o->env_id_base = 0;
    o->n_extras = 0; o->pbrs = 0; o->n_pbrs = -1; o->pbrs_gamma = 0.99; o->pbrs_reward_value = 0.5;  // Builder.pbrs defaults (builder.py:79-80)
    o->state_type = LLE_OBS_STATE; o->state_param = 0;  // ObservationType.STATE (builder.py:22)
    o->obs_dtype = LLE_DTYPE_F32;
}

int lle_vec_destroy(lle_vec* v) {
    if (!v) return LLE_OK;
    cudaSetDevice(v->device);
    if (v->parts_n) lle_vec_parts_abort(v);  // no kernel may be left waiting for actions
    if (v->shadow) lle_vec_destroy(v->shadow);
    if (v->borrows_records) { v->d_records = nullptr; v->d_map_of_env = nullptr; }
    for (auto* b : v->d_blobs) cudaFree(b);
    for (auto* b : v->retired_blobs) cudaFree(b);
    cudaFree((void*)v->d_blob_table); cudaFree(v->d_map_of_env); cudaFree(v->d_records); cudaFree(v->d_obs); cudaFree(v->d_obs_i8); cudaFree(v->d_state);
    cudaFree(v->d_avail); cudaFree(v->d_reward); cudaFree(v->d_done); cudaFree(v->d_events); cudaFree(v->d_actions);
    cudaFree(v->d_err); cudaFree(v->d_sched); cudaFree(v->d_flags); cudaFree(v->d_actions_stage); cudaFree(v->d_timeline); cudaFree(v->d_extras);
    cudaFree(v->d_info); cudaFree(v->d_ep_return); cudaFree(v->d_last_return); cudaFree(v->d_ep_length); cudaFree(v->d_last_length);
    for (int k = 0; k < lle_vec::kPipeSlots; ++k) {
        cudaFree(v->d_stage[k]);
    }
    cudaFree(v->d_pipe_flags);
    cudaFree(v->d_retired_count);
    if (v->h_out_flags) cudaFreeHost(v->h_out_flags);
    if (v->h_part_out) cudaFreeHost(v->h_part_out);
    if (v->d_part_in) cudaFree(v->d_part_in);
    if (v->d_part_count) cudaFree(v->d_part_count);
    if (v->h_retired_seq) cudaFreeHost(v->h_retired_seq);
    if (v->ev_user) cudaEventDestroy(v->ev_user);
    if (v->s_in) cudaStreamDestroy(v->s_in);
    if (v->s_main) cudaStreamDestroy(v->s_main);
    if (v->ev0) cudaEventDestroy(v->ev0);
    if (v->ev1) cudaEventDestroy(v->ev1);
    delete v;
    return LLE_OK;
}

int lle_vec_create(const lle_map* const* maps, int32_t n_maps, const int32_t* map_of_env, int64_t n_envs,
                   const lle_vec_options* opts, lle_vec** out) {
    if (!maps || n_maps < 1 || n_envs < 1 || !opts || !out) return fail(LLE_INVALID_ARGUMENT, "bad argument");
    if (opts->reward_dim != 1 && opts->reward_dim != 4) return fail(LLE_INVALID_ARGUMENT, "reward_dim must be 1 or 4");
    if (opts->obs_dtype != LLE_DTYPE_F32 && opts->obs_dtype != LLE_DTYPE_I8) return fail(LLE_INVALID_ARGUMENT, "obs_dtype must be LLE_DTYPE_F32 or LLE_DTYPE_I8");
    if (opts->obs_dtype == LLE_DTYPE_I8 && (opts->obs_type == LLE_OBS_PARTIAL || opts->obs_type == LLE_OBS_STATE))
        return fail(LLE_INVALID_ARGUMENT, "obs_dtype int8: only layered and perspective observations (partial and state are float32)");
    auto v = std::unique_ptr<lle_vec, int (*)(lle_vec*)>(new lle_vec(), lle_vec_destroy);
    v->opts = *opts;
    v->device = opts->device;
    // The caller's maps are compiled for the plain layered f32 observation; other observation types and int8 observations get
    // their own device tables (channel layout, static planes, patch and agent-plane tables) from the same map text.
    const ObsSpec spec{opts->obs_type, opts->obs_param, opts->obs_dtype};
    v->i8 = opts->obs_dtype == LLE_DTYPE_I8;
    const int64_t es = v->i8 ? 1 : 4;  // bytes per observation element
    std::vector<const CompiledMap*> cms;
    if (spec == ObsSpec()) {
        for (int k = 0; k < n_maps; ++k) cms.push_back(&maps[k]->cm);
    } else {
        try {
            for (int k = 0; k < n_maps; ++k) v->own_maps.push_back(compile_map(maps[k]->cm.text, spec));
        } catch (const MapError& e) {
            return fail(e.status, e.what());
        }
        for (auto& m : v->own_maps) cms.push_back(&m);
    }
    const CompiledMap& m0 = *cms[0];
    v->A = m0.A; v->G = m0.G; v->C = m0.C; v->H = m0.H; v->W = m0.W; v->R = opts->reward_dim;
    v->S = 3 * m0.A + m0.G;
    for (int k = 0; k < n_maps; ++k) {
        const CompiledMap& m = *cms[k];
        if (m.A != v->A || m.G != v->G || m.H != v->H || m.W != v->W)
            return fail(LLE_INVALID_ARGUMENT, "all maps of a vec must share (height, width, n_agents, n_gems)");
        v->NBmax = std::max(v->NBmax, m.NB);
        if (m.header().obs_invalid) v->obs_invalid = 1;
        v->map_texts.push_back(m.text);
        v->map_gem_toplevel.push_back(m.header().gem_toplevel);
        std::vector<SourceState> st;
        for (const auto& src : m.sources) st.push_back(SourceState{src.colour, src.enabled});
        v->src_state.push_back(st);
        v->map_patches.push_back((int)m.header().n_patch);
        v->map_obs_invalid.push_back((int)m.header().obs_invalid);
        v->map_exits.emplace_back();
        v->map_exits_set.push_back(0);
        v->max_beam_len = std::max(v->max_beam_len, m.max_beam_len);
    }
    if (map_of_env)
        for (int64_t e = 0; e < n_envs; ++e)
            if (map_of_env[e] < 0 || map_of_env[e] >= n_maps) return fail(LLE_INVALID_ARGUMENT, "map_of_env out of range");
    if (opts->randomize_lasers) {
        // env.py:198-200 recolours every source at every reset with source.set_colour(random colour), which raises when the
        // beam crosses a start position of another agent (pylaser_source.rs:121-139): such maps cannot be randomised freely
        int64_t V = 1;
        for (int b = 0; b < v->NBmax; ++b) {
            V *= v->A;
            if (V > 4096) return fail(LLE_LIMIT_EXCEEDED, "randomize_lasers: more than 4096 colourings (n_agents ^ n_sources)");
        }
        v->n_variants = (int)V;
        v->randomize = true;
        for (int k = 0; k < n_maps; ++k) {
            const CompiledMap& m = *cms[k];
            for (const auto& l : m.lasers)
                for (int a = 0; a < m.A; ++a)
                    for (const auto& st : m.start_candidates[(size_t)a])
                        if (st == l.pos)
                            return fail(LLE_INVALID_ARGUMENT, "randomize_lasers: a laser crosses a start position (set_colour would raise, pylaser_source.rs:121-139)");
            for (const auto& src : m.sources)
                if (src.colour >= m.A) return fail(LLE_INVALID_ARGUMENT, "randomize_lasers: a source colour is >= n_agents");
            for (int variant = 0; variant < v->n_variants; ++variant) {
                std::vector<SourceState> st;
                int rest = variant;
                for (int b = 0; b < m.NB; ++b) { st.push_back(SourceState{rest % v->A, true}); rest /= v->A; }
                try {
                    v->variant_maps.push_back(compile_map(m.text, spec, &st));
                } catch (const MapError& e) {
                    return fail(e.status, e.what());
                }
            }
        }
    }
    v->N = n_envs;
    v->N_pad = (n_envs + 31) / 32 * 32;
    // LaserSubgoal extras / PotentialShapedLLE source selections
    {
        auto select = [&](int n, const int32_t* src, uint64_t& set, int8_t* cols, int& count) -> int {
            set = 0; count = 0;
            if (n < 0) {
                for (int b = 0; b < v->NBmax; ++b) { set |= 1ull << b; if (cols) cols[count] = (int8_t)b; ++count; }
            } else {
                for (int k = 0; k < n && k < 64; ++k) {
                    if (src[k] < 0 || src[k] >= v->NBmax) return fail(LLE_INVALID_ARGUMENT, "laser source index out of range");
                    set |= 1ull << src[k];
                    if (cols) cols[count] = (int8_t)src[k];
                    ++count;
                }
            }
            return LLE_OK;
        };
        int dummy = 0;
        if (opts->n_extras != 0) { int rc = select(opts->n_extras, opts->extras_src, v->extras_set, v->extras_beam, v->JE); if (rc) return rc; }
        if (opts->pbrs) { int rc = select(opts->n_pbrs, opts->pbrs_src, v->pbrs_set, nullptr, dummy); if (rc) return rc; }
        if (opts->pbrs && opts->reward_dim == 4) v->R = 5;  // np.concat((reward, [potential_reward])) (reward_strategy.py:153)
    }
    v->L = lle_state_layout(v->A, v->G, v->NBmax, v->max_beam_len, v->JE > 0, opts->pbrs != 0);
    // rows are padded to 16 bytes: every row and tile is a legal cp.async.bulk source and destination
    const int64_t per16 = 16 / es;
    v->obs_stride = spec.kind == LLE_OBS_STATE ? (int64_t)v->S : ((int64_t)m0.header().obs_floats + per16 - 1) / per16 * per16;
    v->render = opts->write_obs && spec.kind != LLE_OBS_STATE;  // whether the tile renderer runs

    LLE_CUDA(cudaSetDevice(v->device));
    cudaDeviceProp prop;
    LLE_CUDA(cudaGetDeviceProperties(&prop, v->device));

    // ---- work decomposition and observation tiling.  One bulk store should move a few KB; a warp takes a
    // ticket for `group` consecutive worlds, computes them, then streams their observation tiles.  Sizes are reasoned about in
    // bytes (`es` per element): an int8 row takes a quarter of the bytes of the f32 row and is tiled like an f32 row of that size.
    v->Wd = 1;
    while (v->Wd < v->A) v->Wd *= 2;
    // at least 2 lanes per world (16 worlds per pass, 16 per ticket).  Measured on B200 with narrow-grid pipelining
    // (us/step, lanes per world 1 / 2 / 4): level 1: 40.7 / 40.3 / 45.4; level 3: 51.8 / 51.5 / 58.0
    // tiny observations: the logic dominates, pack more worlds per pass.  In bytes: a level-6 int8 row (1,872 B) is small and
    // runs on the thread-per-world kernel (level 6 x 65,536 on one B200: 45.5 us per step there, 65.9 on the fast kernel)
    const bool small_obs = v->obs_stride * es < 2048;
    v->Wd = std::max(v->Wd, small_obs ? 1 : 2);
    const int64_t stride = v->obs_stride;
    // 4-8 KB per bulk store; partial observations: up to 9.6 KB, one tile buffer and 16 worlds per ticket, which keeps five
    // CTAs per SM (sweep of buffers x tile size x ticket size on level 6 x 65,536, us per step before -> after:
    // partial3x3 72.5 -> 57.9, partial5x5 84.4 -> 79.2, partial7x7 134.7 -> 94.5)
    const bool partial_obs = spec.kind == LLE_OBS_PARTIAL;
    bool random_starts = false;  // start sampling lives in the general kernel only
    for (int k = 0; k < n_maps; ++k) random_starts = random_starts || cms[k]->header().random_starts;
    // a record the thread-per-world kernel (tiny_kernel.cuh) can hold: few agents, at most 8 words, one word per beam, one gem word
    const bool tiny_record = v->A <= 4 && v->L.n_words <= 8 && !v->L.wide_flags && v->L.on_words == 1 && v->L.gem_words <= 1 && v->L.sub_words == 0 &&
                             !v->randomize && !random_starts && opts->write_obs && !env_int("LLE_B200_NO_TINY", 0);
    // Partial observations of such worlds, when the windows of one world (A (2A+3) size^2 floats) are under 2 KB (level 6: 3x3):
    // built by 32 / E lanes in a tile of E worlds; tickets of 32 worlds.  Level 6 x 65,536, us per step, this kernel / the general
    // one: 3x3 52.5 / 58-67, 5x5 90 / 85, 7x7 166 / 98 - with 2,048 tickets a launch is one wave of warps and the step takes as
    // long as one ticket, so larger windows (more rounds per ticket) stay on the general kernel, which has four times the warps.
    const bool tiny_partial = partial_obs && tiny_record && (stride * 4 < 2048 || env_int("LLE_B200_TINY_PARTIAL", 0));
    // (targets and limits in 4-byte units, as measured on f32; elements of the vec's type below)
    const int64_t kTileTargetFloats = (partial_obs ? 2400 : small_obs ? 2048 : 1024) * 4 / es;
    // the partial renderer builds whole worlds (all agents' windows) in one tile: allow up to 48 KB per warp
    const int64_t kTileMaxFloats = (spec.kind == LLE_OBS_PARTIAL ? 12288 : 6144) * 4 / es;
    if (spec.kind == LLE_OBS_PARTIAL && stride > kTileMaxFloats)
        return fail(LLE_LIMIT_EXCEEDED, "partial observation of one world exceeds 48 KB (n_agents * (2 n_agents + 3) * size^2 floats)");
    if (stride <= kTileMaxFloats) {
        v->n_chunks = 1;
        v->E = std::max(1, std::min(32, pow2_floor((int)std::max<int64_t>(1, kTileTargetFloats / stride))));
        v->chunk_floats = (int)stride;
        v->tile_floats = (int)(v->E * stride);
        v->group = tiny_partial ? 32 : partial_obs ? std::max(std::max(v->E, 16), 32 / v->Wd) : small_obs ? 32 : std::max(std::max(v->E, 8), 32 / v->Wd);
        v->n_buf = 1;
    } else {
        v->E = 1;
        v->chunk_floats = lle_chunk_elems(stride, (int)es);  // <= 12 KB, balanced (static_map.h)
        v->n_chunks = (int)((stride + v->chunk_floats - 1) / v->chunk_floats);
        v->tile_floats = v->chunk_floats;
        // A ticket walks its worlds chunk by chunk, so the two tile buffers are rebuilt from the static plane twice per
        // chunk index and ticket: the more worlds per ticket, the fewer rebuilds per world (perspective level 6 x 65,536:
        // 350 / 317 / 299 us/step with 8 / 16 / 32) — as long as there are enough tickets to balance the warps (64x64 x 16,384:
        // 809 / 825 / 1,084 us/step): at least 2,048 tickets.
        // Tickets are also the grain of the dataflow ordering between overlapped steps, so very large ones stall the
        // pipeline (64x64 x 131,072: 2.02e7 / 2.07e7 / 1.72e7 env-steps/s with 8 / 16 / 32): at most 6 MB per ticket.
        v->group = 32;
        while (v->group > std::max(8, 32 / v->Wd) && (v->N_pad / v->group < 2048 || (int64_t)v->group * stride * es > (6 << 20))) v->group >>= 1;
        v->n_buf = 2;
    }
    auto warp_smem_for = [&](int n_buf) {
        size_t bytes = (size_t)n_buf * v->tile_floats * es;            // tiles
        bytes += (size_t)v->group * v->L.stride * 4;                   // records of the group
        bytes += (size_t)n_buf * v->E * v->L.stride * 4;               // records applied to the tiles
        bytes += (size_t)(2 * n_buf * v->E + n_buf + v->group) * 4;    // tags + map ids + fresh flags
        return (int)((bytes + 127) / 128 * 128);
    };
    v->warp_smem = warp_smem_for(v->n_buf);
    v->smem = (size_t)v->warp_smem * kWarps;
    int max_patch = 0;
    for (int k = 0; k < n_maps; ++k) max_patch = std::max(max_patch, (int)cms[k]->header().n_patch);
    for (const auto& m : v->variant_maps) max_patch = std::max(max_patch, (int)m.header().n_patch);
    v->fast = v->n_chunks == 1 && v->n_buf == 1 && max_patch <= 64 && v->L.stride <= 32 && opts->write_obs &&
              spec.kind == LLE_OBS_LAYERED && !v->randomize && !random_starts;
    if (spec.kind == LLE_OBS_PARTIAL) {
        v->by_feature = true;  // a window task costs about three feature tasks (measured on level 6)
        v->feature_limit = 2 * spec.param * spec.param;
        for (int k = 0; k < n_maps; ++k) v->by_feature = v->by_feature && (int)cms[k]->header().n_patch <= v->feature_limit;
        for (const auto& m : v->variant_maps) v->by_feature = v->by_feature && (int)m.header().n_patch <= v->feature_limit;
    }
    // Tiny maps (small observation, few agents, a record of at most 8 words): the step runs one thread per world.
    v->tiny = ((v->fast && small_obs) || tiny_partial) && tiny_record && v->group == 32;
    v->tiny_partial = v->tiny && tiny_partial;
    select_kernels(v.get());
    int blocks_per_sm = -1;  // the grid is shared by the three modes: size it for the most demanding one
    for (KernelFn k : {v->k_step, v->k_step_parts, v->k_reset, v->k_set_state}) LLE_CUDA(configure_kernel(k, v->smem, &blocks_per_sm));
    if (blocks_per_sm < 1) return fail(LLE_CUDA_ERROR, "kernel does not fit on an SM");
    if (v->tiny) {
        // worlds per tile / bulk store (measured on 2^20 5x5 worlds, us per step: 4: 232, 8: 243, 16: 343, 32: 558 - occupancy)
        int e_default = 4;
        // int8 rows: more worlds per tile, up to 4 KB and 16 worlds (measured on 2^20 5x5 worlds, 208 B rows, us per step: 4: 157.7,
        // 8: 145.4, 16: 135.7, 32: 142.8; level 1 x 65,536, 944 B rows: 4: 14.7, 16: 14.4)
        if (v->i8)
            while (e_default < 16 && 2 * e_default * stride <= 4096) e_default *= 2;
        if (tiny_partial) {  // the largest tile of at most 13 KB (level 6 3x3: 8 worlds; measured 2 / 4 / 8: 60.8 / 57.0 / 52.5 us)
            e_default = 1;
            while (e_default < 32 && 2 * e_default * stride * 4 <= 13312) e_default *= 2;
        }
        v->tiny_E = e_default;
        auto tiny_bytes = [&]() {  // the records' columns + the prefetched next records, list pointers, list lengths, the tile
            const size_t bytes = 2 * (size_t)v->L.stride * 32 * 4 + 32 * 8 + 32 * 4 + (tiny_partial ? 32 * 8 : 0) + (size_t)v->tiny_E * stride * es;
            return (bytes + 127) / 128 * 128;
        };
        v->tiny_warp_smem = (int)tiny_bytes();
        v->tiny_smem = (size_t)v->tiny_warp_smem * kWarps;
        int tb = -1;
        LLE_CUDA(configure_kernel(v->k_tiny, v->tiny_smem, &tb));
        if (tb < 1) {
            v->tiny = false;
            v->k_tiny = nullptr;
        }
        const int64_t tickets = v->N_pad / v->group;
        v->tiny_grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)prop.multiProcessorCount * tb, (tickets + kWarps - 1) / kWarps));
    }
    const int64_t n_tickets = v->N_pad / v->group;
    v->grid = (int)std::min<int64_t>((int64_t)prop.multiProcessorCount * blocks_per_sm, (n_tickets + kWarps - 1) / kWarps);
    v->grid = std::max(v->grid, 1);
    {
        // measured on B200 (us/step, 1 CTA per SM vs the full grid): level 6 x 65,536: 76.5 vs 81.4; level 1: 49.7 vs 54.0;
        // 1,024 generated 5x5 maps x 1,024 (instruction-bound, 445 us steps): 467 vs 445 -> tiny observations keep the full grid
        const int step_ctas = small_obs ? blocks_per_sm : std::min(blocks_per_sm, 2);
        v->grid_step = (int)std::min<int64_t>((int64_t)prop.multiProcessorCount * step_ctas, (n_tickets + kWarps - 1) / kWarps);
        v->grid_step = std::max(v->grid_step, 1);
    }
    {
        const int idle_ctas = small_obs ? blocks_per_sm : std::min(blocks_per_sm, 4);
        v->grid_idle = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)prop.multiProcessorCount * idle_ctas, (n_tickets + kWarps - 1) / kWarps));
    }

    // ---- device memory
    std::vector<const uint8_t*> table;
    std::vector<const CompiledMap*> upload;  // blob table: one entry per map, or per (map, colouring) with randomize_lasers
    if (v->randomize) for (const auto& m : v->variant_maps) upload.push_back(&m);
    else upload = cms;
    for (size_t k = 0; k < upload.size(); ++k) {
        const auto& blob = upload[k]->blob;
        uint8_t* d = nullptr;
        LLE_CUDA(cudaMalloc((void**)&d, blob.size()));
        v->d_blobs.push_back(d);
        LLE_CUDA(cudaMemcpy(d, blob.data(), blob.size(), cudaMemcpyHostToDevice));
        table.push_back(d);
    }
    if (!v->randomize) {  // blob 0 is map 0 as given
        v->map0 = host_bind(v->d_blobs[0], upload[0]->header());
        v->has_map0 = true;
    }
    LLE_CUDA(cudaMalloc((void**)&v->d_blob_table, table.size() * sizeof(uint8_t*)));
    LLE_CUDA(cudaMemcpy((void*)v->d_blob_table, table.data(), table.size() * sizeof(uint8_t*), cudaMemcpyHostToDevice));
    if ((map_of_env && n_maps > 1) || v->randomize) {
        std::vector<int32_t> padded((size_t)v->N_pad, 0);
        if (map_of_env) std::copy(map_of_env, map_of_env + n_envs, padded.begin());
        for (int64_t e = n_envs; e < v->N_pad; ++e) padded[(size_t)e] = map_of_env ? map_of_env[n_envs - 1] : 0;
        if (v->randomize)  // entries become blob indices: map * n_variants + the colouring the text describes
            for (auto& id : padded) {
                const CompiledMap& m = *cms[(size_t)id];
                int variant = 0, scale = 1;
                for (int b = 0; b < m.NB; ++b) { variant += m.sources[(size_t)b].colour * scale; scale *= v->A; }
                id = id * v->n_variants + variant;
            }
        LLE_CUDA(dalloc(&v->d_map_of_env, (size_t)v->N_pad));
        LLE_CUDA(cudaMemcpy(v->d_map_of_env, padded.data(), padded.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    } else if (map_of_env && n_maps == 1) {
        v->d_map_of_env = nullptr;
    }
    const size_t Np = (size_t)v->N_pad;
    LLE_CUDA(dalloc(&v->d_records, (size_t)v->L.stride * Np));
    if (opts->write_obs && v->i8) LLE_CUDA(dalloc(&v->d_obs_i8, (size_t)v->obs_stride * Np));
    else if (opts->write_obs) LLE_CUDA(dalloc(&v->d_obs, (size_t)v->obs_stride * Np));
    v->hdr0 = m0.header();
    LLE_CUDA(dalloc(&v->d_state, (size_t)v->S * Np));
    LLE_CUDA(dalloc(&v->d_avail, (size_t)v->A * 5 * Np));
    LLE_CUDA(dalloc(&v->d_reward, (size_t)v->R * Np));
    LLE_CUDA(dalloc(&v->d_done, Np));
    LLE_CUDA(dalloc(&v->d_events, (size_t)v->A * Np));
    LLE_CUDA(dalloc(&v->d_actions, (size_t)v->A * Np));
    LLE_CUDA(dalloc(&v->d_err, Np));
    if (v->JE) LLE_CUDA(dalloc(&v->d_extras, (size_t)v->A * v->JE * Np));
    if (opts->episode_stats) {
        LLE_CUDA(dalloc(&v->d_info, (size_t)(2 + v->A) * Np));
        LLE_CUDA(dalloc(&v->d_ep_return, (size_t)v->R * Np));
        LLE_CUDA(dalloc(&v->d_last_return, (size_t)v->R * Np));
        LLE_CUDA(dalloc(&v->d_ep_length, Np));
        LLE_CUDA(dalloc(&v->d_last_length, Np));
    }
    LLE_CUDA(dalloc(&v->d_sched, (size_t)kSchedSlotWords * kSchedSlots));
    LLE_CUDA(dalloc(&v->d_flags, (size_t)(v->N_pad / v->group)));
    LLE_CUDA(cudaHostAlloc((void**)&v->h_retired_seq, 64 * sizeof(uint32_t), cudaHostAllocMapped));
    std::memset(v->h_retired_seq, 0, 64 * sizeof(uint32_t));
    LLE_CUDA(dalloc(&v->d_retired_count, 1));
    LLE_CUDA(dalloc(&v->d_actions_stage, (size_t)v->A * Np));
    if (env_int("LLE_B200_TIMELINE", 0)) LLE_CUDA(dalloc(&v->d_timeline, (size_t)v->grid * kWarps * 4));
    LLE_CUDA(cudaEventCreate(&v->ev0));
    LLE_CUDA(cudaEventCreate(&v->ev1));

    // World::new resets itself (world.rs:82)
    v->creating = true;
    int rc = lle_vec_reset(v.get(), nullptr, nullptr);
    v->creating = false;
    if (rc != LLE_OK) return rc;
    LLE_CUDA(cudaDeviceSynchronize());
    if (opts->state_type != LLE_OBS_STATE || opts->state_param != 0) {
        lle_vec_options so = *opts;
        so.obs_type = opts->state_type; so.obs_param = opts->state_param;
        so.state_type = LLE_OBS_STATE; so.state_param = 0;
        so.write_obs = 1;
        so.episode_stats = 0;
        so.obs_dtype = LLE_DTYPE_F32;  // the state observation stays float32
        lle_vec* sh = nullptr;
        if (int rc2 = lle_vec_create(maps, n_maps, map_of_env, n_envs, &so, &sh)) return rc2;
        if (sh->L.stride != v->L.stride || sh->N_pad != v->N_pad || (sh->d_map_of_env == nullptr) != (v->d_map_of_env == nullptr)) {
            lle_vec_destroy(sh);
            return fail(LLE_INVALID_ARGUMENT, "state_type: record layouts differ");
        }
        cudaFree(sh->d_records);
        cudaFree(sh->d_map_of_env);
        sh->d_records = v->d_records;
        sh->d_map_of_env = v->d_map_of_env;
        sh->borrows_records = true;
        v->shadow = sh;
        v->pdl = false;  // the re-export launch sits between two steps: they cannot overlap programmatically
        if (int rc2 = lle_vec_refresh(sh, nullptr)) return rc2;
        LLE_CUDA(cudaDeviceSynchronize());
    }
    *out = v.release();
    return LLE_OK;
}

int lle_vec_get_buffers(lle_vec* v, lle_vec_buffers* out) {
    if (!v || !out) return fail(LLE_INVALID_ARGUMENT, "null argument");
    std::memset(out, 0, sizeof *out);
    out->n_envs = v->N;
    out->n_agents = v->A; out->n_gems = v->G; out->n_channels = v->C; out->height = v->H; out->width = v->W;
    out->reward_dim = v->R; out->state_dim = v->S; out->n_beams_max = v->NBmax;
    out->obs_stride = v->obs_stride;
    out->obs = v->d_obs; out->state = v->d_state; out->avail = v->d_avail; out->reward = v->d_reward; out->done = v->d_done;
    out->events = v->d_events; out->actions = v->d_actions; out->err = v->d_err;
    out->record_bytes = (int64_t)v->L.stride * 4;
    out->extras = v->d_extras;
    out->extras_dim = v->JE;
    out->obs_type = v->opts.obs_type; out->obs_param = v->opts.obs_param;
    out->obs_view_agents = v->hdr0.view_agents;
    out->obs_c = v->hdr0.obs_c; out->obs_h = v->hdr0.obs_h; out->obs_w = v->hdr0.obs_w;
    out->obs_invalid = v->obs_invalid;
    out->map_index = v->d_map_of_env;
    out->n_variants = v->n_variants;
    out->info = v->d_info; out->ep_return = v->d_ep_return; out->ep_length = v->d_ep_length; out->last_return = v->d_last_return; out->last_length = v->d_last_length;
    out->obs_i8 = v->d_obs_i8;
    out->obs_dtype = v->opts.obs_dtype;
    if (v->shadow) {
        const lle_vec* sh = v->shadow;
        out->state_obs = sh->d_obs; out->state_obs_stride = sh->obs_stride;
        out->state_type = sh->opts.obs_type; out->state_param = sh->opts.obs_param;
        out->state_view_agents = sh->hdr0.view_agents;
        out->state_c = sh->hdr0.obs_c; out->state_h = sh->hdr0.obs_h; out->state_w = sh->hdr0.obs_w;
        if (sh->obs_invalid) out->obs_invalid = 1;
    } else {
        out->state_type = LLE_OBS_STATE;
    }
    return LLE_OK;
}

int lle_vec_get_sources(lle_vec* v, int32_t map_index, int32_t* out, int32_t cap, int32_t* n) {
    if (!v || !n || map_index < 0 || map_index >= (int)v->src_state.size()) return fail(LLE_INVALID_ARGUMENT, "bad argument");
    const auto& st = v->src_state[(size_t)map_index];
    *n = (int32_t)st.size();
    for (int k = 0; k < (int)st.size() && k < cap && out; ++k) { out[2 * k] = st[k].colour; out[2 * k + 1] = st[k].enabled; }
    return LLE_OK;
}

namespace {
// Recompiles map `map_index` of the vec with the given source states / exits and swaps the device tables.
int swap_map(lle_vec* v, int map_index, const std::vector<SourceState>& sources, const std::vector<Cell>* exits, cudaStream_t s,
             CompiledMap* out_cm) {
    CompiledMap cm;
    try {
        cm = compile_map(v->map_texts[(size_t)map_index], ObsSpec{v->opts.obs_type, v->opts.obs_param, v->opts.obs_dtype}, &sources, exits);
    } catch (const MapError& e) {
        return fail(e.status, e.what());
    }
    if (v->fast && cm.header().n_patch > 64)
        return fail(LLE_LIMIT_EXCEEDED, "the modified map has more than 64 dynamic observation cells (vec was created for the fast tile path)");
    if (v->by_feature && (int)cm.header().n_patch > v->feature_limit)
        return fail(LLE_LIMIT_EXCEEDED, "the modified map has too many features for the feature-driven partial renderer the vec was created with");
    LLE_CUDA(cudaSetDevice(v->device));
    LLE_CUDA(cudaStreamSynchronize(s));  // control-plane operation: nothing of this vec is in flight while its map changes
    uint8_t* d = nullptr;
    LLE_CUDA(cudaMalloc((void**)&d, cm.blob.size()));
    LLE_CUDA(cudaMemcpy(d, cm.blob.data(), cm.blob.size(), cudaMemcpyHostToDevice));
    LLE_CUDA(cudaMemcpy((void*)(v->d_blob_table + map_index), &d, sizeof d, cudaMemcpyHostToDevice));
    v->retired_blobs.push_back(v->d_blobs[(size_t)map_index]);
    v->d_blobs[(size_t)map_index] = d;
    v->map_patches[(size_t)map_index] = (int)cm.header().n_patch;
    v->map_obs_invalid[(size_t)map_index] = (int)cm.header().obs_invalid;
    v->obs_invalid = 0;
    for (int f : v->map_obs_invalid) v->obs_invalid |= f;
    if (map_index == 0) {
        v->hdr0 = cm.header();
        v->map0 = host_bind(d, cm.header());
    }
    v->last_was_step = false;
    if (out_cm) *out_cm = std::move(cm);
    return LLE_OK;
}
}  // namespace

int lle_vec_set_source(lle_vec* v, int32_t map_index, int32_t source_index, int32_t agent_id, int32_t enabled, void* stream) {
    if (!v || map_index < 0 || map_index >= (int)v->src_state.size()) return fail(LLE_INVALID_ARGUMENT, "map index out of range");
    auto& st = v->src_state[(size_t)map_index];
    if (source_index < 0 || source_index >= (int)st.size()) return fail(LLE_INVALID_ARGUMENT, "laser source index out of range");
    if (v->randomize) return fail(LLE_INVALID_ARGUMENT, "source mutators are not available together with randomize_lasers");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    std::vector<SourceState> next = st;
    if (agent_id >= 0) next[(size_t)source_index].colour = agent_id;
    const bool was_enabled = st[(size_t)source_index].enabled;
    if (enabled >= 0) next[(size_t)source_index].enabled = enabled != 0;
    if (v->shadow)
        if (int rc2 = lle_vec_set_source(v->shadow, map_index, source_index, agent_id, enabled, stream)) return rc2;
    cudaStream_t s = (cudaStream_t)stream;
    CompiledMap cm;
    int rc = swap_map(v, map_index, next, v->map_exits_set[(size_t)map_index] ? &v->map_exits[(size_t)map_index] : nullptr, s, &cm);
    if (rc != LLE_OK) return rc;
    st = next;
    if (enabled >= 0 && (enabled != 0) != was_enabled) {  // LaserBeam::enable / disable (laser.rs:69-77)
        const int len = cm.sources[(size_t)source_index].len;
        const uint64_t mask = enabled ? (len >= 64 ? ~0ull : ((1ull << len) - 1ull)) : 0ull;
        const int threads = 256;
        const int blocks = (int)((v->N_pad + threads - 1) / threads);
        lle_set_beam_kernel<<<blocks, threads, 0, s>>>(v->d_records, v->L, v->N_pad, v->d_map_of_env, map_index, source_index, mask);
        LLE_CUDA(cudaGetLastError());
        v->launches++;
    }
    return LLE_OK;
}

int lle_vec_collect_gem(lle_vec* v, int32_t map_index, int32_t gem_index, void* stream) {
    if (!v || map_index < 0 || map_index >= (int)v->src_state.size()) return fail(LLE_INVALID_ARGUMENT, "map index out of range");
    if (gem_index < 0 || gem_index >= v->G) return fail(LLE_INDEX_ERROR, "gem index out of range");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    if (!((v->map_gem_toplevel[(size_t)map_index] >> gem_index) & 1ull))  // pygem.rs:54-62: a gem under a laser tile is a Tile::Laser
        return fail(LLE_INVALID_ARGUMENT, "the tile is not a gem (the gem is wrapped by a laser tile)");
    LLE_CUDA(cudaSetDevice(v->device));
    const int threads = 256;
    const int blocks = (int)((v->N_pad + threads - 1) / threads);
    lle_collect_gem_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(v->d_records, v->L, v->N_pad, v->d_map_of_env, map_index, gem_index);
    LLE_CUDA(cudaGetLastError());
    v->launches++;
    return LLE_OK;
}

int lle_vec_set_exits(lle_vec* v, int32_t map_index, const int32_t* exits_ij, int32_t n_exits, void* stream) {
    if (!v || map_index < 0 || map_index >= (int)v->src_state.size()) return fail(LLE_INVALID_ARGUMENT, "map index out of range");
    if (n_exits < 0 || (n_exits > 0 && !exits_ij)) return fail(LLE_INVALID_ARGUMENT, "bad exit list");
    if (v->randomize) return fail(LLE_INVALID_ARGUMENT, "the exit setter is not available together with randomize_lasers");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    if (v->shadow)
        if (int rc2 = lle_vec_set_exits(v->shadow, map_index, exits_ij, n_exits, stream)) return rc2;
    std::vector<Cell> exits;
    for (int k = 0; k < n_exits; ++k) exits.push_back(Cell{exits_ij[2 * k], exits_ij[2 * k + 1]});
    int rc = swap_map(v, map_index, v->src_state[(size_t)map_index], &exits, (cudaStream_t)stream, nullptr);
    if (rc != LLE_OK) return rc;
    v->map_exits[(size_t)map_index] = exits;
    v->map_exits_set[(size_t)map_index] = 1;
    return LLE_OK;
}

// LLE(state_type=...): after every launch that changes the records, the shadow re-exports the state's observation
#define LLE_SYNC_SHADOW(v, stream)                                          \
    do {                                                                    \
        if ((v)->shadow)                                                    \
            if (int _rc = lle_vec_refresh((v)->shadow, (void*)(stream))) return _rc; \
    } while (0)

int lle_vec_reset(lle_vec* v, const uint8_t* mask_dev, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    LLE_CUDA(cudaSetDevice(v->device));
    v->reset_epoch++;
    KParams p = base_params(v);
    p.mode = MODE_RESET;
    p.reset_mask = mask_dev;
    LLE_CUDA(launch(v, p, (cudaStream_t)stream));
    v->launches++;
    LLE_SYNC_SHADOW(v, stream);
    return LLE_OK;
}

int lle_vec_refresh(lle_vec* v, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    LLE_CUDA(cudaSetDevice(v->device));
    KParams p = base_params(v);
    p.mode = MODE_RESET;
    p.refresh_only = 1;
    LLE_CUDA(launch(v, p, (cudaStream_t)stream));
    v->launches++;
    LLE_SYNC_SHADOW(v, stream);
    return LLE_OK;
}

int lle_vec_step(lle_vec* v, const int8_t* actions_dev, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    LLE_CUDA(cudaSetDevice(v->device));
    KParams p = base_params(v);
    p.mode = MODE_STEP;
    p.actions_in = actions_dev;
    LLE_CUDA(launch(v, p, (cudaStream_t)stream));
    v->launches++;
    v->t++;
    LLE_SYNC_SHADOW(v, stream);
    return LLE_OK;
}

int lle_vec_rollout(lle_vec* v, int32_t n_steps, void* stream) {
    if (!v || n_steps < 1) return fail(LLE_INVALID_ARGUMENT, "bad argument");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    LLE_CUDA(cudaSetDevice(v->device));
    // (step, ticket) pairs are counted in 32 bits on the device: long rollouts over many tickets go out as several launches
    // (bit-identical: the epoch flags order them exactly like the steps of one launch)
    const int64_t n_tickets = v->N_pad / v->group;
    const int32_t max_steps = (int32_t)std::max<int64_t>(1, std::min<int64_t>((int64_t)1 << 20, ((int64_t)1 << 30) / n_tickets));
    for (int32_t left = n_steps; left > 0;) {
        const int32_t k = std::min(left, max_steps);
        KParams p = base_params(v);
        p.mode = MODE_STEP;
        p.actions_in = nullptr;
        p.n_steps = k;
        LLE_CUDA(launch(v, p, (cudaStream_t)stream));
        v->launches++;
        v->t += (uint64_t)k;
        left -= k;
    }
    LLE_SYNC_SHADOW(v, stream);
    return LLE_OK;
}

namespace {
int pipeline_setup(lle_vec* v) {
    if (v->pipe_ready) return LLE_OK;
    LLE_CUDA(resolve_memops());
    LLE_CUDA(cudaStreamCreateWithFlags(&v->s_in, cudaStreamNonBlocking));
    LLE_CUDA(cudaStreamCreateWithFlags(&v->s_main, cudaStreamNonBlocking));
    LLE_CUDA(cudaEventCreateWithFlags(&v->ev_user, cudaEventDisableTiming));
    for (int k = 0; k < lle_vec::kPipeSlots; ++k) LLE_CUDA(dalloc(&v->d_stage[k], (size_t)v->A * v->N_pad));
    LLE_CUDA(dalloc(&v->d_pipe_flags, 2));
    LLE_CUDA(cudaHostAlloc((void**)&v->h_out_flags, lle_vec::kPipeSlots * 32 * sizeof(uint32_t), cudaHostAllocMapped));
    std::memset(v->h_out_flags, 0, lle_vec::kPipeSlots * 32 * sizeof(uint32_t));
    LLE_CUDA(cudaHostGetDevicePointer((void**)&v->d_out_flags, v->h_out_flags, 0));
    LLE_CUDA(cudaDeviceSynchronize());
    v->pipe_ready = true;
    return LLE_OK;
}
}  // namespace

int lle_vec_step_host(lle_vec* v, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    LLE_CUDA(cudaSetDevice(v->device));
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    // pinned buffers: one submit + wait of the pipeline below (one copy, one launch, results written straight to host memory)
    if ((!actions_host || device_view(v, actions_host)) && (!reward_host || device_view(v, reward_host)) && (!done_host || device_view(v, done_host))) {
        int rc = lle_vec_pipeline_submit(v, actions_host, reward_host, done_host, stream);
        if (rc != LLE_OK) return rc;
        return lle_vec_pipeline_wait(v, nullptr);
    }
    // pageable buffers: staged copies on the caller's stream, then a stream synchronisation
    cudaStream_t s = (cudaStream_t)stream;
    const int8_t* dev_actions = nullptr;
    if (actions_host) {
        LLE_CUDA(cudaMemcpyAsync(v->d_actions_stage, actions_host, (size_t)v->N * v->A, cudaMemcpyHostToDevice, s));
        dev_actions = v->d_actions_stage;
    }
    int rc = lle_vec_step(v, dev_actions, stream);
    if (rc != LLE_OK) return rc;
    if (reward_host) LLE_CUDA(cudaMemcpyAsync(reward_host, v->d_reward, (size_t)v->N * v->R * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (done_host) LLE_CUDA(cudaMemcpyAsync(done_host, v->d_done, (size_t)v->N, cudaMemcpyDeviceToHost, s));
    LLE_CUDA(cudaStreamSynchronize(s));
    return LLE_OK;
}

int lle_vec_fetch(lle_vec* v, int which, size_t offset, size_t bytes, void* host_dst, void* stream) {
    if (!v || !host_dst) return fail(LLE_INVALID_ARGUMENT, "null argument");
    const size_t N = (size_t)v->N, A = (size_t)v->A;
    const void* src = nullptr;
    size_t size = 0;
    switch (which) {
        case LLE_BUF_OBS:
            src = v->i8 ? (const void*)v->d_obs_i8 : (const void*)v->d_obs;
            size = N * (size_t)v->obs_stride * (v->i8 ? 1 : 4);
            break;
        case LLE_BUF_STATE: src = v->d_state; size = N * (size_t)v->S * 4; break;
        case LLE_BUF_AVAIL: src = v->d_avail; size = N * A * 5; break;
        case LLE_BUF_REWARD: src = v->d_reward; size = N * (size_t)v->R * 4; break;
        case LLE_BUF_DONE: src = v->d_done; size = N; break;
        case LLE_BUF_EVENTS: src = v->d_events; size = N * A; break;
        case LLE_BUF_ACTIONS: src = v->d_actions; size = N * A; break;
        case LLE_BUF_ERR: src = v->d_err; size = N; break;
        case LLE_BUF_EXTRAS: src = v->d_extras; size = N * A * (size_t)v->JE * 4; break;
        case LLE_BUF_STATE_OBS: src = v->shadow ? v->shadow->d_obs : nullptr; size = v->shadow ? N * (size_t)v->shadow->obs_stride * 4 : 0; break;
        case LLE_BUF_INFO: src = v->d_info; size = N * (2 + A); break;
        default: return fail(LLE_INVALID_ARGUMENT, "unknown buffer");
    }
    if (!src) return fail(LLE_INVALID_ARGUMENT, "the vec does not keep that buffer");
    if (offset > size || bytes > size - offset) return fail(LLE_INDEX_ERROR, "range outside the buffer");
    LLE_CUDA(cudaSetDevice(v->device));
    LLE_CUDA(cudaMemcpyAsync(host_dst, (const uint8_t*)src + offset, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    LLE_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return LLE_OK;
}

int lle_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(LLE_INVALID_ARGUMENT, "null argument");
    LLE_CUDA(cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable | cudaHostAllocMapped));
    return LLE_OK;
}
int lle_host_free(void* ptr) {
    if (ptr) LLE_CUDA(cudaFreeHost(ptr));
    return LLE_OK;
}

int lle_vec_pipeline_submit(lle_vec* v, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* after_stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (v->pipe_submitted - v->pipe_completed >= (uint64_t)lle_vec::kPipeSlots)
        return fail(LLE_INVALID_ARGUMENT, "pipeline full: call lle_vec_pipeline_wait before submitting another step");
    LLE_CUDA(cudaSetDevice(v->device));
    if (int rc = pipeline_setup(v)) return rc;
    // Pinned (page-locked) host buffers are REQUIRED: the step kernel spins on a flag that the copy stream publishes behind the
    // H2D copy (only a truly asynchronous copy keeps the two streams independent of the calling thread), and it writes reward
    // and done straight into the host buffers (zero-copy), followed by a completion word the host polls.
    void* reward_dev = reward_host ? device_view(v, reward_host) : nullptr;
    void* done_dev = done_host ? device_view(v, done_host) : nullptr;
    if ((actions_host && !device_view(v, actions_host)) || (reward_host && !reward_dev) || (done_host && !done_dev))
        return fail(LLE_INVALID_ARGUMENT, "lle_vec_pipeline_submit needs pinned (page-locked) host buffers (lle_host_alloc / cudaHostAlloc / cudaHostRegister)");
    if (v->pipe_submitted == v->pipe_completed && after_stream != LLE_STREAM_NONE) {  // pipeline empty: order it after the caller's stream
        LLE_CUDA(cudaEventRecord(v->ev_user, (cudaStream_t)after_stream));
        LLE_CUDA(cudaStreamWaitEvent(v->s_main, v->ev_user, 0));
    }
    // Nothing is committed to the host bookkeeping until the step kernel has been accepted by the stream.
    const uint64_t next = v->pipe_submitted + 1;
    const uint32_t n = (uint32_t)next;
    const int slot = (int)(v->pipe_submitted % lle_vec::kPipeSlots);
    KParams p = base_params(v);
    p.mode = MODE_STEP;
    if (actions_host) {
        if (v->pipe_submitted == v->pipe_completed) {
            // Nothing of this vec is in flight (a closed loop: the caller waited for the previous step before choosing these
            // actions): the copy simply precedes the kernel on the compute stream.  A kernel that waited for its actions on the
            // device would hold SM slots idle for the ~10 us the copy takes - slots that the other sub-batches of an
            // EnvPool-style loop could use.
            LLE_CUDA(cudaMemcpyAsync(v->d_stage[slot], actions_host, (size_t)v->N * v->A, cudaMemcpyHostToDevice, v->s_main));
            p.actions_in = v->d_stage[slot];
        } else {
            // Steps already in flight: the copy travels on its own stream, overlapping the kernels ahead, and the kernel waits
            // for it on the device (no stream-level dependency between consecutive step kernels: they stay programmatically
            // dependent launches).
            LLE_CUDA(cudaMemcpyAsync(v->d_stage[slot], actions_host, (size_t)v->N * v->A, cudaMemcpyHostToDevice, v->s_in));
            if (g_write_value32((CUstream)v->s_in, (CUdeviceptr)(uintptr_t)(v->d_pipe_flags + 0), n, CU_STREAM_WRITE_VALUE_DEFAULT) != CUDA_SUCCESS)
                return fail(LLE_CUDA_ERROR, "cuStreamWriteValue32 failed");
            p.actions_in = v->d_stage[slot];
            p.in_flag = v->d_pipe_flags + 0;
            p.in_need = n;
        }
    }
    p.out_flag = v->d_out_flags + slot * 32;  // one 128-byte line per slot
    p.out_value = n;
    p.reward2 = (float*)reward_dev;
    p.done2 = (uint8_t*)done_dev;
    LLE_CUDA(launch(v, p, v->s_main));
    v->launches++;
    v->t++;
    v->pipe_submitted = next;
    LLE_SYNC_SHADOW(v, v->s_main);
    return LLE_OK;
}

int lle_vec_pipeline_wait(lle_vec* v, int32_t* outstanding) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (v->pipe_submitted == v->pipe_completed) {
        if (outstanding) *outstanding = 0;
        return fail(LLE_INVALID_ARGUMENT, "pipeline empty: nothing to wait for");
    }
    const int slot = (int)(v->pipe_completed % lle_vec::kPipeSlots);
    const uint32_t n = (uint32_t)(v->pipe_completed + 1);
    volatile uint32_t* flag = v->h_out_flags + slot * 32;
    // The last warp of the step writes n here after a system-scope fence behind every result byte.  Poll; look at the stream
    // now and then so that a failed launch surfaces as an error instead of a hang.
    for (uint64_t spins = 0; (int32_t)(*flag - n) < 0; ++spins) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0xFFFFF) == 0xFFFFF) {
            cudaSetDevice(v->device);
            cudaError_t e = cudaStreamQuery(v->s_main);
            if (e != cudaSuccess && e != cudaErrorNotReady)
                return fail(LLE_CUDA_ERROR, std::string("step kernel failed: ") + cudaGetErrorString(e));
            if (e == cudaSuccess && (int32_t)(*flag - n) < 0)  // the stream drained without publishing: should not happen
                return fail(LLE_CUDA_ERROR, "the step retired without publishing its completion");
        }
    }
    __sync_synchronize();
    v->pipe_completed++;
    if (outstanding) *outstanding = (int32_t)(v->pipe_submitted - v->pipe_completed);
    return LLE_OK;
}

// ---- closed loop over parts of one batch (include/lle_b200.h)
int lle_vec_parts_begin(lle_vec* v, int32_t n_parts, const int8_t* actions_host, float* reward_host, uint8_t* done_host, void* after_stream) {
    if (!v || !actions_host) return fail(LLE_INVALID_ARGUMENT, "null argument");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    if (v->shadow) return fail(LLE_INVALID_ARGUMENT, "lle_vec_parts_*: not with a state_type observation (its second pass is ordered by whole launches)");
    // parts are cut over the tickets that hold real envs; the padding tickets behind N (N_pad is a multiple of 32) join the last part
    const int64_t tickets = (v->N + v->group - 1) / v->group;
    if (n_parts < 1 || n_parts > 1024) return fail(LLE_INVALID_ARGUMENT, "n_parts must be in 1..1024");
    n_parts = (int32_t)std::min<int64_t>(n_parts, tickets);  // at least one ticket per part: fewer parts than asked for (lle_vec_parts_count)
    LLE_CUDA(cudaSetDevice(v->device));
    if (int rc = pipeline_setup(v)) return rc;
    void* a = device_view(v, actions_host);
    void* r = reward_host ? device_view(v, reward_host) : nullptr;
    void* d = done_host ? device_view(v, done_host) : nullptr;
    if (!a || (reward_host && !r) || (done_host && !d))
        return fail(LLE_INVALID_ARGUMENT, "lle_vec_parts_begin needs pinned (page-locked) host buffers (lle_host_alloc / cudaHostAlloc / cudaHostRegister)");
    if (n_parts > v->parts_cap) {
        if (v->h_part_out) cudaFreeHost(v->h_part_out);
        if (v->d_part_in) cudaFree(v->d_part_in);
        if (v->d_part_count) cudaFree(v->d_part_count);
        v->h_part_out = v->d_part_in = v->d_part_count = nullptr;
        v->parts_cap = 0;
        LLE_CUDA(cudaMalloc((void**)&v->d_part_in, (size_t)n_parts * 32 * sizeof(uint32_t)));
        LLE_CUDA(cudaMalloc((void**)&v->d_part_count, (size_t)n_parts * sizeof(uint32_t)));
        LLE_CUDA(cudaHostAlloc((void**)&v->h_part_out, (size_t)n_parts * 32 * sizeof(uint32_t), cudaHostAllocMapped));
        LLE_CUDA(cudaHostGetDevicePointer((void**)&v->d_part_out, v->h_part_out, 0));
        v->parts_cap = n_parts;
    }
    if (after_stream != LLE_STREAM_NONE) {  // order the loop after the caller's stream
        LLE_CUDA(cudaEventRecord(v->ev_user, (cudaStream_t)after_stream));
        LLE_CUDA(cudaStreamWaitEvent(v->s_main, v->ev_user, 0));
    }
    LLE_CUDA(cudaMemsetAsync(v->d_part_in, 0, (size_t)n_parts * 32 * sizeof(uint32_t), v->s_main));
    LLE_CUDA(cudaMemsetAsync(v->d_part_count, 0, (size_t)n_parts * sizeof(uint32_t), v->s_main));
    LLE_CUDA(cudaStreamSynchronize(v->s_main));
    std::memset(v->h_part_out, 0, (size_t)n_parts * 32 * sizeof(uint32_t));
    __sync_synchronize();
    v->parts_tpp = (uint32_t)((tickets + n_parts - 1) / n_parts);
    v->parts_n = (int)((tickets + v->parts_tpp - 1) / v->parts_tpp);  // the last part may be shorter; never an empty one
    v->parts_launched = 0;
    v->parts_fed.assign((size_t)v->parts_n, 0);
    v->parts_read.assign((size_t)v->parts_n, 0);
    v->parts_actions_dev = (const int8_t*)a;
    v->parts_reward = (float*)r;
    v->parts_done = (uint8_t*)d;
    return LLE_OK;
}

int lle_vec_parts_count(lle_vec* v, int32_t* n_parts) {
    if (!v || !n_parts) return fail(LLE_INVALID_ARGUMENT, "null argument");
    *n_parts = v->parts_n;
    return LLE_OK;
}

int lle_vec_parts_range(lle_vec* v, int32_t part, int64_t* first_env, int64_t* n_envs) {
    if (!v || !first_env || !n_envs) return fail(LLE_INVALID_ARGUMENT, "null argument");
    if (!v->parts_n || part < 0 || part >= v->parts_n) return fail(LLE_INDEX_ERROR, "no such part (or no parts loop open)");
    const int64_t lo = (int64_t)part * v->parts_tpp * v->group;
    const int64_t hi = part == v->parts_n - 1 ? v->N : std::min<int64_t>(v->N, lo + (int64_t)v->parts_tpp * v->group);
    *first_env = lo;
    *n_envs = hi - lo;
    return LLE_OK;
}

int lle_vec_parts_launch(lle_vec* v) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (!v->parts_n) return fail(LLE_INVALID_ARGUMENT, "no parts loop open: call lle_vec_parts_begin first");
    uint64_t oldest = v->parts_launched;
    for (uint64_t r : v->parts_read) oldest = std::min(oldest, r);
    if (v->parts_launched - oldest >= 4) return fail(LLE_INVALID_ARGUMENT, "four steps in flight: wait for the parts of the oldest one before launching another");
    LLE_CUDA(cudaSetDevice(v->device));
    KParams p = base_params(v);
    p.mode = MODE_STEP;
    p.actions_in = v->parts_actions_dev;
    p.reward2 = v->parts_reward;
    p.done2 = v->parts_done;
    p.part_in = v->d_part_in;
    p.part_out = v->d_part_out;
    p.part_count = v->d_part_count;
    p.part_tickets = v->parts_tpp;
    p.part_last = (uint32_t)(v->parts_n - 1);
    p.in_need = p.out_value = (uint32_t)(v->parts_launched + 1);
    LLE_CUDA(launch(v, p, v->s_main));
    v->launches++;
    v->t++;
    v->parts_launched++;
    return LLE_OK;
}

int lle_vec_parts_feed(lle_vec* v, int32_t part) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (!v->parts_n || part < 0 || part >= v->parts_n) return fail(LLE_INDEX_ERROR, "no such part (or no parts loop open)");
    if (v->parts_fed[(size_t)part] != v->parts_read[(size_t)part])
        return fail(LLE_INVALID_ARGUMENT, "the part's previous step has not been waited for: its actions may still be read");
    // The step kernel reads the part's actions in place (pinned host memory, L1 bypassed): the host's stores are complete before
    // the stream memory operation that releases them.  (A staging copy per part on the copy stream was measured too: one more
    // driver call per part and 91-99 us per step instead of 84-88.)
    __sync_synchronize();
    const uint32_t n = (uint32_t)(v->parts_fed[(size_t)part] + 1);
    if (g_write_value32((CUstream)v->s_in, (CUdeviceptr)(uintptr_t)(v->d_part_in + (size_t)part * 32), n, CU_STREAM_WRITE_VALUE_DEFAULT) != CUDA_SUCCESS)
        return fail(LLE_CUDA_ERROR, "cuStreamWriteValue32 failed");
    v->parts_fed[(size_t)part]++;
    return LLE_OK;
}

int lle_vec_parts_wait(lle_vec* v, int32_t part) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (!v->parts_n || part < 0 || part >= v->parts_n) return fail(LLE_INDEX_ERROR, "no such part (or no parts loop open)");
    const uint64_t need = v->parts_read[(size_t)part] + 1;
    if (v->parts_fed[(size_t)part] < need) return fail(LLE_INVALID_ARGUMENT, "nothing to wait for: feed the part first");
    if (v->parts_launched < need) return fail(LLE_INVALID_ARGUMENT, "nothing to wait for: the step has not been launched (lle_vec_parts_launch)");
    volatile uint32_t* flag = v->h_part_out + (size_t)part * 32;
    const uint32_t n = (uint32_t)need;
    for (uint64_t spins = 0; (int32_t)(*flag - n) < 0; ++spins) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0xFFFFF) == 0xFFFFF) {
            cudaSetDevice(v->device);
            cudaError_t e = cudaStreamQuery(v->s_main);
            if (e != cudaSuccess && e != cudaErrorNotReady) return fail(LLE_CUDA_ERROR, std::string("step kernel failed: ") + cudaGetErrorString(e));
            if (e == cudaSuccess && (int32_t)(*flag - n) < 0) return fail(LLE_CUDA_ERROR, "the step retired without publishing the part");
        }
    }
    __sync_synchronize();
    v->parts_read[(size_t)part]++;
    return LLE_OK;
}

// Releases whatever a launched step is still waiting for (the actions it then reads are whatever the buffer holds), drains the
// streams and closes the loop: for error paths and lle_vec_destroy, so that no kernel is left spinning on the device.
int lle_vec_parts_abort(lle_vec* v) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (!v->parts_n) return LLE_OK;
    LLE_CUDA(cudaSetDevice(v->device));
    for (int k = 0; k < v->parts_n; ++k)
        if (v->parts_fed[(size_t)k] < v->parts_launched &&
            g_write_value32((CUstream)v->s_in, (CUdeviceptr)(uintptr_t)(v->d_part_in + (size_t)k * 32), (uint32_t)v->parts_launched, CU_STREAM_WRITE_VALUE_DEFAULT) != CUDA_SUCCESS)
            return fail(LLE_CUDA_ERROR, "cuStreamWriteValue32 failed");
    LLE_CUDA(cudaStreamSynchronize(v->s_in));
    LLE_CUDA(cudaStreamSynchronize(v->s_main));
    v->parts_n = 0;
    return LLE_OK;
}

int lle_vec_parts_end(lle_vec* v) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    if (!v->parts_n) return LLE_OK;
    for (int k = 0; k < v->parts_n; ++k)
        if (v->parts_fed[(size_t)k] != v->parts_launched || v->parts_read[(size_t)k] != v->parts_launched)
            return fail(LLE_INVALID_ARGUMENT, "every launched step must be fed and waited for on every part before the loop ends (a launched step waits for its actions on the device)");
    LLE_CUDA(cudaSetDevice(v->device));
    LLE_CUDA(cudaStreamSynchronize(v->s_in));
    LLE_CUDA(cudaStreamSynchronize(v->s_main));
    v->parts_n = 0;
    return LLE_OK;
}

int lle_vec_set_state(lle_vec* v, const int32_t* pos_dev, const uint8_t* gems_dev, const uint8_t* alive_dev, void* stream) {
    if (!v || !pos_dev || !alive_dev || (v->G > 0 && !gems_dev)) return fail(LLE_INVALID_ARGUMENT, "null argument");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    LLE_CUDA(cudaSetDevice(v->device));
    KParams p = base_params(v);
    p.mode = MODE_SET_STATE;
    p.ss_pos = pos_dev; p.ss_gems = gems_dev; p.ss_alive = alive_dev;
    LLE_CUDA(launch(v, p, (cudaStream_t)stream));
    v->launches++;
    LLE_SYNC_SHADOW(v, stream);
    return LLE_OK;
}


int lle_vec_export_raw(lle_vec* v, int16_t* pos, uint8_t* alive, uint8_t* arrived, uint8_t* slot, uint64_t* beam_on,
                       uint64_t* collected, uint8_t* counters, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    RawState r;
    std::memset(&r, 0, sizeof r);
    r.pos = pos; r.alive = alive; r.arrived = arrived; r.slot = slot; r.beam_on = v->NBmax ? beam_on : nullptr; r.collected = collected; r.counters = counters;
    return raw_state_launch<false>(v, r, stream);
}

int lle_vec_export_raw_state(lle_vec* v, const lle_raw_state* dst, void* stream) {
    if (!v || !dst) return fail(LLE_INVALID_ARGUMENT, "null argument");
    return raw_state_launch<false>(v, raw_of(dst, v->NBmax), stream);
}

int lle_vec_import_raw_state(lle_vec* v, const lle_raw_state* src, void* stream) {
    if (!v || !src) return fail(LLE_INVALID_ARGUMENT, "null argument");
    if (v->pipe_submitted != v->pipe_completed || v->parts_n) return fail(LLE_INVALID_ARGUMENT, "pipelined steps outstanding: drain with lle_vec_pipeline_wait (or close the parts loop with lle_vec_parts_end) first");
    if (!src->pos || !src->alive || !src->arrived || !src->slot || !src->counters || !src->avail_cache || (v->G && !src->collected) ||
        (v->NBmax && !src->beam_on) || (v->JE && !src->subgoals_extras) || (v->opts.pbrs && !src->subgoals_pbrs))
        return fail(LLE_INVALID_ARGUMENT, "lle_vec_import_raw_state needs every array of the engine record this vec keeps");
    v->last_was_step = false;  // the import is an ordinary launch: the next step must not overlap it
    if (int rc = raw_state_launch<true>(v, raw_of(src, v->NBmax), stream)) return rc;
    return lle_vec_refresh(v, stream);
}

int lle_vec_get_reset_count(lle_vec* v, uint32_t* out) { if (!v || !out) return fail(LLE_INVALID_ARGUMENT, "null"); *out = v->reset_epoch; return LLE_OK; }
int lle_vec_set_reset_count(lle_vec* v, uint32_t value) { if (!v) return fail(LLE_INVALID_ARGUMENT, "null"); v->reset_epoch = value; return LLE_OK; }

int lle_vec_debug_timeline(lle_vec* v, uint64_t* out_host, int64_t cap_warps, int64_t* n_warps) {
    if (!v || !n_warps) return fail(LLE_INVALID_ARGUMENT, "null argument");
    *n_warps = v->d_timeline ? (int64_t)v->grid * kWarps : 0;
    if (v->d_timeline && out_host) {
        LLE_CUDA(cudaSetDevice(v->device));
        LLE_CUDA(cudaDeviceSynchronize());
        LLE_CUDA(cudaMemcpy(out_host, v->d_timeline, (size_t)std::min<int64_t>(cap_warps, *n_warps) * 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    }
    return LLE_OK;
}

int lle_vec_set_seed(lle_vec* v, uint64_t seed) { if (!v) return fail(LLE_INVALID_ARGUMENT, "null"); v->opts.seed = seed; return LLE_OK; }
int lle_vec_get_step_count(lle_vec* v, uint64_t* out) { if (!v || !out) return fail(LLE_INVALID_ARGUMENT, "null"); *out = v->t; return LLE_OK; }
int lle_vec_set_step_count(lle_vec* v, uint64_t value) { if (!v) return fail(LLE_INVALID_ARGUMENT, "null"); v->t = value; return LLE_OK; }
int lle_vec_launch_count(lle_vec* v, uint64_t* out) { if (!v || !out) return fail(LLE_INVALID_ARGUMENT, "null"); *out = v->launches; return LLE_OK; }

int lle_vec_timing_begin(lle_vec* v, void* stream) {
    if (!v) return fail(LLE_INVALID_ARGUMENT, "null vec");
    LLE_CUDA(cudaSetDevice(v->device));
    v->timing_launches0 = v->launches;
    LLE_CUDA(cudaEventRecord(v->ev0, (cudaStream_t)stream));
    return LLE_OK;
}
int lle_vec_timing_end(lle_vec* v, void* stream, float* total_ms, uint64_t* launches) {
    if (!v || !total_ms) return fail(LLE_INVALID_ARGUMENT, "null argument");
    LLE_CUDA(cudaSetDevice(v->device));
    LLE_CUDA(cudaEventRecord(v->ev1, (cudaStream_t)stream));
    LLE_CUDA(cudaEventSynchronize(v->ev1));
    LLE_CUDA(cudaEventElapsedTime(total_ms, v->ev0, v->ev1));
    if (launches) *launches = v->launches - v->timing_launches0;
    return LLE_OK;
}

}  // extern "C"
