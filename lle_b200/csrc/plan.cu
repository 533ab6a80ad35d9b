// lle_b200 — the device planner (include/lle_b200.h: lle_plan): exact shortest death-free joint plans, one map per CTA.
//
// The search and its rules are plan_core.cuh's; this file runs it level-synchronously inside a CTA.  A persistent grid takes
// maps by atomic ticket.  Per depth, the CTA's threads share the (frontier entry, joint action) pairs of the depth: each copies
// the entry's record into its own shared-memory column, steps it (TinyWorld, tiny_core.cuh), claims the successor's key in the
// map's dense claim table with a 64-bit atomicMin, and appends the successor to the next frontier when its claim was the first
// of the key.  The claim table and both frontier queues sit in shared memory when the map's K is small enough (the 5x5
// two-agent maps of the generated batches need about 20 KB), otherwise in a slab of global memory owned by the CTA.  At the
// end of the depth that reaches a goal, one thread walks the parents back from the smallest goal key.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/lle_b200.h"
#include "map_compiler.hpp"
#include "plan_core.cuh"

namespace lle {

int fail(int code, const std::string& msg);  // vec_world.cu: sets lle_last_error

namespace {

constexpr int kPlanThreads = 256;
constexpr int kPlanRecWords = 8;                          // record columns: [8][kPlanThreads] words
constexpr size_t kPlanSmemScratchMax = 64 * 1024;         // claim table + queues of a map searched in shared memory
constexpr size_t kPlanSlabBudget = size_t(8) << 30;       // global scratch of all CTAs together (at most)

struct PlanMapDev {
    const uint8_t* blob;
    const uint16_t* cell_index;
    TinyLayout L;
    int32_t W, n_cells, n_words, in_smem;
    uint32_t K;
    int32_t out;  // index of the map in the caller's arrays
};

struct PlanParams {
    const PlanMapDev* maps;
    uint32_t n_maps;
    int32_t max_steps;
    uint32_t all_gems;
    uint32_t* ticket;
    uint8_t* slab;
    size_t slab_bytes;  // per CTA
    int32_t* length;
    int64_t* n_states;
    int8_t* actions;    // [n][max_steps][4], filled with -1 by the host
};

struct PlanColumn {  // word k of this thread's record: a column of shared memory
    uint32_t* base;
    __device__ __forceinline__ uint32_t& operator()(int word) const { return base[word * kPlanThreads]; }
};

size_t plan_scratch_bytes(uint32_t K, int n_words) { return (size_t)K * 8 + 2 * (size_t)K * (size_t)(1 + n_words) * 4; }

}  // namespace

// Three CTAs per SM: 77-80 registers and no spills for every A_ (without a minimum, ptxas picks 64 registers and spills)
template <int A_>
__global__ void __launch_bounds__(kPlanThreads, 3) lle_plan_kernel(const PlanParams p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint32_t* cols = reinterpret_cast<uint32_t*>(smem_raw);
    uint8_t* sscratch = smem_raw + kPlanRecWords * kPlanThreads * 4;
    __shared__ uint32_t s_map, s_n_cur, s_n_next, s_new, s_goal;
    __shared__ int s_done;
    constexpr uint32_t J = A_ == 1 ? 5 : A_ == 2 ? 25 : A_ == 3 ? 125 : 625;
    const int tid = threadIdx.x;
    uint8_t* gscratch = p.slab ? p.slab + (size_t)blockIdx.x * p.slab_bytes : nullptr;
    PlanWorld<A_, PlanColumn> pw;
    pw.w.rec = PlanColumn{cols + tid};
    pw.all_gems = p.all_gems != 0;
    for (;;) {
        if (tid == 0) s_map = atomicAdd(p.ticket, 1u);
        __syncthreads();
        const uint32_t t = s_map;
        if (t >= p.n_maps) break;
        const PlanMapDev md = p.maps[t];
        const int nw = md.n_words, ew = 1 + nw;
        uint64_t* table = reinterpret_cast<uint64_t*>(md.in_smem ? sscratch : gscratch);
        uint32_t* queue[2] = {reinterpret_cast<uint32_t*>(table + md.K), reinterpret_cast<uint32_t*>(table + md.K) + (size_t)md.K * ew};
        pw.w.L = md.L;
        pw.w.W = md.W;
        pw.w.bind(md.blob);
        pw.cell_index = md.cell_index;
        pw.n_cells = (uint32_t)md.n_cells;
        for (uint32_t i = tid; i < md.K; i += kPlanThreads) table[i] = kPlanEmpty;
        __syncthreads();
        int64_t states = 1;  // thread 0's running count
        if (tid == 0) {
            const uint32_t k0 = pw.reset();
            table[k0] = 0;
            s_n_cur = 0; s_n_next = 0; s_new = 0; s_goal = 0xFFFFFFFFu; s_done = 0;
            pw.w.unpack();
            if (pw.goal()) {
                p.length[md.out] = 0;
                s_done = 1;
            } else if (pw.w.n_arrived == (uint32_t)A_) {
                p.length[md.out] = -1;
                s_done = 1;
            } else {
                queue[0][0] = k0;
                for (int q = 0; q < nw; ++q) queue[0][1 + q] = pw.w.rec(q);
                s_n_cur = 1;
            }
        }
        __syncthreads();
        for (int depth = 0; !s_done; ++depth) {
            const uint32_t* cur = queue[depth & 1];
            uint32_t* nxt = queue[(depth & 1) ^ 1];
            const uint32_t n_items = s_n_cur * J;
            for (uint32_t item = tid; item < n_items; item += kPlanThreads) {
                const uint32_t e = item / J, j = item - e * J;
                const uint32_t* ent = cur + (size_t)e * ew;
                for (int q = 0; q < nw; ++q) pw.w.rec(q) = ent[1 + q];
                uint32_t k;
                if (!pw.expand(j, &k)) continue;
                const unsigned long long old =
                    atomicMin(reinterpret_cast<unsigned long long*>(table + k), (unsigned long long)plan_claim((uint32_t)depth + 1, ent[0], j));
                if (old != kPlanEmpty) continue;
                atomicAdd(&s_new, 1u);
                if (pw.goal()) {
                    atomicMin(&s_goal, k);
                    continue;
                }
                if (pw.w.n_arrived == (uint32_t)A_) continue;
                uint32_t* out = nxt + (size_t)atomicAdd(&s_n_next, 1u) * ew;
                out[0] = k;
                for (int q = 0; q < nw; ++q) out[1 + q] = pw.w.rec(q);
            }
            __syncthreads();
            if (tid == 0) {
                states += s_new;
                s_new = 0;
                if (s_goal != 0xFFFFFFFFu) {
                    p.length[md.out] = depth + 1;
                    plan_walk_back(table, s_goal, depth + 1, A_, p.actions + (size_t)md.out * p.max_steps * 4);
                    s_done = 1;
                } else if (s_n_next == 0 || depth + 1 >= p.max_steps) {
                    p.length[md.out] = -1;
                    s_done = 1;
                }
                s_n_cur = s_n_next;
                s_n_next = 0;
            }
            __syncthreads();
        }
        if (tid == 0) p.n_states[md.out] = states;
    }
}

}  // namespace lle

using namespace lle;

#define LLE_PLAN_CUDA(expr)                                                                                                  \
    do {                                                                                                                     \
        cudaError_t _e = (expr);                                                                                             \
        if (_e != cudaSuccess)                                                                                               \
            return fail(_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver ? LLE_NO_DEVICE : LLE_CUDA_ERROR,       \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                                 \
    } while (0)

namespace {

struct DeviceAllocs {  // everything lle_plan allocates on the device, freed on every way out
    std::vector<void*> ptrs;
    template <class T>
    cudaError_t alloc(T** p, size_t bytes) {
        void* q = nullptr;
        const cudaError_t e = cudaMalloc(&q, bytes ? bytes : 1);
        if (e == cudaSuccess) ptrs.push_back(q);
        *p = static_cast<T*>(q);
        return e;
    }
    ~DeviceAllocs() {
        for (void* q : ptrs) cudaFree(q);
    }
};

using PlanKernel = void (*)(PlanParams);
const PlanKernel kPlanKernels[LLE_PLAN_MAX_AGENTS] = {lle_plan_kernel<1>, lle_plan_kernel<2>, lle_plan_kernel<3>, lle_plan_kernel<4>};

}  // namespace

// lle_plan (vec_world.cu) once the handles are unwrapped
int lle::plan_run(const CompiledMap* const* maps, int32_t n_maps, int32_t max_steps, uint32_t flags, int32_t device, int32_t* length,
                  int64_t* n_states, int8_t* actions) {
    if (n_maps < 0 || (n_maps > 0 && (!length || !n_states || !actions))) return fail(LLE_INVALID_ARGUMENT, "lle_plan: null argument");
    if (max_steps < 1 || max_steps > LLE_PLAN_MAX_STEPS) return fail(LLE_INVALID_ARGUMENT, "lle_plan: max_steps must be in [1, 1024]");
    if (flags & ~(uint32_t)LLE_PLAN_ALL_GEMS) return fail(LLE_INVALID_ARGUMENT, "lle_plan: unknown flag");
    if (device < 0) return fail(LLE_INVALID_ARGUMENT, "lle_plan: negative device ordinal");
    const bool all_gems = (flags & LLE_PLAN_ALL_GEMS) != 0;
    std::vector<PlanSpec> specs((size_t)n_maps);
    for (int m = 0; m < n_maps; ++m) {
        const char* why = "";
        const int rc = plan_prepare(maps[m]->blob.data(), all_gems, specs[(size_t)m], &why);
        if (rc != LLE_OK) return fail(rc, "lle_plan: map " + std::to_string(m) + ": " + why);
    }
    if (n_maps == 0) return LLE_OK;

    LLE_PLAN_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    LLE_PLAN_CUDA(cudaGetDeviceProperties(&prop, device));
    // one upload of every blob and cell-index table (16-byte aligned pieces), then one launch per agent count
    std::vector<size_t> blob_off((size_t)n_maps), ci_off((size_t)n_maps);
    size_t bytes = 0;
    for (int m = 0; m < n_maps; ++m) {
        blob_off[(size_t)m] = bytes;
        bytes += (maps[m]->blob.size() + 15) / 16 * 16;
        ci_off[(size_t)m] = bytes;
        bytes += (specs[(size_t)m].cell_index.size() * 2 + 15) / 16 * 16;
    }
    std::vector<uint8_t> host(bytes, 0);
    for (int m = 0; m < n_maps; ++m) {
        std::memcpy(host.data() + blob_off[(size_t)m], maps[m]->blob.data(), maps[m]->blob.size());
        std::memcpy(host.data() + ci_off[(size_t)m], specs[(size_t)m].cell_index.data(), specs[(size_t)m].cell_index.size() * 2);
    }
    DeviceAllocs dev;
    uint8_t* d_tables = nullptr;
    PlanMapDev* d_maps = nullptr;
    uint32_t* d_tickets = nullptr;
    int32_t* d_length = nullptr;
    int64_t* d_states = nullptr;
    int8_t* d_actions = nullptr;
    const size_t act_bytes = (size_t)n_maps * (size_t)max_steps * 4;
    LLE_PLAN_CUDA(dev.alloc(&d_tables, bytes));
    LLE_PLAN_CUDA(dev.alloc(&d_maps, sizeof(PlanMapDev) * (size_t)n_maps));
    LLE_PLAN_CUDA(dev.alloc(&d_tickets, sizeof(uint32_t) * LLE_PLAN_MAX_AGENTS));
    LLE_PLAN_CUDA(dev.alloc(&d_length, sizeof(int32_t) * (size_t)n_maps));
    LLE_PLAN_CUDA(dev.alloc(&d_states, sizeof(int64_t) * (size_t)n_maps));
    LLE_PLAN_CUDA(dev.alloc(&d_actions, act_bytes));
    LLE_PLAN_CUDA(cudaMemcpy(d_tables, host.data(), bytes, cudaMemcpyHostToDevice));
    LLE_PLAN_CUDA(cudaMemset(d_tickets, 0, sizeof(uint32_t) * LLE_PLAN_MAX_AGENTS));
    LLE_PLAN_CUDA(cudaMemset(d_actions, 0xFF, act_bytes));

    // maps grouped by agent count (the kernel's template argument), in the caller's order within a group
    std::vector<PlanMapDev> md;
    int first[LLE_PLAN_MAX_AGENTS + 1] = {0};
    for (int A = 1; A <= LLE_PLAN_MAX_AGENTS; ++A) {
        first[A - 1] = (int)md.size();
        for (int m = 0; m < n_maps; ++m) {
            const PlanSpec& s = specs[(size_t)m];
            if (s.A != A) continue;
            PlanMapDev d;
            d.blob = d_tables + blob_off[(size_t)m];
            d.cell_index = reinterpret_cast<const uint16_t*>(d_tables + ci_off[(size_t)m]);
            d.L = s.L;
            d.W = s.W; d.n_cells = s.n_cells; d.n_words = s.n_words;
            d.K = (uint32_t)s.K;
            d.in_smem = plan_scratch_bytes(d.K, s.n_words) <= kPlanSmemScratchMax;
            d.out = m;
            md.push_back(d);
        }
    }
    first[LLE_PLAN_MAX_AGENTS] = (int)md.size();
    LLE_PLAN_CUDA(cudaMemcpy(d_maps, md.data(), sizeof(PlanMapDev) * md.size(), cudaMemcpyHostToDevice));

    for (int A = 1; A <= LLE_PLAN_MAX_AGENTS; ++A) {
        const int n = first[A] - first[A - 1];
        if (n == 0) continue;
        size_t smem_scratch = 0, slab = 0;
        for (int q = first[A - 1]; q < first[A]; ++q) {
            const size_t b = plan_scratch_bytes(md[(size_t)q].K, md[(size_t)q].n_words);
            if (md[(size_t)q].in_smem) smem_scratch = std::max(smem_scratch, b);
            else slab = std::max(slab, (b + 255) / 256 * 256);
        }
        const size_t smem = (size_t)kPlanRecWords * kPlanThreads * 4 + smem_scratch;
        const PlanKernel kern = kPlanKernels[A - 1];
        LLE_PLAN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        LLE_PLAN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kPlanThreads, smem));
        int64_t grid = std::min<int64_t>(n, (int64_t)prop.multiProcessorCount * std::max(1, per_sm));
        uint8_t* d_slab = nullptr;
        if (slab) {
            size_t free_b = 0, total_b = 0;
            LLE_PLAN_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const size_t budget = std::min(kPlanSlabBudget, free_b / 2);
            grid = std::min<int64_t>(grid, std::max<int64_t>(1, (int64_t)(budget / slab)));
            LLE_PLAN_CUDA(dev.alloc(&d_slab, slab * (size_t)grid));
        }
        PlanParams p;
        p.maps = d_maps + first[A - 1];
        p.n_maps = (uint32_t)n;
        p.max_steps = max_steps;
        p.all_gems = all_gems ? 1u : 0u;
        p.ticket = d_tickets + (A - 1);
        p.slab = d_slab;
        p.slab_bytes = slab;
        p.length = d_length;
        p.n_states = d_states;
        p.actions = d_actions;
        kern<<<(unsigned)grid, kPlanThreads, smem>>>(p);
        LLE_PLAN_CUDA(cudaGetLastError());
    }
    LLE_PLAN_CUDA(cudaDeviceSynchronize());
    LLE_PLAN_CUDA(cudaMemcpy(length, d_length, sizeof(int32_t) * (size_t)n_maps, cudaMemcpyDeviceToHost));
    LLE_PLAN_CUDA(cudaMemcpy(n_states, d_states, sizeof(int64_t) * (size_t)n_maps, cudaMemcpyDeviceToHost));
    LLE_PLAN_CUDA(cudaMemcpy(actions, d_actions, act_bytes, cudaMemcpyDeviceToHost));
    return LLE_OK;
}
