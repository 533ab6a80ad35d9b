// lle_b200 — the device expert (include/lle_b200.h: lle_vec_expert_*): exact distance-to-goal tables for every map of a vec, and
// the optimal joint action of every world from its current engine record.
//
// The rules are expert_core.cuh's.  The build runs over all maps at once:
//   seed       one thread per map steps World::reset and claims the reset key; the reset states are entries 0 .. n_maps-1 of
//              one global state array (map, key, record).
//   forward    one launch per depth.  A work item is a (frontier entry, joint action) pair; the frontier of a depth is the
//              contiguous slice of the state array appended by the depth before, whatever the map, so a batch of a thousand
//              small maps and one map with millions of states both fill the device.  A successor claims its key in its map's
//              table with atomicCAS; the first claimer appends (map, key, record) with a warp-aggregated atomicAdd.
//   backward   one launch per level over the open states (collected from the state array once, compacted after each level):
//              a thread scans the joint actions of its state in increasing order and resolves it with one 32-bit store.
// A query is one thread per world: key from the record (through the vec's layout), one table load, A action bytes.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/lle_b200.h"
#include "expert_core.cuh"
#include "map_compiler.hpp"

namespace lle {

int fail(int code, const std::string& msg);  // vec_world.cu: sets lle_last_error

namespace {

constexpr int kExpertThreads = 256;
constexpr int kExpertRecWords = 8;  // record columns: [8][kExpertThreads] words of shared memory

struct ExpertMapDev {
    const uint8_t* blob;
    const uint16_t* cell_index;  // [H*W]
    uint32_t* table;             // [K] words (expert_core.cuh)
    TinyLayout L;
    int32_t W, n_cells, n_words;
    uint32_t K;
};

struct ExpertColumn {  // word k of this thread's record: a column of shared memory
    uint32_t* base;
    __device__ __forceinline__ uint32_t& operator()(int word) const { return base[word * kExpertThreads]; }
};

struct ExpertBuildParams {
    const ExpertMapDev* maps;
    uint32_t n_maps;
    uint32_t all_gems;
    uint32_t* states;       // [capacity][ew]: map, key, record words
    int32_t ew;
    uint32_t lo, hi;        // forward: the frontier [lo, hi) of the state array
    uint32_t* n_total;      // forward: entries of the state array
    uint32_t* n_per_map;    // forward: reached states of every map
    const uint32_t* open_in;  // backward: state indices still open, n_open of them
    uint32_t n_open;
    uint32_t* open_out;     // backward / collect: the states left open
    uint32_t* n_open_out;
    uint32_t level;         // backward: d
};

struct ExpertActParams {
    const ExpertMapDev* maps;
    const uint32_t* records;
    const int32_t* map_of_env;
    int64_t N;
    int32_t stride, w_flags, w_gems, use_gems;  // use_gems: the key has the gem mask on top (all_gems and the map has gems)
    int32_t W;
    int8_t* actions;
    int32_t* dist;
};

template <int A_>
__device__ __forceinline__ void bind_map(PlanWorld<A_, ExpertColumn>& pw, const ExpertMapDev& md) {
    pw.w.L = md.L;
    pw.w.W = md.W;
    pw.w.bind(md.blob);
    pw.cell_index = md.cell_index;
    pw.n_cells = (uint32_t)md.n_cells;
}

// The lanes of a warp whose `take` is set get consecutive slots of *counter (one atomicAdd per warp); every lane of the warp calls it
__device__ __forceinline__ uint32_t warp_append(bool take, uint32_t* counter, uint32_t* slot) {
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, take);
    if (!ballot) return 0;
    const uint32_t lane = threadIdx.x & 31u, leader = (uint32_t)__ffs(ballot) - 1u;
    uint32_t first = 0;
    if (lane == leader) first = atomicAdd(counter, (uint32_t)__popc(ballot));
    first = __shfl_sync(0xFFFFFFFFu, first, (int)leader);
    *slot = first + (uint32_t)__popc(ballot & ((1u << lane) - 1u));
    return ballot;
}

}  // namespace

// Three CTAs per SM for the kernels that step records (without a minimum, ptxas caps them at 64 registers and some spill)
template <int A_>
__global__ void __launch_bounds__(kExpertThreads, 3) lle_expert_seed_kernel(const ExpertBuildParams p) {
    __shared__ uint32_t cols[kExpertRecWords * kExpertThreads];
    const uint32_t m = blockIdx.x * kExpertThreads + threadIdx.x;
    if (m >= p.n_maps) return;
    PlanWorld<A_, ExpertColumn> pw;
    pw.w.rec = ExpertColumn{cols + threadIdx.x};
    pw.all_gems = p.all_gems != 0;
    const ExpertMapDev md = p.maps[m];
    bind_map(pw, md);
    const uint32_t k0 = pw.reset();
    pw.w.unpack();
    md.table[k0] = expert_first_word(pw);
    uint32_t* out = p.states + (size_t)m * p.ew;
    out[0] = m;
    out[1] = k0;
    for (int q = 0; q < md.n_words; ++q) out[2 + q] = pw.w.rec(q);
    p.n_per_map[m] = 1;
}

template <int A_>
__global__ void __launch_bounds__(kExpertThreads, 3) lle_expert_forward_kernel(const ExpertBuildParams p) {
    __shared__ uint32_t cols[kExpertRecWords * kExpertThreads];
    constexpr uint32_t J = expert_joint_count(A_);
    PlanWorld<A_, ExpertColumn> pw;
    pw.w.rec = ExpertColumn{cols + threadIdx.x};
    pw.all_gems = p.all_gems != 0;
    const uint64_t n_items = (uint64_t)(p.hi - p.lo) * J;
    const uint64_t stride = (uint64_t)gridDim.x * kExpertThreads;
    // warp-uniform trip count: every lane reaches the ballot of warp_append
    for (uint64_t base = (uint64_t)blockIdx.x * kExpertThreads + (threadIdx.x & ~31u); base < n_items; base += stride) {
        const uint64_t item = base + (threadIdx.x & 31u);
        bool fresh = false;
        uint32_t m = 0, k = 0;
        int nw = 0;
        if (item < n_items) {
            const uint32_t e = p.lo + (uint32_t)(item / J), j = (uint32_t)(item % J);
            const uint32_t* ent = p.states + (size_t)e * p.ew;
            m = ent[0];
            const ExpertMapDev md = p.maps[m];
            nw = md.n_words;
            // a state where every agent has arrived is not expanded
            if (((ent[2 + md.L.w_flags] >> 24) & 0xFu) != (uint32_t)A_) {
                bind_map(pw, md);
                for (int q = 0; q < nw; ++q) pw.w.rec(q) = ent[2 + q];
                if (pw.expand(j, &k)) fresh = atomicCAS(md.table + k, kExpertEmpty, expert_first_word(pw)) == kExpertEmpty;
            }
        }
        uint32_t slot;
        if (warp_append(fresh, p.n_total, &slot) && fresh) {
            uint32_t* out = p.states + (size_t)slot * p.ew;
            out[0] = m;
            out[1] = k;
            for (int q = 0; q < nw; ++q) out[2 + q] = pw.w.rec(q);
            atomicAdd(p.n_per_map + m, 1u);
        }
    }
}

// the open states of the whole state array (the first input of the backward levels)
__global__ void __launch_bounds__(kExpertThreads) lle_expert_collect_kernel(const ExpertBuildParams p) {
    const uint32_t stride = gridDim.x * kExpertThreads;
    for (uint32_t base = blockIdx.x * kExpertThreads + (threadIdx.x & ~31u); base < p.n_open; base += stride) {
        const uint32_t e = base + (threadIdx.x & 31u);
        bool open = false;
        if (e < p.n_open) {
            const uint32_t* ent = p.states + (size_t)e * p.ew;
            open = p.maps[ent[0]].table[ent[1]] == kExpertOpen;
        }
        uint32_t slot;
        if (warp_append(open, p.n_open_out, &slot) && open) p.open_out[slot] = e;
    }
}

template <int A_>
__global__ void __launch_bounds__(kExpertThreads, 3) lle_expert_backward_kernel(const ExpertBuildParams p) {
    __shared__ uint32_t cols[kExpertRecWords * kExpertThreads];
    PlanWorld<A_, ExpertColumn> pw;
    pw.w.rec = ExpertColumn{cols + threadIdx.x};
    pw.all_gems = p.all_gems != 0;
    const uint32_t stride = gridDim.x * kExpertThreads;
    for (uint32_t base = blockIdx.x * kExpertThreads + (threadIdx.x & ~31u); base < p.n_open; base += stride) {
        const uint32_t idx = base + (threadIdx.x & 31u);
        bool still = false;
        uint32_t e = 0;
        if (idx < p.n_open) {
            e = p.open_in[idx];
            const uint32_t* ent = p.states + (size_t)e * p.ew;
            const ExpertMapDev md = p.maps[ent[0]];
            bind_map(pw, md);
            const uint32_t w = expert_resolve(pw, md.table, p.level, [&] {
                for (int q = 0; q < md.n_words; ++q) pw.w.rec(q) = ent[2 + q];
            });
            if (w == kExpertOpen) still = true;
            else md.table[ent[1]] = w;  // holds `level`, never level - 1: no other item of this launch reads it as a match
        }
        uint32_t slot;
        if (warp_append(still, p.n_open_out, &slot) && still) p.open_out[slot] = e;
    }
}

// the states still open after the last level that resolved something: no death-free way to a goal
__global__ void __launch_bounds__(kExpertThreads) lle_expert_close_kernel(const ExpertBuildParams p) {
    const uint32_t idx = blockIdx.x * kExpertThreads + threadIdx.x;
    if (idx >= p.n_open) return;
    const uint32_t* ent = p.states + (size_t)p.open_in[idx] * p.ew;
    p.maps[ent[0]].table[ent[1]] = kExpertNone;
}

template <int A_>
__global__ void __launch_bounds__(kExpertThreads) lle_expert_act_kernel(const ExpertActParams p) {
    const int64_t e = (int64_t)blockIdx.x * kExpertThreads + threadIdx.x;
    if (e >= p.N) return;
    const uint32_t* rec = p.records + e * p.stride;
    const ExpertMapDev& md = p.maps[p.map_of_env ? p.map_of_env[e] : 0];
    int32_t dist = -2;
    uint32_t j = 0;
    if ((rec[p.w_flags] & 0xFFu) == (1u << A_) - 1u) {  // a world with a dead agent is in no table
        uint32_t k = p.use_gems ? rec[p.w_gems] : 0u;
        bool standable = true;
        LLE_UNROLL
        for (int a = A_ - 1; a >= 0; --a) {
            const uint32_t w = rec[a >> 1];
            const uint32_t q = (a & 1) ? (w >> 16) : (w & 0xFFFFu);
            const uint32_t c = md.cell_index[(q >> 8) * (uint32_t)p.W + (q & 0xFFu)];
            standable = standable && c != 0xFFFFu;
            k = k * (uint32_t)md.n_cells + c;
        }
        if (standable && k < md.K) {
            const uint32_t w = md.table[k];
            dist = expert_dist(w);
            j = w & 1023u;
        }
    }
    int8_t* act = p.actions + e * A_;
    LLE_UNROLL
    for (int a = 0; a < A_; ++a) {
        act[a] = dist > 0 ? (int8_t)(j % 5u) : (int8_t)4;
        j /= 5u;
    }
    if (p.dist) p.dist[e] = dist;
}

}  // namespace lle

using namespace lle;

#define LLE_EXPERT_CUDA(expr)                                                                                                \
    do {                                                                                                                     \
        cudaError_t _e = (expr);                                                                                             \
        if (_e != cudaSuccess)                                                                                               \
            return fail(_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver ? LLE_NO_DEVICE : LLE_CUDA_ERROR,       \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                                 \
    } while (0)

struct lle::ExpertTables {
    int device = 0, A = 0;
    bool all_gems = false;
    std::vector<int64_t> K;
    std::vector<size_t> table_off;  // words
    uint32_t* d_tables = nullptr;
    uint16_t* d_cell_index = nullptr;
    ExpertMapDev* d_maps = nullptr;
    ~ExpertTables() {
        cudaFree(d_tables);
        cudaFree(d_cell_index);
        cudaFree(d_maps);
    }
};

void lle::expert_free(ExpertTables* t) { delete t; }

namespace {

struct ScratchAllocs {  // the build's temporary device memory, freed on every way out
    std::vector<void*> ptrs;
    template <class T>
    cudaError_t alloc(T** p, size_t bytes) {
        void* q = nullptr;
        const cudaError_t e = cudaMalloc(&q, bytes ? bytes : 1);
        if (e == cudaSuccess) ptrs.push_back(q);
        *p = static_cast<T*>(q);
        return e;
    }
    ~ScratchAllocs() {
        for (void* q : ptrs) cudaFree(q);
    }
};

struct ExpertKernels {
    void (*seed)(ExpertBuildParams);
    void (*forward)(ExpertBuildParams);
    void (*backward)(ExpertBuildParams);
    void (*act)(ExpertActParams);
};
const ExpertKernels kExpertKernels[LLE_PLAN_MAX_AGENTS] = {
    {lle_expert_seed_kernel<1>, lle_expert_forward_kernel<1>, lle_expert_backward_kernel<1>, lle_expert_act_kernel<1>},
    {lle_expert_seed_kernel<2>, lle_expert_forward_kernel<2>, lle_expert_backward_kernel<2>, lle_expert_act_kernel<2>},
    {lle_expert_seed_kernel<3>, lle_expert_forward_kernel<3>, lle_expert_backward_kernel<3>, lle_expert_act_kernel<3>},
    {lle_expert_seed_kernel<4>, lle_expert_forward_kernel<4>, lle_expert_backward_kernel<4>, lle_expert_act_kernel<4>},
};

unsigned grid_for(uint64_t items, int max_blocks) {
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((items + kExpertThreads - 1) / kExpertThreads, (uint64_t)max_blocks));
}

}  // namespace

int lle::expert_build(const ExpertVecView& v, uint32_t flags, int64_t* n_states, void* stream, ExpertTables** out) {
    const bool all_gems = (flags & LLE_PLAN_ALL_GEMS) != 0;
    const int n_maps = (int)v.maps.size();
    std::vector<PlanSpec> specs((size_t)n_maps);
    int nw_max = 0;
    uint64_t keys = 0;
    for (int m = 0; m < n_maps; ++m) {
        const char* why = "";
        const int rc = plan_prepare(v.maps[(size_t)m]->blob.data(), all_gems, specs[(size_t)m], &why);
        if (rc != LLE_OK) return fail(rc, "lle_vec_expert_build: map " + std::to_string(m) + ": " + why);
        nw_max = std::max(nw_max, specs[(size_t)m].n_words);
        keys += (uint64_t)specs[(size_t)m].K;
    }
    // the state array holds the reached set of every map: at most sum K entries, indexed by 32-bit words
    const int ew = 2 + nw_max;
    const size_t cells = (size_t)v.maps[0]->H * (size_t)v.maps[0]->W;
    const size_t scratch = (size_t)keys * ((size_t)ew + 2) * 4;  // state array + two open lists
    const size_t keep = (size_t)keys * 4 + (size_t)n_maps * cells * 2 + sizeof(ExpertMapDev) * (size_t)n_maps;
    if (keys >= (uint64_t(1) << 32)) return fail(LLE_LIMIT_EXCEEDED, "lle_vec_expert_build: the maps have 2^32 joint states or more together");
    LLE_EXPERT_CUDA(cudaSetDevice(v.device));
    size_t free_b = 0, total_b = 0;
    LLE_EXPERT_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if (scratch + keep > free_b)
        return fail(LLE_LIMIT_EXCEEDED, "lle_vec_expert_build: the tables and the state array (" + std::to_string((scratch + keep) >> 20) +
                                            " MB) do not fit the free device memory (" + std::to_string(free_b >> 20) + " MB)");

    cudaStream_t s = (cudaStream_t)stream;
    auto t = std::unique_ptr<ExpertTables>(new ExpertTables());
    t->device = v.device;
    t->A = v.A;
    t->all_gems = all_gems;
    std::vector<uint16_t> ci((size_t)n_maps * cells);
    size_t off = 0;
    for (int m = 0; m < n_maps; ++m) {
        t->K.push_back(specs[(size_t)m].K);
        t->table_off.push_back(off);
        off += (size_t)specs[(size_t)m].K;
        std::memcpy(ci.data() + (size_t)m * cells, specs[(size_t)m].cell_index.data(), cells * 2);
    }
    LLE_EXPERT_CUDA(cudaMalloc((void**)&t->d_tables, std::max<size_t>(off, 1) * 4));
    LLE_EXPERT_CUDA(cudaMalloc((void**)&t->d_cell_index, ci.size() * 2));
    LLE_EXPERT_CUDA(cudaMalloc((void**)&t->d_maps, sizeof(ExpertMapDev) * (size_t)n_maps));
    std::vector<ExpertMapDev> md((size_t)n_maps);
    for (int m = 0; m < n_maps; ++m) {
        const PlanSpec& sp = specs[(size_t)m];
        ExpertMapDev& d = md[(size_t)m];
        d.blob = v.blobs[(size_t)m];
        d.cell_index = t->d_cell_index + (size_t)m * cells;
        d.table = t->d_tables + t->table_off[(size_t)m];
        d.L = sp.L;
        d.W = sp.W; d.n_cells = sp.n_cells; d.n_words = sp.n_words;
        d.K = (uint32_t)sp.K;
    }
    LLE_EXPERT_CUDA(cudaMemcpyAsync(t->d_cell_index, ci.data(), ci.size() * 2, cudaMemcpyHostToDevice, s));
    LLE_EXPERT_CUDA(cudaMemcpyAsync(t->d_maps, md.data(), sizeof(ExpertMapDev) * md.size(), cudaMemcpyHostToDevice, s));
    LLE_EXPERT_CUDA(cudaMemsetAsync(t->d_tables, 0xFF, off * 4, s));

    ScratchAllocs tmp;
    uint32_t *d_states = nullptr, *d_open[2] = {nullptr, nullptr}, *d_counts = nullptr, *d_per_map = nullptr;
    LLE_EXPERT_CUDA(tmp.alloc(&d_states, (size_t)keys * (size_t)ew * 4));
    LLE_EXPERT_CUDA(tmp.alloc(&d_open[0], (size_t)keys * 4));
    LLE_EXPERT_CUDA(tmp.alloc(&d_open[1], (size_t)keys * 4));
    LLE_EXPERT_CUDA(tmp.alloc(&d_counts, 2 * 4));  // [0] entries of the state array, [1] open states written by the last launch
    LLE_EXPERT_CUDA(tmp.alloc(&d_per_map, (size_t)n_maps * 4));
    const ExpertKernels& k = kExpertKernels[v.A - 1];
    int sms = 0, per_sm_fwd = 0, per_sm_bwd = 0;
    LLE_EXPERT_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, v.device));
    LLE_EXPERT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_fwd, k.forward, kExpertThreads, 0));
    LLE_EXPERT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_bwd, k.backward, kExpertThreads, 0));
    const int max_fwd = sms * std::max(1, per_sm_fwd), max_bwd = sms * std::max(1, per_sm_bwd);

    ExpertBuildParams p;
    std::memset(&p, 0, sizeof p);
    p.maps = t->d_maps;
    p.n_maps = (uint32_t)n_maps;
    p.all_gems = all_gems ? 1u : 0u;
    p.states = d_states;
    p.ew = ew;
    p.n_total = d_counts;
    p.n_per_map = d_per_map;
    p.n_open_out = d_counts + 1;
    const uint32_t n0 = (uint32_t)n_maps;
    LLE_EXPERT_CUDA(cudaMemcpyAsync(d_counts, &n0, 4, cudaMemcpyHostToDevice, s));
    k.seed<<<grid_for((uint64_t)n_maps, 1 << 20), kExpertThreads, 0, s>>>(p);
    LLE_EXPERT_CUDA(cudaGetLastError());
    // forward: one launch per depth over the slice appended by the depth before
    uint32_t counts[2] = {0, 0};
    for (uint32_t lo = 0, hi = n0; lo < hi;) {
        p.lo = lo;
        p.hi = hi;
        k.forward<<<grid_for((uint64_t)(hi - lo) * expert_joint_count(v.A), max_fwd), kExpertThreads, 0, s>>>(p);
        LLE_EXPERT_CUDA(cudaGetLastError());
        LLE_EXPERT_CUDA(cudaMemcpyAsync(counts, d_counts, 4, cudaMemcpyDeviceToHost, s));
        LLE_EXPERT_CUDA(cudaStreamSynchronize(s));
        lo = hi;
        hi = counts[0];
    }
    const uint32_t n_total = counts[0];
    // backward: the open states, then one launch per level until a level resolves nothing
    LLE_EXPERT_CUDA(cudaMemsetAsync(d_counts + 1, 0, 4, s));
    p.n_open = n_total;
    p.open_out = d_open[0];
    lle_expert_collect_kernel<<<grid_for(n_total, max_bwd * 4), kExpertThreads, 0, s>>>(p);
    LLE_EXPERT_CUDA(cudaGetLastError());
    LLE_EXPERT_CUDA(cudaMemcpyAsync(counts + 1, d_counts + 1, 4, cudaMemcpyDeviceToHost, s));
    LLE_EXPERT_CUDA(cudaStreamSynchronize(s));
    uint32_t n_open = counts[1];
    int cur = 0;
    for (uint32_t d = 1; n_open > 0; ++d) {
        LLE_EXPERT_CUDA(cudaMemsetAsync(d_counts + 1, 0, 4, s));
        p.open_in = d_open[cur];
        p.n_open = n_open;
        p.open_out = d_open[cur ^ 1];
        p.level = d;
        k.backward<<<grid_for(n_open, max_bwd), kExpertThreads, 0, s>>>(p);
        LLE_EXPERT_CUDA(cudaGetLastError());
        LLE_EXPERT_CUDA(cudaMemcpyAsync(counts + 1, d_counts + 1, 4, cudaMemcpyDeviceToHost, s));
        LLE_EXPERT_CUDA(cudaStreamSynchronize(s));
        cur ^= 1;
        if (counts[1] == n_open) break;  // nothing resolved: the rest has no way to a goal
        n_open = counts[1];
    }
    if (n_open > 0) {
        p.open_in = d_open[cur];
        p.n_open = n_open;
        lle_expert_close_kernel<<<grid_for(n_open, 1 << 20), kExpertThreads, 0, s>>>(p);
        LLE_EXPERT_CUDA(cudaGetLastError());
    }
    std::vector<uint32_t> per_map((size_t)n_maps);
    LLE_EXPERT_CUDA(cudaMemcpyAsync(per_map.data(), d_per_map, (size_t)n_maps * 4, cudaMemcpyDeviceToHost, s));
    LLE_EXPERT_CUDA(cudaStreamSynchronize(s));
    if (n_states)
        for (int m = 0; m < n_maps; ++m) n_states[m] = per_map[(size_t)m];
    *out = t.release();
    return LLE_OK;
}

int lle::expert_act(const ExpertVecView& v, const ExpertTables* t, int8_t* actions, int32_t* dist, void* stream) {
    LLE_EXPERT_CUDA(cudaSetDevice(v.device));
    ExpertActParams p;
    p.maps = t->d_maps;
    p.records = v.records;
    p.map_of_env = v.map_of_env;
    p.N = v.N;
    p.stride = v.L.stride;
    p.w_flags = v.L.w_flags;
    p.w_gems = v.L.w_gems;
    p.use_gems = t->all_gems && v.L.gem_words > 0 ? 1 : 0;
    p.W = v.W;
    p.actions = actions;
    p.dist = dist;
    const unsigned blocks = (unsigned)((v.N + kExpertThreads - 1) / kExpertThreads);
    kExpertKernels[v.A - 1].act<<<blocks, kExpertThreads, 0, (cudaStream_t)stream>>>(p);
    LLE_EXPERT_CUDA(cudaGetLastError());
    return LLE_OK;
}

int lle::expert_table(const ExpertTables* t, int32_t map_index, int32_t* dist, int16_t* joint, int64_t cap, int64_t* n_keys) {
    const int64_t K = t->K[(size_t)map_index];
    *n_keys = K;
    const int64_t n = std::min(K, cap);
    if (n <= 0 || (!dist && !joint)) return LLE_OK;
    LLE_EXPERT_CUDA(cudaSetDevice(t->device));
    std::vector<uint32_t> words((size_t)n);
    LLE_EXPERT_CUDA(cudaMemcpy(words.data(), t->d_tables + t->table_off[(size_t)map_index], (size_t)n * 4, cudaMemcpyDeviceToHost));
    expert_decode(words.data(), n, dist, joint);
    return LLE_OK;
}
