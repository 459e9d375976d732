// C ABI of libfmc_b200.so (include/fmc.h): context, forest specialisation/upload, the tree-predict
// kernel launch and the persistent simulation kernel launch.  No CPU fallback anywhere: every
// compute entry point launches a kernel or fails.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "fmc_sim.cuh"
#include "fmc_sim_memo.cuh"

using namespace fmc;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(FMC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
    } while (0)

// ---------------------------------------------------------------------------------------------
// tree-predict kernel: one lane per row, all lanes of a warp walk the same trees
// ---------------------------------------------------------------------------------------------
struct PredictArgs {
    const double *rows;     // [n][17]
    double *out;            // [n][n_outputs]
    long long n;
    uint32_t win_lo, win_hi;
    const uint4 *stream;
    const uint2 *consts;
    uint32_t stream_off[8], consts_off[8], n_groups[8];
    int n_outputs, n_num, multi_window;
    int zero_is_missing;
    double base[8];
    int n_scaled;
    int scaler_cols[16];
    double scaler_mean[16], scaler_scale[16];
    unsigned long long *stats;   // [2]: warp-level node gathers, lane-level node gathers of live rows (roofline accounting)
};

constexpr int kPredThreads = 256;
constexpr int kPredChunkFloats = kPredRows * 32;

template <bool SKL>
__global__ void __launch_bounds__(kPredThreads) predict_kernel(const PredictArgs a) {
    __shared__ float rows[(kPredThreads / 32) * kPredChunkFloats];   // [warp][feature][lane]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float inf = __int_as_float(0x7f800000);
    for (int i = tid; i < (kPredThreads / 32) * 32; i += kPredThreads)
        rows[(i >> 5) * kPredChunkFloats + kPredNinfRow * 32 + (i & 31)] = -inf;
    unsigned long long steps = 0ULL, visits = 0ULL;
    for (long long base = (long long)blockIdx.x * kPredThreads; base < a.n; base += (long long)gridDim.x * kPredThreads) {
        for (int i = tid; i < kPredThreads * kNumMax; i += kPredThreads) {
            const int r = i / kNumMax, k = i - r * kNumMax;
            const long long idx = base + r;
            if (idx >= a.n || k >= a.n_num) continue;
            double x = a.rows[idx * kNumMax + k];
            for (int j = 0; j < a.n_scaled; ++j)
                if (a.scaler_cols[j] == k) x = (x - a.scaler_mean[j]) / a.scaler_scale[j];
            const float v = (float)x;
            const bool flag = (k == 3 || k == 12 || k == 13 || k == 14 || k == 16);
            float *col = rows + (r >> 5) * kPredChunkFloats + (r & 31);
            if (SKL) {
                col[k * 32] = v;
            } else if (flag) {
                // 0/1 flags have no B view: a missing flag of a CSR-fed booster is an absent one (the host entry points
                // reject NaN flags for the dense-fed boosters)
                col[k * 32] = (x != x) ? 0.f : v;
            } else {
                // xgboost: NaN is missing, and so is an exact zero for the CSR-fed boosters -> A view -inf (default-left
                // nodes), B view +inf (default-right nodes); the B views follow the 17 numerics in the order of the non-flags
                int nb = kNumMax;
                for (int q = 0; q < k; ++q) nb += !(q == 3 || q == 12 || q == 13 || q == 14 || q == 16);
                const bool miss = (x != x) || (a.zero_is_missing && v == 0.f);
                col[k * 32] = miss ? -inf : v;
                col[nb * 32] = miss ? inf : v;
            }
        }
        __syncthreads();
        const bool live = base + tid < a.n;
        const uint32_t fcol = (uint32_t)__cvta_generic_to_shared(rows + warp * kPredChunkFloats + lane);
        for (int o = 0; o < a.n_outputs; ++o) {
            ForestView F;
            F.win_lo = a.win_lo; F.win_hi = a.win_hi;
            F.stream = a.stream + a.stream_off[o];
            F.consts = a.consts + a.consts_off[o];
            F.n_groups = a.n_groups[o];
            F.multi_window = a.multi_window != 0;
            uint32_t levels;
            const double v = a.multi_window ? walk_output<SKL, true>(F, fcol, lane, a.base[o], levels)
                                            : walk_output<SKL, false>(F, fcol, lane, a.base[o], levels);
            if (live) a.out[(base + tid) * a.n_outputs + o] = v;
            steps += (unsigned long long)levels * kIlp;
            visits += live ? (unsigned long long)levels * kIlp : 0ULL;
        }
        __syncthreads();
    }
    if (a.stats) {
        if (lane == 0) atomicAdd(a.stats, steps);
        for (int s = 16; s >= 1; s >>= 1) visits += __shfl_xor_sync(0xFFFFFFFFu, visits, s);
        if (lane == 0) atomicAdd(a.stats + 1, visits);
    }
}

// ---------------------------------------------------------------------------------------------
// Device placement of packed forests: node tables go into 1 MiB-aligned windows (a table never
// straddles a window, see fmc_pack.hpp), root streams and constants side streams are concatenated.
// ---------------------------------------------------------------------------------------------
struct TablePlacement {
    uint64_t window_addr;                 // device address of the table's window
    uint32_t stream_off[8], consts_off[8], n_groups[8];   // in uint4 / uint2 / groups
};

struct TableArena {
    std::vector<uint64_t> h_nodes, h_stream, h_consts;
    std::vector<size_t> win_index;        // window of each placed table, resolved to an address at upload
    char *d_raw = nullptr, *d_nodes = nullptr;
    uint4 *d_stream = nullptr;
    uint2 *d_consts = nullptr;
    size_t cap_nodes = 0, cap_stream = 0, cap_consts = 0;

    void clear() { h_nodes.clear(); h_stream.clear(); h_consts.clear(); win_index.clear(); }
    // Relocates `pf` to its place and appends it; returns the table id.
    int place(PackedForest &pf, TablePlacement &pl) {
        size_t cursor = (h_nodes.size() * 8 + 127) / 128 * 128;
        const size_t bytes = pf.slots.size() * 8;
        // a table of at most one window must not straddle a window boundary; larger tables start on one (their
        // groups were laid out against 1 MiB boundaries of the table by the packer)
        if (bytes > kWindowBytes || cursor % kWindowBytes + bytes > kWindowBytes)
            cursor = (cursor + kWindowBytes - 1) / kWindowBytes * kWindowBytes;
        pf.relocate((uint32_t)(cursor % kWindowBytes));
        h_nodes.resize(cursor / 8, 0);
        h_nodes.insert(h_nodes.end(), pf.slots.begin(), pf.slots.end());
        while (h_stream.size() % 2) h_stream.push_back(0);
        const size_t s0 = h_stream.size(), c0 = h_consts.size();
        h_stream.insert(h_stream.end(), pf.stream.begin(), pf.stream.end());
        h_consts.insert(h_consts.end(), pf.consts.begin(), pf.consts.end());
        for (int k = 0; k < 8; ++k) {
            pl.stream_off[k] = (uint32_t)((s0 + pf.stream_off[k]) / 2);
            pl.consts_off[k] = (uint32_t)(c0 + pf.consts_off[k]);
            pl.n_groups[k] = pf.n_groups[k];
        }
        win_index.push_back(cursor / kWindowBytes);
        pl.window_addr = 0;
        return (int)win_index.size() - 1;
    }
    uint64_t window_addr(int table) const { return (uint64_t)(uintptr_t)d_nodes + win_index[table] * kWindowBytes; }
    cudaError_t upload(cudaStream_t st, bool sync_copy) {
        cudaError_t e;
        const size_t nb = h_nodes.size() * 8 + kWindowBytes, sb = (h_stream.size() + 2) * 8, cb = (h_consts.size() + 1) * 8;
        if (nb > cap_nodes) {
            cudaFree(d_raw); d_raw = nullptr; cap_nodes = 0;
            if ((e = cudaMalloc(&d_raw, nb)) != cudaSuccess) return e;
            cap_nodes = nb;
        }
        d_nodes = (char *)(((uintptr_t)d_raw + kWindowBytes - 1) / kWindowBytes * kWindowBytes);
        if (sb > cap_stream) {
            cudaFree(d_stream); d_stream = nullptr; cap_stream = 0;
            if ((e = cudaMalloc(&d_stream, sb)) != cudaSuccess) return e;
            cap_stream = sb;
        }
        if (cb > cap_consts) {
            cudaFree(d_consts); d_consts = nullptr; cap_consts = 0;
            if ((e = cudaMalloc(&d_consts, cb)) != cudaSuccess) return e;
            cap_consts = cb;
        }
        (void)st; (void)sync_copy;
        if (!h_nodes.empty() && (e = cudaMemcpy(d_nodes, h_nodes.data(), h_nodes.size() * 8, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
        if (!h_stream.empty() && (e = cudaMemcpy(d_stream, h_stream.data(), h_stream.size() * 8, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
        if (!h_consts.empty() && (e = cudaMemcpy(d_consts, h_consts.data(), h_consts.size() * 8, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
        return cudaSuccess;
    }
    void release() {
        cudaFree(d_raw); cudaFree(d_stream); cudaFree(d_consts);
        d_raw = d_nodes = nullptr; d_stream = nullptr; d_consts = nullptr;
        cap_nodes = cap_stream = cap_consts = 0;
    }
};

#ifdef FMC_DEBUG_CHECKS
static void debug_set_range(const TableArena &A) {
    const unsigned long long lo = (unsigned long long)(uintptr_t)A.d_nodes, hi = lo + A.h_nodes.size() * 8;
    cudaMemcpyToSymbol(g_dbg_lo, &lo, 8);
    cudaMemcpyToSymbol(g_dbg_hi, &hi, 8);
}
#endif

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
struct fmc_ctx {
    int device = 0;
    cudaDeviceProp prop;
    HostForest forest[FMC_N_MODELS];
    fmc_params params;
    std::vector<fmc_matchup> matchups;
    std::vector<fmc_game_state> starts;  // [n_matchups] start state of every entry (fmc_set_start_states), kickoff by default
    std::vector<fmc_team_usage> usage;   // [n_matchups][2] or empty (shipped configuration: every name "Unknown")
    struct NameRows { int8_t row[3][FMC_MAX_USAGE]; };
    std::vector<NameRows> name_rows;     // per team: the 0/1 feature row of every usage entry (-1: no model knows the name)
    int n_slots = 0;
    int n_prow = 0, n_trow = 0, n_rrow = 0;   // name rows the current usage tables need (max over the teams)
    fmc_player_rec *d_box_scratch = nullptr;   // running box of every resident lane [grid x threads][2][n_slots]
    size_t box_scratch_bytes = 0;
    bool tables_dirty = true;
    bool usage_pending = false;          // fmc_set_matchups kept the tables of an identical list; usage must be confirmed
    // device-side state of the last set_matchups
    TableArena sim_tables;
    MatchupDev *d_matchups = nullptr;
    std::vector<MatchupDev> h_matchups;  // host copy of d_matchups: the range and start words are patched here, then copied
    int n_specs = 0;                     // distinct specialisations of the current tables (memo ids 0 .. n_specs - 1)
    unsigned long long *d_next = nullptr;
    std::vector<unsigned long long> h_next;
    std::vector<int32_t> packed_slots;   // [n_matchups][FMC_N_MODELS][2]
    // exact memo (fmc_memo.hpp): rank specs of the current tables, table regions, mode
    RankSpec *d_specs = nullptr;         // [n_specs][kMemoFams][2]
    std::vector<uint8_t> memo_ok;        // [n_specs][kMemoFams][2] the forest's ranks fit the key
    std::vector<std::string> memo_why;   // why not, for diagnostics
    int memo_mode = 1, memo_max_trips = 8, memo_break_parked = 16, memo_break_waiting = kMemoThreads / 64;
    uint64_t memo_max_bytes = 0;
    char *d_memo = nullptr;
    size_t memo_bytes = 0;
    MemoRegion memo_region[kMemoFams];
    bool memo_valid = false;             // mode 2: the table belongs to the current node tables
    unsigned long long *d_pred_stats = nullptr;   // [2] node gathers of the fmc_tree_predict launches since the last reset
    cudaEvent_t ev_done = nullptr;       // completion of the last fmc_simulate launch
    bool launched = false;
    // fmc_simulate_host: device scratch + pinned staging, kept between calls
    struct Scratch { void *dev = nullptr; size_t dev_bytes = 0; };
    // 0..7 fmc_simulate_host's buffers, 8 the period rows of fmc_simulate_segments, 9..10 its host path, 11 the sequence
    // rows of fmc_simulate_markets, 12..13 its host path, 14..15 the host path of fmc_simulate_overtime
    Scratch scr[16];
    // pinned staging of the large device -> host copies of fmc_simulate_host (two buffers: the DMA of one chunk overlaps
    // the host copy of the previous one into the caller's pageable buffer)
    void *pin[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copy_ev[2] = {nullptr, nullptr};
    // fmc_tree_predict: packed + uploaded tables are kept per (model, tree range, hot columns) until the model
    // or its columns change -- a stream of predict calls on the same model re-uses them
    struct PredEntry {
        int id = -1, tb = 0, te = 0, c0 = 0, c1 = 0;
        uint64_t version = 0, last_use = 0;
        TableArena arena;
        TablePlacement pl;
        int table = 0;
        bool multi_window = false;
    };
    static constexpr int kPredEntries = 12;
    PredEntry pred[kPredEntries];
    uint64_t forest_version[FMC_N_MODELS] = {0};
    uint64_t pred_clock = 0;
};

extern "C" void fmc_destroy(fmc_ctx *c);
// inside fmc_create: a failing CUDA call must not leak the half-built context
#define CKC(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            fmc_destroy(c);                                                                        \
            return fail(FMC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
        }                                                                                          \
    } while (0)

extern "C" const char *fmc_last_error(void) { return g_err.c_str(); }
extern "C" int fmc_abi_version(void) { return FMC_ABI_VERSION; }

// the dynamic shared memory every instantiation of one hook mask (and overtime rule) may use
template <int HOOKS, bool OT = false>
static cudaError_t set_smem_limits() {
    cudaError_t e = cudaSuccess;
    auto set = [&](const void *f, size_t bytes) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    };
    set((const void *)sim_kernel<false, false, HOOKS, OT>, sim_smem_bytes(false));
    set((const void *)sim_kernel<true, false, HOOKS, OT>, sim_smem_bytes(false));
    set((const void *)sim_kernel<false, true, HOOKS, OT>, sim_smem_bytes(true));
    set((const void *)sim_kernel<true, true, HOOKS, OT>, sim_smem_bytes(true));
    set((const void *)sim_memo_kernel<false, HOOKS, OT>, sim_memo_smem_bytes());
    set((const void *)sim_memo_kernel<true, HOOKS, OT>, sim_memo_smem_bytes());
    return e;
}

extern "C" int fmc_create(int device, fmc_ctx **out) {
    if (!out) return fail(FMC_ERR_INVALID, "fmc_create: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(FMC_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                           " (libfmc_b200 has no CPU fallback)");
    if (device < 0 || device >= n) return fail(FMC_ERR_INVALID, "fmc_create: bad device index");
    fmc_ctx *c = new fmc_ctx();
    c->device = device;
    CKC(cudaSetDevice(device));
    CKC(cudaGetDeviceProperties(&c->prop, device));
    if (c->prop.major != 10) {
        std::string nm = c->prop.name;
        fmc_destroy(c);
        return fail(FMC_ERR_NO_DEVICE, "device '" + nm + "' is not sm_100 (this library is built for sm_100a only)");
    }
    std::memset(&c->params, 0, sizeof(c->params));
    c->params.play_temp = 1.0;
    c->params.pass_class = 1;
    c->params.qy_noise = 0.5;
    c->params.stage2_standin[0] = (double)0.78f;
    c->params.stage2_standin[1] = (double)0.05f;
    c->params.stage2_standin[2] = (double)0.17f;
    CKC(set_smem_limits<0>());
    // the instantiations with hooks: period outputs (fmc_simulate_segments), sequence outputs, both (fmc_simulate_markets)
    CKC(set_smem_limits<kHookPeriods>());
    CKC(set_smem_limits<kHookSequence>());
    CKC(set_smem_limits<kHookPeriods | kHookSequence>());
    CKC((set_smem_limits<0, true>()));      // overtime (fmc_simulate_overtime)
    CKC(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
    CKC(cudaMalloc(&c->d_pred_stats, 16));
    CKC(cudaMemset(c->d_pred_stats, 0, 16));
    std::memset(c->memo_region, 0, sizeof(c->memo_region));
    *out = c;
    return FMC_OK;
}

extern "C" void fmc_destroy(fmc_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    c->sim_tables.release();
    for (auto &e : c->pred) e.arena.release();
    cudaDeviceSynchronize();
    cudaFree(c->d_matchups); cudaFree(c->d_next); cudaFree(c->d_box_scratch);
    cudaFree(c->d_specs); cudaFree(c->d_memo); cudaFree(c->d_pred_stats);
    for (auto &q : c->scr) cudaFree(q.dev);
    for (int b = 0; b < 2; ++b) { if (c->pin[b]) cudaFreeHost(c->pin[b]); if (c->copy_ev[b]) cudaEventDestroy(c->copy_ev[b]); }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->ev_done) cudaEventDestroy(c->ev_done);
    delete c;
}

extern "C" int fmc_device_info(fmc_ctx *c, int32_t *sm_count, int32_t *smem_per_block, char *name, int32_t name_len) {
    if (!c) return fail(FMC_ERR_INVALID, "ctx is NULL");
    if (sm_count) *sm_count = c->prop.multiProcessorCount;
    if (smem_per_block) *smem_per_block = (int32_t)c->prop.sharedMemPerBlockOptin;
    if (name && name_len > 0) { std::strncpy(name, c->prop.name, name_len - 1); name[name_len - 1] = 0; }
    return FMC_OK;
}

extern "C" int fmc_load_forest(fmc_ctx *c, int32_t id, const fmc_forest_desc *d) {
    if (!c || !d || id < 0 || id >= FMC_N_MODELS) return fail(FMC_ERR_INVALID, "fmc_load_forest: bad argument");
    if (d->n_outputs < 1 || d->n_outputs > 8 || d->n_nodes <= 0 || d->n_trees <= 0 || d->n_num > kNumMax)
        return fail(FMC_ERR_INVALID, "fmc_load_forest: bad shape");
    if (!d->feat || !d->thr || !d->left || !d->right || !d->default_left || !d->value || !d->tree_root || !d->tree_out)
        return fail(FMC_ERR_INVALID, "fmc_load_forest: NULL array");
    for (int32_t i = 0; i < d->n_nodes; ++i) {
        const int32_t l = d->left[i], r = d->right[i];
        if (l < 0) continue;                                  // leaf
        if (l >= d->n_nodes || r < 0 || r >= d->n_nodes) return fail(FMC_ERR_INVALID, "fmc_load_forest: child index out of range");
        if (d->feat[i] < 0 || d->feat[i] >= d->n_features) return fail(FMC_ERR_INVALID, "fmc_load_forest: split column out of range");
    }
    for (int32_t t = 0; t < d->n_trees; ++t) {
        if (d->tree_root[t] < 0 || d->tree_root[t] >= d->n_nodes) return fail(FMC_ERR_INVALID, "fmc_load_forest: tree root out of range");
        if (d->tree_out[t] < 0 || d->tree_out[t] >= d->n_outputs) return fail(FMC_ERR_INVALID, "fmc_load_forest: tree output out of range");
    }
    if (d->num_base < 0 || d->n_num < 0 || d->num_base + d->n_num > d->n_features) return fail(FMC_ERR_INVALID, "fmc_load_forest: numeric columns out of range");
    const int32_t keep0 = c->forest[id].active[0], keep1 = c->forest[id].active[1];
    const bool had = c->forest[id].loaded;
    c->forest[id].assign(*d);
    c->forest_version[id]++;
    if (!had) { c->forest[id].active[0] = -1; c->forest[id].active[1] = -1; }
    else { c->forest[id].active[0] = keep0; c->forest[id].active[1] = keep1; }
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_set_scaler(fmc_ctx *c, int32_t id, int32_t n, const int32_t *cols, const double *mean, const double *scale) {
    if (!c || id < 0 || id >= FMC_N_MODELS || n < 0 || n > 16) return fail(FMC_ERR_INVALID, "fmc_set_scaler: bad argument");
    if (n > 0 && (!cols || !mean || !scale)) return fail(FMC_ERR_INVALID, "fmc_set_scaler: NULL array");
    for (int i = 0; i < n; ++i)
        if (cols[i] < 0 || cols[i] >= kNumMax) return fail(FMC_ERR_INVALID, "fmc_set_scaler: column outside the 17 numerics");
    HostForest &f = c->forest[id];
    f.n_scaled = n;
    for (int i = 0; i < n; ++i) { f.scaler_cols[i] = cols[i]; f.scaler_mean[i] = mean[i]; f.scaler_scale[i] = scale[i]; }
    c->forest_version[id]++;
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_set_active_columns(fmc_ctx *c, int32_t id, int32_t col0, int32_t col1) {
    if (!c || id < 0 || id >= FMC_N_MODELS) return fail(FMC_ERR_INVALID, "fmc_set_active_columns: bad argument");
    c->forest[id].active[0] = col0;
    c->forest[id].active[1] = col1;
    c->forest_version[id]++;
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_set_params(fmc_ctx *c, const fmc_params *p) {
    if (!c || !p) return fail(FMC_ERR_INVALID, "fmc_set_params: bad argument");
    if (p->policy < 0 || p->policy > 1 || p->sampler < 0 || p->sampler > 1 || p->stage2_mode < 0 || p->stage2_mode > 1)
        return fail(FMC_ERR_INVALID, "fmc_set_params: unknown mode");
    if (p->pass_class < 0 || p->pass_class > 4) return fail(FMC_ERR_INVALID, "fmc_set_params: pass_class out of range");
    c->params = *p;
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_set_memo(fmc_ctx *c, int32_t mode, uint64_t max_bytes, int32_t max_trips, int32_t break_parked) {
    if (!c || mode < 0 || mode > 2) return fail(FMC_ERR_INVALID, "fmc_set_memo: mode must be 0, 1 or 2");
    if (max_trips < 0 || max_trips > 4096 || break_parked < 0 || break_parked > 32) return fail(FMC_ERR_INVALID, "fmc_set_memo: bad scheduling knob");
    c->memo_mode = mode;
    c->memo_max_bytes = max_bytes;
    c->memo_max_trips = max_trips > 0 ? max_trips : 8;
    c->memo_break_parked = break_parked > 0 ? break_parked : 16;
    if (const char *e = std::getenv("FMC_MEMO_BREAK_WAITING")) { const int v = std::atoi(e); if (v > 0) c->memo_break_waiting = v; }
    c->memo_valid = false;
    return FMC_OK;
}

static fmc_game_state kickoff_state() {
    fmc_game_state s;
    std::memset(&s, 0, sizeof(s));
    s.offense = -1; s.seconds = 3600; s.down = 1; s.distance = 10.0; s.yards_to_goal = 75.0;
    return s;
}
static StartDev start_dev(const fmc_game_state &s) {
    StartDev d;
    std::memset(&d, 0, sizeof(d));
    d.dist = s.distance; d.ytg = s.yards_to_goal; d.sec = s.seconds; d.down = s.down; d.offense = s.offense;
    d.score[0] = s.score[0]; d.score[1] = s.score[1];
    return d;
}

extern "C" int fmc_set_matchups(fmc_ctx *c, int32_t n, const fmc_matchup *m) {
    if (!c || n <= 0 || !m) return fail(FMC_ERR_INVALID, "fmc_set_matchups: bad argument");
    for (int i = 0; i < n; ++i)
        if (m[i].game_end < m[i].game_begin) return fail(FMC_ERR_INVALID, "fmc_set_matchups: game_end < game_begin");
    // The same pairs again (only the game ranges may differ): the specialised tables, the rank specs and, in mode 2, the
    // memo stay valid -- a caller that simulates one matchup repeatedly (FMC:1739-1760 loops over seeds / weeks) pays the
    // specialisation once.  Only the three range words of every device record are refreshed.
    bool same = !c->tables_dirty && (int)c->matchups.size() == n && c->d_matchups != nullptr;
    for (int i = 0; same && i < n; ++i)
        same = std::memcmp(c->matchups[i].sp, m[i].sp, sizeof(m[i].sp)) == 0 &&
               c->matchups[i].coach_col[0] == m[i].coach_col[0] && c->matchups[i].coach_col[1] == m[i].coach_col[1] &&
               // a matchup that had no games has no tables (build_tables skips it)
               (c->matchups[i].game_end > c->matchups[i].game_begin || m[i].game_end == m[i].game_begin);
    // start states belong to a matchup list: every entry starts at the kickoff again
    c->starts.assign(n, kickoff_state());
    if (same) {
        CK(cudaSetDevice(c->device));
        CK(cudaDeviceSynchronize());           // a launch in flight reads the ranges
        for (int i = 0; i < n; ++i) {
            MatchupDev &M = c->h_matchups[i];
            M.game_begin = m[i].game_begin; M.game_end = m[i].game_end; M.out_offset = m[i].out_offset;
            M.start = start_dev(c->starts[i]);
        }
        CK(cudaMemcpy(c->d_matchups, c->h_matchups.data(), c->h_matchups.size() * sizeof(MatchupDev), cudaMemcpyHostToDevice));
        c->matchups.assign(m, m + n);
        c->usage_pending = !c->usage.empty();   // the caller must repeat fmc_set_usage (or clear it): checked there
        return FMC_OK;
    }
    c->matchups.assign(m, m + n);
    c->usage.clear();          // usage belongs to a matchup list: set it again after fmc_set_matchups
    c->name_rows.clear();
    c->n_slots = 0;
    c->usage_pending = false;
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_set_start_states(fmc_ctx *c, int32_t n, const fmc_game_state *states) {
    if (!c) return fail(FMC_ERR_INVALID, "fmc_set_start_states: ctx is NULL");
    if (n != (int)c->matchups.size()) return fail(FMC_ERR_INVALID, "fmc_set_start_states: n_matchups differs from the last fmc_set_matchups");
    std::vector<fmc_game_state> st(n, kickoff_state());
    if (states) {
        for (int i = 0; i < n; ++i) {
            const fmc_game_state &s = states[i];
            const std::string at = "fmc_set_start_states: entry " + std::to_string(i) + ": ";
            if (s.offense < -1 || s.offense > 1) return fail(FMC_ERR_INVALID, at + "offense must be -1, 0 or 1");
            if (s.seconds < 0 || s.seconds > 3600) return fail(FMC_ERR_INVALID, at + "seconds must be in 0..3600");
            if (s.down < 1 || s.down > 4) return fail(FMC_ERR_INVALID, at + "down must be in 1..4");
            if (s.score[0] < 0 || s.score[0] > 250 || s.score[1] < 0 || s.score[1] > 250)
                return fail(FMC_ERR_INVALID, at + "scores must be in 0..250");
            if (!std::isfinite(s.distance) || !(s.distance > 0.0) || s.distance > 100.0)
                return fail(FMC_ERR_INVALID, at + "distance must be finite and in (0, 100]");
            if (!(s.yards_to_goal > 0.0 && s.yards_to_goal < 100.0)) return fail(FMC_ERR_INVALID, at + "yards_to_goal must be in (0, 100)");
            if (s.reserved != 0) return fail(FMC_ERR_INVALID, at + "reserved must be 0");
            st[i] = s;
        }
    }
    if (st.size() == c->starts.size() && std::memcmp(st.data(), c->starts.data(), st.size() * sizeof(fmc_game_state)) == 0)
        return FMC_OK;                         // nothing changes (e.g. kickoff again after fmc_set_matchups)
    c->starts.swap(st);
    // the device records of the current tables get their new start words; dirty tables take them when they are built
    if (!c->tables_dirty && c->d_matchups && c->h_matchups.size() == (size_t)n) {
        CK(cudaSetDevice(c->device));
        CK(cudaDeviceSynchronize());           // a launch in flight reads the start words
        for (int i = 0; i < n; ++i) c->h_matchups[i].start = start_dev(c->starts[i]);
        CK(cudaMemcpy(c->d_matchups, c->h_matchups.data(), c->h_matchups.size() * sizeof(MatchupDev), cudaMemcpyHostToDevice));
    }
    return FMC_OK;
}

extern "C" int fmc_set_usage(fmc_ctx *c, int32_t n, const fmc_team_usage *teams, int32_t n_slots) {
    if (!c) return fail(FMC_ERR_INVALID, "fmc_set_usage: ctx is NULL");
    if (!teams) {
        if (!c->usage.empty()) c->tables_dirty = true;
        c->usage.clear(); c->name_rows.clear(); c->n_slots = 0; c->usage_pending = false;
        return FMC_OK;
    }
    if (n != (int)c->matchups.size()) return fail(FMC_ERR_INVALID, "fmc_set_usage: n_matchups differs from the last fmc_set_matchups");
    if (!c->tables_dirty && c->usage.size() == 2 * (size_t)n && c->n_slots == n_slots &&
        std::memcmp(c->usage.data(), teams, sizeof(fmc_team_usage) * 2 * (size_t)n) == 0) {
        c->usage_pending = false;              // the same tables again: nothing to rebuild
        return FMC_OK;
    }
    if (n_slots < 0 || n_slots > 3 * FMC_MAX_USAGE) return fail(FMC_ERR_INVALID, "fmc_set_usage: bad n_slots");
    std::vector<fmc_ctx::NameRows> rows(2 * (size_t)n);
    for (int i = 0; i < 2 * n; ++i)
        for (int r = 0; r < 3; ++r) {
            const fmc_usage &u = teams[i].role[r];
            if (u.n < 1 || u.n > FMC_MAX_USAGE) return fail(FMC_ERR_CAPACITY, "fmc_set_usage: a usage table must have 1.." + std::to_string(FMC_MAX_USAGE) + " entries");
            double tot = 0.0;
            int next_row = 0;
            const int cap = r == 0 ? FMC_MAX_PASSER_ROWS : FMC_MAX_NAME_ROWS;
            for (int e = 0; e < FMC_MAX_USAGE; ++e) rows[i].row[r][e] = -1;
            for (int e = 0; e < u.n; ++e) {
                if (!(u.share[e] >= 0.0) || !std::isfinite(u.share[e])) return fail(FMC_ERR_INVALID, "fmc_set_usage: shares must be finite and >= 0");
                if (u.slot[e] >= n_slots) return fail(FMC_ERR_INVALID, "fmc_set_usage: slot out of range");
                tot += u.share[e];
                bool known = false;      // some model has a one-hot column for this name
                for (int m = 0; m < FMC_N_MODELS; ++m) known = known || u.col[m][e] >= 0;
                if (known) {
                    if (next_row >= cap)
                        return fail(FMC_ERR_CAPACITY, "fmc_set_usage: more than " + std::to_string(cap) + " names of one role that the models have columns for");
                    rows[i].row[r][e] = (int8_t)next_row++;
                }
            }
            if (!(tot > 0.0)) return fail(FMC_ERR_INVALID, "fmc_set_usage: shares sum to zero");
        }
    c->usage.assign(teams, teams + 2 * (size_t)n);
    c->n_prow = c->n_trow = c->n_rrow = 0;
    for (size_t i = 0; i < rows.size(); ++i)
        for (int r = 0; r < 3; ++r) {
            int used = 0;
            for (int e = 0; e < FMC_MAX_USAGE; ++e) used = rows[i].row[r][e] + 1 > used ? rows[i].row[r][e] + 1 : used;
            int &dst = r == 0 ? c->n_prow : (r == 1 ? c->n_rrow : c->n_trow);
            if (used > dst) dst = used;
        }
    c->name_rows.swap(rows);
    c->n_slots = n_slots;
    c->usage_pending = false;
    c->tables_dirty = true;
    return FMC_OK;
}

// Dynamic one-hot columns of (family, team on offense): the sampled names of a play are feature rows
// (fmc_sim.cuh kDynRow0...), every other name column folds to 0.
static void dyn_columns(const fmc_team_usage &tu, const fmc_ctx::NameRows &nr, int fam, int n_prow, PackSpec &s) {
    s.n_dyn = 0;
    auto add = [&](int role, int row0) {
        const fmc_usage &u = tu.role[role];
        for (int e = 0; e < u.n; ++e)
            if (u.col[fam][e] >= 0) { s.dyn_col[s.n_dyn] = u.col[fam][e]; s.dyn_row[s.n_dyn] = (int8_t)(row0 + nr.row[role][e]); s.n_dyn++; }
    };
    if (fam == FMC_RUN_YARDS) add(1, kDynRow0);
    else if (fam != FMC_PLAY_MODEL) { add(0, kDynRow0); add(2, kDynRow0 + n_prow); }   // target rows follow the passer rows in use
}

static bool family_needed(const fmc_ctx *c, int fam) {
    if (fam == FMC_PASS_STAGE2) return c->params.stage2_mode == 1;
    if (fam == FMC_PLAY_MODEL) return c->params.policy == 1;
    return fam <= FMC_SACK_YARDS;
}

// What the specialisation of an entry's forests depends on: the SP+ ratings folded into them, the coaches' play-model
// columns and, in player mode, the usage tables and their name rows.  Entries with equal bytes here get the same tables.
static std::string spec_inputs(const fmc_ctx *c, int i) {
    const fmc_matchup &mu = c->matchups[i];
    std::string k(reinterpret_cast<const char *>(mu.sp), sizeof(mu.sp));
    k.append(reinterpret_cast<const char *>(mu.coach_col), sizeof(mu.coach_col));
    if (!c->usage.empty()) {
        k.append(reinterpret_cast<const char *>(&c->usage[(size_t)i * 2]), 2 * sizeof(fmc_team_usage));
        k.append(reinterpret_cast<const char *>(&c->name_rows[(size_t)i * 2]), 2 * sizeof(fmc_ctx::NameRows));
    }
    return k;
}

// Specialise + pack every needed forest for both orientations of every distinct specialisation; upload.  Entries with
// games whose specialisation inputs are equal share the tables, the rank specs and the memo id of the first of them.
static int build_tables(fmc_ctx *c) {
    if (c->matchups.empty()) return fail(FMC_ERR_INVALID, "fmc_set_matchups has not been called");
    for (int fam = 0; fam < kNumFam; ++fam)
        if (family_needed(c, fam) && !c->forest[fam].loaded)
            return fail(FMC_ERR_INVALID, "model " + std::to_string(fam) + " is required by the current fmc_params but not loaded");
    // a launch in flight still reads the tables, the matchup records and the work counters that are replaced below
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    c->memo_valid = false;
    const int n = (int)c->matchups.size();
    std::vector<MatchupDev> md(n);
    struct Pending { int matchup, fam, off, table; };
    std::vector<Pending> placed;
    TableArena &A = c->sim_tables;
    A.clear();
    c->packed_slots.assign((size_t)n * FMC_N_MODELS * 2, 0);
    // ---- the representative of every entry with games: the first entry with games specialised alike (itself for a
    // slate without repeated pairs); memo ids number the representatives in entry order
    std::vector<int> rep(n, -1), memo_id(n, 0), reps;
    {
        std::unordered_map<std::string, int> first;
        for (int i = 0; i < n; ++i) {
            // a matchup without games on this context (another rank owns it: api.slate_specs(shard="matchups")) is never
            // selected by the kernels, so it needs no tables: a rank specialises only the forests it will walk
            if (c->matchups[i].game_end == c->matchups[i].game_begin) continue;
            auto it = first.emplace(spec_inputs(c, i), i).first;
            rep[i] = it->second;
            if (rep[i] == i) { memo_id[i] = (int)reps.size(); reps.push_back(i); }
            else memo_id[i] = memo_id[rep[i]];
        }
    }
    c->n_specs = (int)reps.size();
    const int ns = c->n_specs;
    // ---- specialise + pack every (representative, orientation, family) forest; the jobs are independent, a slate
    // of hundreds of matchups is packed by all host threads
    struct Job { int matchup, off, fam; PackedForest pf; std::string err, memo_why; RankSpec spec; };
    std::vector<Job> jobs;
    for (int i : reps) {
        for (int off = 0; off < 2; ++off)
            for (int fam = 0; fam < kNumFam; ++fam)
                if (family_needed(c, fam)) { jobs.emplace_back(); jobs.back().matchup = i; jobs.back().off = off; jobs.back().fam = fam; }
    }
    auto run_job = [&](Job &j) {
        const fmc_matchup &mu = c->matchups[j.matchup];
        const int off = j.off, de = off ^ 1, fam = j.fam;
        const HostForest &f = c->forest[fam];
        PackSpec s;
        preset_sim(s);
        s.active[0] = f.active[0]; s.active[1] = f.active[1];
        if (!c->usage.empty()) {      // player mode: every name comes from the usage tables
            s.active[0] = -1; s.active[1] = -1;
            dyn_columns(c->usage[(size_t)j.matchup * 2 + off], c->name_rows[(size_t)j.matchup * 2 + off], fam, c->n_prow, s);
        }
        if (fam == FMC_PLAY_MODEL) { s.active[0] = mu.coach_col[off]; s.active[1] = -1; }
        s.fold_value[6] = 3.0; s.fold_value[7] = 3.0;    // timeouts are never spent (FMC:911-912)
        s.fold_value[8] = mu.sp[off][0]; s.fold_value[9] = mu.sp[off][1];
        s.fold_value[10] = mu.sp[de][2]; s.fold_value[11] = mu.sp[de][0];
        s.n_scaled = f.n_scaled;
        for (int k = 0; k < f.n_scaled; ++k) { s.scaler_cols[k] = f.scaler_cols[k]; s.scaler_mean[k] = f.scaler_mean[k]; s.scaler_scale[k] = f.scaler_scale[k]; }
        j.err = pack_forest(f, s, j.pf);
        if (j.err.empty() && fam < kMemoFams) {
            RankSpecInput in;
            in.xgb = f.kind == FMC_KIND_XGB;
            in.zm = in.xgb && f.zero_is_missing;
            in.play_model = fam == FMC_PLAY_MODEL;
            if (in.play_model)
                for (int k = 0; k < f.n_scaled; ++k) {
                    const int col = f.scaler_cols[k];
                    if (col >= 0 && col < 6) { in.pm_scaled[col] = 1; in.pm_mean[col] = f.scaler_mean[k]; in.pm_scale[col] = f.scaler_scale[k]; }
                }
            j.memo_why = build_rank_spec(j.pf.row_thr, in, j.spec);
        }
    };
    {
        unsigned nt = std::thread::hardware_concurrency();
        if (nt == 0) nt = 1;
        if (nt > 32) nt = 32;
        if (jobs.size() < 24) nt = 1;
        if (nt <= 1) {
            for (Job &j : jobs) run_job(j);
        } else {
            std::atomic<size_t> next{0};
            std::vector<std::thread> pool;
            for (unsigned t = 0; t < nt; ++t)
                pool.emplace_back([&]() { for (size_t k; (k = next.fetch_add(1)) < jobs.size();) run_job(jobs[k]); });
            for (auto &th : pool) th.join();
        }
    }
    for (int i = 0; i < n; ++i) {
        const fmc_matchup &mu = c->matchups[i];
        MatchupDev &M = md[i];
        std::memset(&M, 0, sizeof(M));
        M.game_begin = mu.game_begin; M.game_end = mu.game_end; M.out_offset = mu.out_offset;
        M.start = start_dev(c->starts[i]);
        M.memo_id = memo_id[i];
        for (int off = 0; off < 2; ++off) {
            const int de = off ^ 1;
            const double O = mu.sp[off][1], D = mu.sp[de][2];
            M.bias[off] = 0.12 * (O - D) / 40.0;                 // matchup_bias FMC:431-433
            M.ymul[off] = 1.0 + 0.10 * std::tanh((O - D) / 30.0);  // yardage_multiplier FMC:435-437
            M.mz[off] = (O - D) / 40.0;                          // mismatch_z FMC:440-442
            M.tanh35[off] = std::tanh((O - D) / 35.0);           // FMC:448, 456
            if (!c->usage.empty()) {
                const fmc_team_usage &tu = c->usage[(size_t)i * 2 + off];
                for (int r = 0; r < 3; ++r) {
                    const fmc_usage &u = tu.role[r];
                    UsageDev &U = M.usage[off];
                    U.n[r] = (int8_t)u.n;
                    double acc = 0.0;
                    for (int e = 0; e < u.n; ++e) { acc += u.share[e]; U.cdf[r][e] = acc; }   // np.cumsum
                    for (int e = 0; e < u.n; ++e) U.cdf[r][e] /= acc;                          // cdf /= cdf[-1]
                    for (int e = 0; e < FMC_MAX_USAGE; ++e) {
                        U.slot[r][e] = (int8_t)(e < u.n ? u.slot[e] : -1);
                        U.row[r][e] = c->name_rows[(size_t)i * 2 + off].row[r][e];
                    }
                }
            }
        }
    }
    std::vector<RankSpec> specs((size_t)(ns > 0 ? ns : 1) * kMemoFams * 2);
    std::memset(specs.data(), 0, specs.size() * sizeof(RankSpec));
    c->memo_ok.assign((size_t)ns * kMemoFams * 2, 0);
    c->memo_why.assign((size_t)ns * kMemoFams * 2, "family not in use");
    for (Job &j : jobs) {
        if (!j.err.empty()) return fail(FMC_ERR_CAPACITY, "packing model " + std::to_string(j.fam) + ": " + j.err);
        if (j.fam < kMemoFams) {
            const size_t si = ((size_t)memo_id[j.matchup] * kMemoFams + j.fam) * 2 + j.off;
            specs[si] = j.spec;
            c->memo_ok[si] = j.spec.enabled ? 1 : 0;
            c->memo_why[si] = j.memo_why;
        }
        PackedForest &pf = j.pf;
        const HostForest &f = c->forest[j.fam];
        if (pf.n_outputs > 5) return fail(FMC_ERR_CAPACITY, "more than 5 outputs in a simulation model");
        TableRef &T = md[j.matchup].tbl[j.fam][j.off];
        TablePlacement pl;
        const int table = A.place(pf, pl);
        for (int k = 0; k < pf.n_outputs; ++k) {
            if (pl.n_groups[k] > 0xFFFFu) return fail(FMC_ERR_CAPACITY, "too many tree groups in one output");
            T.stream_off[k] = pl.stream_off[k]; T.consts_off[k] = pl.consts_off[k]; T.n_groups[k] = (uint16_t)pl.n_groups[k];
        }
        T.n_outputs = (uint8_t)pf.n_outputs;
        T.max_depth = (uint8_t)pf.max_depth;
        T.multi_window = pf.table_bytes() > kWindowBytes ? 1 : 0;
        for (int k = 0; k < 5 && k < f.n_outputs; ++k) T.base[k] = (float)f.base[k];
        for (int k = 0; k < 3 && k < f.n_outputs; ++k) T.base64[k] = f.base[k];
        placed.push_back({j.matchup, j.fam, j.off, table});
        c->packed_slots[((size_t)j.matchup * FMC_N_MODELS + j.fam) * 2 + j.off] = (int32_t)pf.slots.size();
        PackedForest().slots.swap(pf.slots);     // release as we go
    }
    CK(cudaSetDevice(c->device));
    CK(A.upload(nullptr, true));
    for (const Pending &q : placed) {
        const uint64_t w = A.window_addr(q.table);
        TableRef &T = md[q.matchup].tbl[q.fam][q.off];
        T.win_lo = (uint32_t)w; T.win_hi = (uint32_t)(w >> 32);
    }
    // entries specialised like an earlier one share its tables
    for (int i = 0; i < n; ++i) {
        if (rep[i] < 0 || rep[i] == i) continue;
        std::memcpy(md[i].tbl, md[rep[i]].tbl, sizeof(md[i].tbl));
        std::memcpy(c->packed_slots.data() + (size_t)i * FMC_N_MODELS * 2, c->packed_slots.data() + (size_t)rep[i] * FMC_N_MODELS * 2,
                    sizeof(int32_t) * FMC_N_MODELS * 2);
    }
    cudaFree(c->d_matchups); cudaFree(c->d_next);
    c->d_matchups = nullptr; c->d_next = nullptr;
    CK(cudaMalloc(&c->d_matchups, md.size() * sizeof(MatchupDev)));
    CK(cudaMalloc(&c->d_next, (size_t)n * 8));
    CK(cudaMemcpy(c->d_matchups, md.data(), md.size() * sizeof(MatchupDev), cudaMemcpyHostToDevice));
    c->h_matchups.swap(md);
    cudaFree(c->d_specs);
    c->d_specs = nullptr;
    CK(cudaMalloc(&c->d_specs, specs.size() * sizeof(RankSpec)));
    CK(cudaMemcpy(c->d_specs, specs.data(), specs.size() * sizeof(RankSpec), cudaMemcpyHostToDevice));
    c->h_next.resize(n);
    c->tables_dirty = false;
    return FMC_OK;
}

// skl leaves are stored pre-multiplied by the learning rate: scale * value is the same IEEE product
// whether it is formed at pack time or per row (sklearn: out += scale * value[leaf]).
static void prescale(HostForest &f) {
    if (f.kind == FMC_KIND_SKL && f.scale != 1.0) {
        for (size_t i = 0; i < f.value.size(); ++i)
            if (f.left[i] < 0) f.value[i] = f.scale * f.value[i];
        f.scale = 1.0;
    }
}

// fmc_set_matchups documents that usage must be set again afterwards: a caller that did not, after the fast path kept
// the old tables, gets what the documented behaviour gives -- no usage.
static void settle_usage(fmc_ctx *c) {
    if (!c->usage_pending) return;
    c->usage.clear(); c->name_rows.clear(); c->n_slots = 0;
    c->usage_pending = false;
    c->tables_dirty = true;
}

extern "C" int fmc_packed_slots(fmc_ctx *c, int32_t m, int32_t *out) {
    if (!c || !out) return fail(FMC_ERR_INVALID, "fmc_packed_slots: bad argument");
    settle_usage(c);
    if (c->tables_dirty) {
        for (int i = 0; i < FMC_N_MODELS; ++i) prescale(c->forest[i]);
        int rc = build_tables(c);
        if (rc) return rc;
    }
    if (m < 0 || m >= (int)c->matchups.size()) return fail(FMC_ERR_INVALID, "fmc_packed_slots: bad matchup");
    std::memcpy(out, c->packed_slots.data() + (size_t)m * FMC_N_MODELS * 2, sizeof(int32_t) * FMC_N_MODELS * 2);
    return FMC_OK;
}

// Sizes the memo regions for a launch of `games` games and (re)allocates them; families that are not in use get
// no region.  Returns the bytes in use (0 = no memo).
static size_t memo_layout(fmc_ctx *c, uint64_t games, MemoRegion (&R)[kMemoFams]) {
    auto pow2_at_least = [](uint64_t v) { uint64_t p = 1; while (p < v) p <<= 1; return p; };
    auto clampu = [](uint64_t v, uint64_t lo, uint64_t hi) { return v < lo ? lo : (v > hi ? hi : v); };
    uint64_t slots[kMemoFams];
    // distinct keys per game measured on configs[1] (scripts/memo_study.py): the boosters see tens of distinct rank
    // vectors per game (their second-resolution clock thresholds), the quantile families a few hundred thousand in all
    // (stage 1: 4.4 M keys after 60 k games, 6.2 M after 100 k, of the order of 1.5e8 after 10 M; quantile families
    // 3e5 after 100 k games).  The table is direct mapped, so it is sized a few times the expected key count.
    slots[0] = clampu(pow2_at_least(games * 96), 1u << 16, 1u << 28);
    slots[1] = clampu(pow2_at_least(games * 48), 1u << 15, 1u << 27);
    slots[2] = slots[3] = clampu(pow2_at_least(games * 4), 1u << 16, 1u << 22);
    slots[4] = clampu(pow2_at_least(games * 2), 1u << 15, 1u << 21);
    slots[5] = clampu(pow2_at_least(games * 64), 1u << 16, 1u << 26);
    bool used[kMemoFams];
    for (int f = 0; f < kMemoFams; ++f) used[f] = family_needed(c, f);
    uint64_t budget = c->memo_max_bytes;
    if (budget == 0) {
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) fr = 0;
        budget = (uint64_t)(fr + c->memo_bytes) / 4;
        if (budget > (16ull << 30)) budget = 16ull << 30;
    }
    auto total = [&]() { uint64_t t = 0; for (int f = 0; f < kMemoFams; ++f) if (used[f]) t += slots[f] << memo_slot_shift(f); return t; };
    while (total() > budget) {      // halve the largest region until the tables fit
        int big = -1;
        for (int f = 0; f < kMemoFams; ++f)
            if (used[f] && slots[f] > 1024 && (big < 0 || (slots[f] << memo_slot_shift(f)) > (slots[big] << memo_slot_shift(big)))) big = f;
        if (big < 0) return 0;
        slots[big] >>= 1;
    }
    const size_t need = (size_t)total();
    if (need == 0) return 0;
    if (need > c->memo_bytes) {
        cudaFree(c->d_memo); c->d_memo = nullptr; c->memo_bytes = 0;
        if (cudaMalloc(&c->d_memo, need) != cudaSuccess) { cudaGetLastError(); return 0; }
        c->memo_bytes = need;
        c->memo_valid = false;
    }
    uint64_t off = 0;
    for (int f = 0; f < kMemoFams; ++f) {
        MemoRegion r;
        r.base = 0; r.slot_mask = 0; r.slot_shift = (uint32_t)memo_slot_shift(f);
        if (used[f]) {
            r.base = (unsigned long long)(uintptr_t)c->d_memo + off;
            r.slot_mask = (uint32_t)(slots[f] - 1);
            off += slots[f] << memo_slot_shift(f);
        }
        if (r.base != R[f].base || r.slot_mask != R[f].slot_mask) c->memo_valid = false;     // the layout changed
        R[f] = r;
    }
    return need;
}

static cudaError_t scratch(fmc_ctx *c, int slot, size_t bytes, void **out);

// The kernel of a launch: player mode, the memo kernel or the plain one; injected draws / traces (TEST); the hooks of
// the optional outputs (HOOKS); overtime (OT).
template <int HOOKS, bool OT = false>
static void launch_sim(const SimKernelArgs &a, const MemoArgs *mm, bool players, bool test, int grid, int mgrid, size_t smem,
                       cudaStream_t st) {
    if (players) {
        if (test) sim_kernel<true, true, HOOKS, OT><<<grid, kSimThreads, smem, st>>>(a);
        else sim_kernel<false, true, HOOKS, OT><<<grid, kSimThreads, smem, st>>>(a);
    } else if (mm) {
        if (test) sim_memo_kernel<true, HOOKS, OT><<<mgrid, kMemoThreads, sim_memo_smem_bytes(), st>>>(a, *mm);
        else sim_memo_kernel<false, HOOKS, OT><<<mgrid, kMemoThreads, sim_memo_smem_bytes(), st>>>(a, *mm);
    } else {
        if (test) sim_kernel<true, false, HOOKS, OT><<<grid, kSimThreads, sim_smem_bytes(false), st>>>(a);
        else sim_kernel<false, false, HOOKS, OT><<<grid, kSimThreads, sim_smem_bytes(false), st>>>(a);
    }
}

// grow-only device scratch for the per-game rows of a hook when the caller did not ask for them
static int hook_rows(fmc_ctx *c, int slot, uint64_t out_games, int words, uint32_t **rows) {
    if (*rows || !out_games) return FMC_OK;
    void *p = nullptr;
    CK(scratch(c, slot, (size_t)out_games * words * sizeof(uint32_t), &p));
    *rows = (uint32_t *)p;
    return FMC_OK;
}

// Every simulation entry point: seg / seq may be NULL or hold only NULL pointers; ot NULL is the reference's end at 0:00.
static int simulate_impl(fmc_ctx *c, const fmc_sim_args *g, const fmc_segment_args *seg, const fmc_sequence_args *seq,
                         const fmc_overtime_args *ot) {
    if (!c || !g) return fail(FMC_ERR_INVALID, "fmc_simulate: bad argument");
    if (ot) {
        if (ot->max_periods < 1 || ot->max_periods > FMC_OT_MAX_PERIODS)
            return fail(FMC_ERR_INVALID, "fmc_simulate_overtime: max_periods must be 1.." + std::to_string(FMC_OT_MAX_PERIODS));
        if (ot->snap_clock < 1 || ot->snap_clock > 900)
            return fail(FMC_ERR_INVALID, "fmc_simulate_overtime: snap_clock must be 1..900");
        if ((seg && (seg->period_scores_dev || seg->segment_hist_dev)) || (seq && (seq->sequence_dev || seq->sequence_hist_dev)))
            return fail(FMC_ERR_INVALID, "fmc_simulate_overtime: overtime has no period or sequence outputs");
    }
    CK(cudaSetDevice(c->device));
    settle_usage(c);
    if (c->tables_dirty) {
        for (int i = 0; i < FMC_N_MODELS; ++i) prescale(c->forest[i]);
        int rc = build_tables(c);
        if (rc) return rc;
    }
    if (g->n_matchups != (int)c->matchups.size()) return fail(FMC_ERR_INVALID, "fmc_simulate: n_matchups mismatch");
    cudaStream_t st = (cudaStream_t)g->stream;
    // one launch in flight per context: the work counters, the running player boxes and the memo are per context
    if (c->launched) CK(cudaStreamWaitEvent(st, c->ev_done, 0));
    uint64_t games = 0, out_games = 0;
    for (size_t i = 0; i < c->matchups.size(); ++i) {
        c->h_next[i] = c->matchups[i].game_begin;
        games += c->matchups[i].game_end - c->matchups[i].game_begin;
        const uint64_t hi = c->matchups[i].out_offset + (c->matchups[i].game_end - c->matchups[i].game_begin);
        if (hi > out_games) out_games = hi;
    }
    // the per-game rows are the state of the hooks: device scratch when the caller only wants the histograms
    const bool segs = seg && (seg->period_scores_dev || seg->segment_hist_dev);
    uint32_t *rows = segs ? seg->period_scores_dev : nullptr;
    if (segs) { int rc = hook_rows(c, 8, out_games, 3, &rows); if (rc) return rc; }
    const bool seqs = seq && (seq->sequence_dev || seq->sequence_hist_dev);
    uint32_t *seq_rows = seqs ? seq->sequence_dev : nullptr;
    if (seqs) { int rc = hook_rows(c, 11, out_games, 2, &seq_rows); if (rc) return rc; }
    CK(cudaMemcpyAsync(c->d_next, c->h_next.data(), c->h_next.size() * 8, cudaMemcpyHostToDevice, st));
    SimKernelArgs a;
    std::memset(&a, 0, sizeof(a));
    a.matchups = c->d_matchups; a.n_matchups = (int)c->matchups.size(); a.next_game = c->d_next;
    a.root_stream = c->sim_tables.d_stream; a.consts = c->sim_tables.d_consts;
    a.seed_lo = (uint32_t)g->seed; a.seed_hi = (uint32_t)(g->seed >> 32);
    a.policy = c->params.policy; a.sampler = c->params.sampler; a.stage2_mode = c->params.stage2_mode;
    a.pass_class = c->params.pass_class;
    if (a.policy == 1 && a.pass_class >= c->forest[FMC_PLAY_MODEL].n_outputs)
        return fail(FMC_ERR_INVALID, "fmc_simulate: pass_class is not a class of the play model");
    a.play_temp = (float)c->params.play_temp; a.qy_noise = c->params.qy_noise;
    for (int k = 0; k < 3; ++k) a.standin[k] = c->params.stage2_standin[k];
    const HostForest &pm = c->forest[FMC_PLAY_MODEL];
    for (int k = 0; k < 6; ++k) { a.pm_scaled[k] = 0; a.pm_mean[k] = 0.0; a.pm_scale[k] = 1.0; }
    for (int j = 0; j < pm.n_scaled; ++j) {
        const int k = pm.scaler_cols[j];
        if (k >= 0 && k < 6) { a.pm_scaled[k] = 1; a.pm_mean[k] = pm.scaler_mean[j]; a.pm_scale[k] = pm.scaler_scale[j]; }
    }
    a.scores = g->scores_dev; a.hist = g->hist_dev; a.counters = (unsigned long long *)g->counters_dev;
    a.stream = g->stream_dev; a.trace = g->trace_dev; a.iters = g->iters_dev;
    a.period_scores = rows; a.segment_hist = segs ? seg->segment_hist_dev : nullptr;
    a.sequence = seq_rows; a.sequence_hist = seqs ? seq->sequence_hist_dev : nullptr;
    if (ot) {
        a.ot_max_periods = ot->max_periods; a.ot_snap_clock = ot->snap_clock;
        a.ot_periods = ot->ot_periods_dev; a.ot_hist = ot->ot_hist_dev;
    }
    const bool players = !c->usage.empty();
    if ((g->players_dev || g->player_hist_dev) && !players)
        return fail(FMC_ERR_INVALID, "fmc_simulate: players_dev / player_hist_dev need fmc_set_usage");
    const int grid = c->prop.multiProcessorCount * kSimCtasPerSm;
    a.n_slots = c->n_slots;
    if (players && c->n_slots > 0) {
        a.players = g->players_dev; a.player_hist = g->player_hist_dev;
        const size_t need = (size_t)grid * kSimThreads * 2 * (size_t)c->n_slots * sizeof(fmc_player_rec);
        if (need > c->box_scratch_bytes) {
            CK(cudaDeviceSynchronize());
            cudaFree(c->d_box_scratch); c->d_box_scratch = nullptr; c->box_scratch_bytes = 0;
            CK(cudaMalloc(&c->d_box_scratch, need));
            c->box_scratch_bytes = need;
        }
        CK(cudaMemsetAsync(c->d_box_scratch, 0, need, st));
        a.box_scratch = c->d_box_scratch;
    }
#ifdef FMC_DEBUG_CHECKS
    debug_set_range(c->sim_tables);
#endif
    const bool test = a.stream || a.trace;      // parity-test instantiation
    size_t smem = 0;
    MemoArgs mm;
    bool memo = false;
    if (players) {
        a.n_prow = c->n_prow; a.n_trow = c->n_trow; a.n_rrow = c->n_rrow;
        a.name_rows = c->n_prow + c->n_trow > c->n_rrow ? c->n_prow + c->n_trow : c->n_rrow;
        smem = sim_smem_bytes_players(a.name_rows);
    } else if (c->memo_mode != 0 && c->n_specs <= 1024) {     // the memo key has 10 bits for the specialisation
        // exact memo in front of the walk (fmc_sim_memo.cuh)
        memo = true;
        std::memset(&mm, 0, sizeof(mm));
        const bool was_valid = c->memo_valid;
        size_t bytes = memo_layout(c, games, c->memo_region);
        if (bytes && !(c->memo_mode == 2 && was_valid && c->memo_valid)) CK(cudaMemsetAsync(c->d_memo, 0, bytes, st));
        for (int f = 0; f < kMemoFams; ++f) mm.region[f] = c->memo_region[f];
        mm.specs = c->d_specs;
        mm.enabled = bytes ? 1 : 0;
        mm.max_trips = c->memo_max_trips;
        mm.break_parked = c->memo_break_parked;
        mm.break_waiting = c->memo_break_waiting;
        c->memo_valid = bytes != 0;
    }
    const int mgrid = c->prop.multiProcessorCount * kMemoCtasPerSm;
    const MemoArgs *mp = memo ? &mm : nullptr;
    if (ot) launch_sim<0, true>(a, mp, players, test, grid, mgrid, smem, st);
    else switch ((segs ? kHookPeriods : 0) | (seqs ? kHookSequence : 0)) {
    case 0: launch_sim<0>(a, mp, players, test, grid, mgrid, smem, st); break;
    case kHookPeriods: launch_sim<kHookPeriods>(a, mp, players, test, grid, mgrid, smem, st); break;
    case kHookSequence: launch_sim<kHookSequence>(a, mp, players, test, grid, mgrid, smem, st); break;
    default: launch_sim<kHookPeriods | kHookSequence>(a, mp, players, test, grid, mgrid, smem, st); break;
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev_done, st));
    c->launched = true;
    return FMC_OK;
}

extern "C" int fmc_simulate(fmc_ctx *c, const fmc_sim_args *g) { return simulate_impl(c, g, nullptr, nullptr, nullptr); }

extern "C" int fmc_simulate_segments(fmc_ctx *c, const fmc_sim_args *g, const fmc_segment_args *seg) {
    return simulate_impl(c, g, seg, nullptr, nullptr);
}

extern "C" int fmc_simulate_markets(fmc_ctx *c, const fmc_sim_args *g, const fmc_segment_args *seg, const fmc_sequence_args *seq) {
    return simulate_impl(c, g, seg, seq, nullptr);
}

extern "C" int fmc_simulate_overtime(fmc_ctx *c, const fmc_sim_args *g, const fmc_overtime_args *ot) {
    return simulate_impl(c, g, nullptr, nullptr, ot);
}

// Device scratch of fmc_simulate_host, kept in the context between calls (grow-only): no cudaMalloc / cudaFree per call.
static cudaError_t scratch(fmc_ctx *c, int slot, size_t bytes, void **out) {
    fmc_ctx::Scratch &q = c->scr[slot];
    if (bytes > q.dev_bytes) {
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return e;
        cudaFree(q.dev); q.dev = nullptr; q.dev_bytes = 0;
        if ((e = cudaMalloc(&q.dev, bytes)) != cudaSuccess) return e;
        q.dev_bytes = bytes;
    }
    *out = q.dev;
    return cudaSuccess;
}

// Device -> pageable host copy through the context's pinned staging buffers (large results only: the per-game score words,
// the per-game player box); the device is idle when this runs (fmc_simulate_host synchronises first).
static cudaError_t d2h_staged(fmc_ctx *c, void *dst, const void *src, size_t bytes) {
    constexpr size_t kChunk = 8u << 20;
    if (bytes <= kChunk) return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
    cudaError_t e;
    for (int b = 0; b < 2; ++b) {
        if (!c->pin[b] && (e = cudaHostAlloc(&c->pin[b], kChunk, cudaHostAllocDefault)) != cudaSuccess) { c->pin[b] = nullptr; cudaGetLastError(); return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost); }
        if (!c->copy_ev[b] && (e = cudaEventCreateWithFlags(&c->copy_ev[b], cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    if (!c->copy_stream && (e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
    const size_t n = (bytes + kChunk - 1) / kChunk;
    auto len = [&](size_t i) { return i + 1 < n ? kChunk : bytes - i * kChunk; };
    auto issue = [&](size_t i) -> cudaError_t {
        cudaError_t r = cudaMemcpyAsync(c->pin[i & 1], (const char *)src + i * kChunk, len(i), cudaMemcpyDeviceToHost, c->copy_stream);
        return r != cudaSuccess ? r : cudaEventRecord(c->copy_ev[i & 1], c->copy_stream);
    };
    auto drain = [&](size_t i) -> cudaError_t {
        cudaError_t r = cudaEventSynchronize(c->copy_ev[i & 1]);
        if (r == cudaSuccess) std::memcpy((char *)dst + i * kChunk, c->pin[i & 1], len(i));
        return r;
    };
    if ((e = issue(0)) != cudaSuccess) return e;
    for (size_t i = 1; i < n; ++i) {
        if ((e = issue(i)) != cudaSuccess) return e;          // buffer i & 1 was drained as chunk i - 2 in the previous turn
        if ((e = drain(i - 1)) != cudaSuccess) return e;
    }
    return drain(n - 1);
}

static int simulate_host_impl(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                              uint64_t *counters_host, const double *stream_host, double *trace_host,
                              uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                              uint32_t *period_host, uint32_t *seg_hist_host, uint32_t *seq_host, uint32_t *seq_hist_host,
                              const fmc_overtime_args *ot_host = nullptr) {
    if (!c) return fail(FMC_ERR_INVALID, "ctx is NULL");
    if (c->matchups.empty()) return fail(FMC_ERR_INVALID, "fmc_set_matchups has not been called");
    CK(cudaSetDevice(c->device));
    settle_usage(c);
    size_t games = 0;
    for (auto &m : c->matchups) {
        const size_t hi = (size_t)(m.out_offset + (m.game_end - m.game_begin));
        if (hi > games) games = hi;
    }
    const size_t nm = c->matchups.size();
    const size_t hist_n = nm * 2 * FMC_HIST_BINS * FMC_HIST_BINS;
    uint32_t *d_scores = nullptr, *d_hist = nullptr;
    uint64_t *d_cnt = nullptr;
    double *d_stream = nullptr, *d_trace = nullptr;
    uint16_t *d_iters = nullptr;
    fmc_player_rec *d_players = nullptr;
    const size_t players_n = games * 2 * (size_t)c->n_slots;
    if ((players_host || player_hist_host) && c->usage.empty()) return fail(FMC_ERR_INVALID, "players output needs fmc_set_usage");
    uint32_t *d_phist = nullptr, *d_period = nullptr, *d_seg = nullptr, *d_seq = nullptr, *d_seqh = nullptr;
    const size_t seg_n = nm * 2 * FMC_N_SEGMENTS * FMC_HIST_BINS * FMC_HIST_BINS;
    const size_t seqh_n = nm * 2 * FMC_SEQ_BINS;
    const size_t oth_n = nm * 2 * (FMC_OT_MAX_PERIODS + 1) * 3;
    uint8_t *d_otp = nullptr;
    uint32_t *d_oth = nullptr;
    const size_t phist_n = c->matchups.size() * 2 * (size_t)c->n_slots * FMC_PH_BINS;
    int rc = FMC_OK;
    cudaError_t e = cudaSuccess;
    auto bail = [&](cudaError_t err, const char *what) { rc = fail(FMC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(err)); };
    // the copies below run on the legacy default stream: order them after a launch the caller left in flight
    if (c->launched && (e = cudaEventSynchronize(c->ev_done)) != cudaSuccess) return fail(FMC_ERR_CUDA, std::string("previous launch: ") + cudaGetErrorString(e));
    do {
        if (scores_host && games) { if ((e = scratch(c, 0, games * 4, (void **)&d_scores)) != cudaSuccess) { bail(e, "cudaMalloc scores"); break; } }
        if (hist_host) {
            if ((e = scratch(c, 1, hist_n * 4, (void **)&d_hist)) != cudaSuccess) { bail(e, "cudaMalloc hist"); break; }
            if ((e = cudaMemsetAsync(d_hist, 0, hist_n * 4)) != cudaSuccess) { bail(e, "memset hist"); break; }
        }
        if ((e = scratch(c, 2, FMC_N_COUNTERS * 8, (void **)&d_cnt)) != cudaSuccess) { bail(e, "cudaMalloc counters"); break; }
        if ((e = cudaMemsetAsync(d_cnt, 0, FMC_N_COUNTERS * 8)) != cudaSuccess) { bail(e, "memset counters"); break; }
        if (stream_host && games) {
            const size_t b = games * FMC_MAX_ITERS * FMC_N_SLOTS * 8;
            if ((e = scratch(c, 3, b, (void **)&d_stream)) != cudaSuccess) { bail(e, "cudaMalloc stream"); break; }
            if ((e = cudaMemcpy(d_stream, stream_host, b, cudaMemcpyHostToDevice)) != cudaSuccess) { bail(e, "H2D stream"); break; }
        }
        if (trace_host && games) {
            const size_t b = games * FMC_MAX_ITERS * FMC_TRACE_COLS * 8;
            if ((e = scratch(c, 4, b, (void **)&d_trace)) != cudaSuccess) { bail(e, "cudaMalloc trace"); break; }
            if ((e = cudaMemsetAsync(d_trace, 0xFF, b)) != cudaSuccess) { bail(e, "memset trace"); break; }   // NaN fill
        }
        if (iters_host && games) { if ((e = scratch(c, 5, games * 2, (void **)&d_iters)) != cudaSuccess) { bail(e, "cudaMalloc iters"); break; } }
        if (players_host && players_n) {
            if ((e = scratch(c, 6, players_n * sizeof(fmc_player_rec), (void **)&d_players)) != cudaSuccess) { bail(e, "cudaMalloc players"); break; }
        }
        if (player_hist_host && phist_n) {
            if ((e = scratch(c, 7, phist_n * 4, (void **)&d_phist)) != cudaSuccess) { bail(e, "cudaMalloc player hist"); break; }
            if ((e = cudaMemsetAsync(d_phist, 0, phist_n * 4)) != cudaSuccess) { bail(e, "memset player hist"); break; }
        }
        if (period_host && games) {
            if ((e = scratch(c, 9, games * 3 * 4, (void **)&d_period)) != cudaSuccess) { bail(e, "cudaMalloc period scores"); break; }
        }
        if (seg_hist_host) {
            if ((e = scratch(c, 10, seg_n * 4, (void **)&d_seg)) != cudaSuccess) { bail(e, "cudaMalloc segment hist"); break; }
            if ((e = cudaMemsetAsync(d_seg, 0, seg_n * 4)) != cudaSuccess) { bail(e, "memset segment hist"); break; }
        }
        if (seq_host && games) {
            if ((e = scratch(c, 12, games * 2 * 4, (void **)&d_seq)) != cudaSuccess) { bail(e, "cudaMalloc sequence"); break; }
        }
        if (seq_hist_host) {
            if ((e = scratch(c, 13, seqh_n * 4, (void **)&d_seqh)) != cudaSuccess) { bail(e, "cudaMalloc sequence hist"); break; }
            if ((e = cudaMemsetAsync(d_seqh, 0, seqh_n * 4)) != cudaSuccess) { bail(e, "memset sequence hist"); break; }
        }
        if (ot_host && ot_host->ot_periods_dev && games) {
            if ((e = scratch(c, 14, games, (void **)&d_otp)) != cudaSuccess) { bail(e, "cudaMalloc overtime periods"); break; }
        }
        if (ot_host && ot_host->ot_hist_dev) {
            if ((e = scratch(c, 15, oth_n * 4, (void **)&d_oth)) != cudaSuccess) { bail(e, "cudaMalloc overtime hist"); break; }
            if ((e = cudaMemsetAsync(d_oth, 0, oth_n * 4)) != cudaSuccess) { bail(e, "memset overtime hist"); break; }
        }
        fmc_sim_args g;
        std::memset(&g, 0, sizeof(g));
        g.player_hist_dev = d_phist;
        g.seed = seed; g.n_matchups = (int)nm; g.scores_dev = d_scores; g.hist_dev = d_hist; g.counters_dev = d_cnt;
        g.stream_dev = d_stream; g.trace_dev = d_trace; g.iters_dev = d_iters; g.stream = nullptr;
        g.players_dev = d_players;
        fmc_segment_args sg;
        sg.period_scores_dev = d_period; sg.segment_hist_dev = d_seg;
        fmc_sequence_args sq;
        sq.sequence_dev = d_seq; sq.sequence_hist_dev = d_seqh;
        fmc_overtime_args ov;
        if (ot_host) { ov = *ot_host; ov.ot_periods_dev = d_otp; ov.ot_hist_dev = d_oth; }
        rc = simulate_impl(c, &g, &sg, &sq, ot_host ? &ov : nullptr);
        if (rc) break;
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) { bail(e, "sim_kernel"); break; }
        if (scores_host && games && (e = d2h_staged(c, scores_host, d_scores, games * 4)) != cudaSuccess) { bail(e, "D2H scores"); break; }
        if (hist_host && (e = cudaMemcpy(hist_host, d_hist, hist_n * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H hist"); break; }
        if (counters_host && (e = cudaMemcpy(counters_host, d_cnt, FMC_N_COUNTERS * 8, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H counters"); break; }
        if (trace_host && games && (e = cudaMemcpy(trace_host, d_trace, games * FMC_MAX_ITERS * FMC_TRACE_COLS * 8, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H trace"); break; }
        if (iters_host && games && (e = cudaMemcpy(iters_host, d_iters, games * 2, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H iters"); break; }
        if (d_players && (e = d2h_staged(c, players_host, d_players, players_n * sizeof(fmc_player_rec))) != cudaSuccess) { bail(e, "D2H players"); break; }
        if (d_phist && (e = cudaMemcpy(player_hist_host, d_phist, phist_n * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H player hist"); break; }
        if (d_period && (e = d2h_staged(c, period_host, d_period, games * 3 * 4)) != cudaSuccess) { bail(e, "D2H period scores"); break; }
        if (d_seg && (e = cudaMemcpy(seg_hist_host, d_seg, seg_n * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H segment hist"); break; }
        if (d_seq && (e = d2h_staged(c, seq_host, d_seq, games * 2 * 4)) != cudaSuccess) { bail(e, "D2H sequence"); break; }
        if (d_seqh && (e = cudaMemcpy(seq_hist_host, d_seqh, seqh_n * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H sequence hist"); break; }
        if (d_otp && (e = cudaMemcpy(ot_host->ot_periods_dev, d_otp, games, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H overtime periods"); break; }
        if (d_oth && (e = cudaMemcpy(ot_host->ot_hist_dev, d_oth, oth_n * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) { bail(e, "D2H overtime hist"); break; }
    } while (0);
    // big test-mode buffers (injected draws, traces: 46 KB per game) are not worth keeping
    for (int slot : {3, 4})
        if (c->scr[slot].dev_bytes > (256u << 20)) { cudaFree(c->scr[slot].dev); c->scr[slot].dev = nullptr; c->scr[slot].dev_bytes = 0; }
    return rc;
}

extern "C" int fmc_simulate_host(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                                 uint64_t *counters_host, const double *stream_host, double *trace_host,
                                 uint16_t *iters_host) {
    return simulate_host_impl(c, seed, scores_host, hist_host, counters_host, stream_host, trace_host, iters_host, nullptr, nullptr,
                              nullptr, nullptr, nullptr, nullptr);
}

extern "C" int fmc_simulate_players_host(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                                         uint64_t *counters_host, const double *stream_host, double *trace_host,
                                         uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host) {
    return simulate_host_impl(c, seed, scores_host, hist_host, counters_host, stream_host, trace_host, iters_host, players_host,
                              player_hist_host, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int fmc_simulate_segments_host(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                                          uint64_t *counters_host, const double *stream_host, double *trace_host,
                                          uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                                          uint32_t *period_scores_host, uint32_t *segment_hist_host) {
    return simulate_host_impl(c, seed, scores_host, hist_host, counters_host, stream_host, trace_host, iters_host, players_host,
                              player_hist_host, period_scores_host, segment_hist_host, nullptr, nullptr);
}

extern "C" int fmc_simulate_markets_host(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                                         uint64_t *counters_host, const double *stream_host, double *trace_host,
                                         uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                                         uint32_t *period_scores_host, uint32_t *segment_hist_host, uint32_t *sequence_host,
                                         uint32_t *sequence_hist_host) {
    return simulate_host_impl(c, seed, scores_host, hist_host, counters_host, stream_host, trace_host, iters_host, players_host,
                              player_hist_host, period_scores_host, segment_hist_host, sequence_host, sequence_hist_host);
}

extern "C" int fmc_simulate_overtime_host(fmc_ctx *c, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                                          uint64_t *counters_host, const double *stream_host, double *trace_host,
                                          uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                                          int32_t max_periods, int32_t snap_clock, uint8_t *ot_periods_host, uint32_t *ot_hist_host) {
    // host pointers in the device fields: simulate_host_impl stages them through device scratch
    const fmc_overtime_args ot{max_periods, snap_clock, ot_periods_host, ot_hist_host};
    return simulate_host_impl(c, seed, scores_host, hist_host, counters_host, stream_host, trace_host, iters_host, players_host,
                              player_hist_host, nullptr, nullptr, nullptr, nullptr, &ot);
}

extern "C" int fmc_tree_predict(fmc_ctx *c, int32_t id, const double *rows_dev, int64_t n, double *out_dev,
                                int32_t tree_begin, int32_t tree_end, int32_t coach_col, void *stream) {
    if (!c || id < 0 || id >= FMC_N_MODELS || !c->forest[id].loaded) return fail(FMC_ERR_INVALID, "fmc_tree_predict: model not loaded");
    if (n < 0 || (n > 0 && (!rows_dev || !out_dev))) return fail(FMC_ERR_INVALID, "fmc_tree_predict: bad buffers");
    if (n == 0) return FMC_OK;
    CK(cudaSetDevice(c->device));
    HostForest &f = c->forest[id];
    prescale(f);
    cudaStream_t st = (cudaStream_t)stream;
    const int c0 = id == FMC_PLAY_MODEL ? coach_col : f.active[0], c1 = id == FMC_PLAY_MODEL ? -1 : f.active[1];
    fmc_ctx::PredEntry *E = nullptr, *lru = &c->pred[0];
    for (auto &e : c->pred) {
        if (e.id == id && e.tb == tree_begin && e.te == tree_end && e.c0 == c0 && e.c1 == c1 && e.version == c->forest_version[id]) { E = &e; break; }
        if (e.last_use < lru->last_use) lru = &e;
    }
    if (!E) {
        PackSpec s;
        preset_predict(s);
        s.active[0] = c0; s.active[1] = c1;
        s.tree_begin = tree_begin; s.tree_end = tree_end;
        PackedForest pf;
        const std::string err = pack_forest(f, s, pf);
        if (!err.empty()) return fail(FMC_ERR_CAPACITY, "packing model " + std::to_string(id) + ": " + err);
        CK(cudaDeviceSynchronize());     // a launch in flight may still read the entry that is being replaced
        E = lru;
        E->id = -1;
        E->arena.clear();
        E->table = E->arena.place(pf, E->pl);
        CK(E->arena.upload(st, true));
        E->multi_window = pf.table_bytes() > kWindowBytes;
        E->id = id; E->tb = tree_begin; E->te = tree_end; E->c0 = c0; E->c1 = c1; E->version = c->forest_version[id];
    }
    E->last_use = ++c->pred_clock;
    TableArena &A = E->arena;
    const TablePlacement &pl = E->pl;
    const int table = E->table;
    PredictArgs a;
    std::memset(&a, 0, sizeof(a));
    a.rows = rows_dev; a.out = out_dev; a.n = n;
    const uint64_t w = A.window_addr(table);
    a.win_lo = (uint32_t)w; a.win_hi = (uint32_t)(w >> 32);
    a.stream = A.d_stream; a.consts = A.d_consts;
    for (int k = 0; k < 8; ++k) { a.stream_off[k] = pl.stream_off[k]; a.consts_off[k] = pl.consts_off[k]; a.n_groups[k] = pl.n_groups[k]; }
    a.n_outputs = f.n_outputs; a.n_num = f.n_num;
    a.multi_window = E->multi_window ? 1 : 0;
    a.zero_is_missing = (f.kind == FMC_KIND_XGB && f.zero_is_missing) ? 1 : 0;
    for (int k = 0; k < 8; ++k) a.base[k] = f.base[k];
    a.n_scaled = f.n_scaled;
    for (int j = 0; j < f.n_scaled; ++j) { a.scaler_cols[j] = f.scaler_cols[j]; a.scaler_mean[j] = f.scaler_mean[j]; a.scaler_scale[j] = f.scaler_scale[j]; }
    a.stats = c->d_pred_stats;
#ifdef FMC_DEBUG_CHECKS
    debug_set_range(A);
#endif
    long long blocks = (n + kPredThreads - 1) / kPredThreads;
    const long long cap = (long long)c->prop.multiProcessorCount * 8;
    if (blocks > cap) blocks = cap;
    if (f.kind == FMC_KIND_SKL) predict_kernel<true><<<(int)blocks, kPredThreads, 0, st>>>(a);
    else predict_kernel<false><<<(int)blocks, kPredThreads, 0, st>>>(a);
    CK(cudaGetLastError());
    return FMC_OK;
}

// NaN inputs: xgboost treats them as missing (the node's default branch), which the predict kernel honours for every
// numeric that has a B view; scikit-learn's Pipeline.predict raises on them.
static int check_nan_rows(const HostForest &f, const double *rows, int64_t n, const char *who) {
    const bool skl = f.kind == FMC_KIND_SKL, dense_xgb = !skl && !f.zero_is_missing;
    if (!skl && !dense_xgb) return FMC_OK;
    for (int64_t i = 0; i < n; ++i)
        for (int k = 0; k < f.n_num && k < kNumMax; ++k) {
            const double x = rows[i * kNumMax + k];
            if (x == x) continue;
            if (skl) return fail(FMC_ERR_INVALID, std::string(who) + ": Input X contains NaN (scikit-learn model)");
            if (k == 3 || k == 12 || k == 13 || k == 14 || k == 16)
                return fail(FMC_ERR_INVALID, std::string(who) + ": NaN in a 0/1 flag column of a dense-fed booster is not supported");
        }
    return FMC_OK;
}

extern "C" int fmc_tree_predict_host(fmc_ctx *c, int32_t id, const double *rows_host, int64_t n, double *out_host,
                                     int32_t tree_begin, int32_t tree_end, int32_t coach_col) {
    if (!c || id < 0 || id >= FMC_N_MODELS || !c->forest[id].loaded) return fail(FMC_ERR_INVALID, "fmc_tree_predict_host: model not loaded");
    if (n <= 0) return FMC_OK;
    if (int rc_nan = check_nan_rows(c->forest[id], rows_host, n, "fmc_tree_predict_host")) return rc_nan;
    CK(cudaSetDevice(c->device));
    const int no = c->forest[id].n_outputs;
    double *d_rows = nullptr, *d_out = nullptr;
    CK(cudaMalloc(&d_rows, (size_t)n * kNumMax * 8));
    cudaError_t e = cudaMalloc(&d_out, (size_t)n * no * 8);
    if (e != cudaSuccess) { cudaFree(d_rows); return fail(FMC_ERR_CUDA, std::string("cudaMalloc out: ") + cudaGetErrorString(e)); }
    int rc = FMC_OK;
    e = cudaMemcpy(d_rows, rows_host, (size_t)n * kNumMax * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = fmc_tree_predict(c, id, d_rows, n, d_out, tree_begin, tree_end, coach_col, nullptr);
        if (rc == FMC_OK) e = cudaDeviceSynchronize();
        if (rc == FMC_OK && e == cudaSuccess) e = cudaMemcpy(out_host, d_out, (size_t)n * no * 8, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_rows); cudaFree(d_out);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(FMC_ERR_CUDA, std::string("fmc_tree_predict_host: ") + cudaGetErrorString(e));
    return FMC_OK;
}

// Per-row names (FMC:744, 756, 784-809: every row of a DataFrame carries its own passer / target / rusher): rows are
// grouped by their pair of hot one-hot columns, every distinct pair gets its own specialised table (packed by all host
// threads, uploaded once), and one predict launch per group walks its rows.  Outputs come back in row order.
extern "C" int fmc_tree_predict_cols_host(fmc_ctx *c, int32_t id, const double *rows_host, int64_t n, const int32_t *hot_cols_host,
                                          double *out_host, int32_t tree_begin, int32_t tree_end) {
    if (!c || id < 0 || id >= FMC_N_MODELS || !c->forest[id].loaded) return fail(FMC_ERR_INVALID, "fmc_tree_predict_cols_host: model not loaded");
    if (n < 0 || (n > 0 && (!rows_host || !out_host || !hot_cols_host))) return fail(FMC_ERR_INVALID, "fmc_tree_predict_cols_host: bad buffers");
    if (n == 0) return FMC_OK;
    CK(cudaSetDevice(c->device));
    HostForest &f = c->forest[id];
    prescale(f);
    if (int rc_nan = check_nan_rows(f, rows_host, n, "fmc_tree_predict_cols_host")) return rc_nan;
    for (int64_t i = 0; i < 2 * n; ++i)
        if (hot_cols_host[i] < -1 || hot_cols_host[i] >= f.n_features || (hot_cols_host[i] >= f.num_base && hot_cols_host[i] < f.num_base + f.n_num))
            return fail(FMC_ERR_INVALID, "fmc_tree_predict_cols_host: a hot column must be -1 or a one-hot column of the model");
    // ---- group the rows by their column pair (first-appearance order)
    struct Group { int32_t c0, c1; std::vector<int64_t> rows; PackedForest pf; std::string err; TablePlacement pl; int table = 0; bool multi = false; };
    std::vector<Group> groups;
    {
        std::vector<std::pair<uint64_t, int>> index;     // sorted (pair -> group)
        for (int64_t i = 0; i < n; ++i) {
            const uint64_t k = ((uint64_t)(uint32_t)hot_cols_host[2 * i] << 32) | (uint32_t)hot_cols_host[2 * i + 1];
            auto it = std::lower_bound(index.begin(), index.end(), std::make_pair(k, -1));
            int g;
            if (it != index.end() && it->first == k) g = it->second;
            else {
                g = (int)groups.size();
                groups.emplace_back();
                groups.back().c0 = hot_cols_host[2 * i]; groups.back().c1 = hot_cols_host[2 * i + 1];
                index.insert(it, std::make_pair(k, g));
            }
            groups[(size_t)g].rows.push_back(i);
        }
    }
    // ---- specialise + pack every pair on all host threads
    auto run = [&](Group &g) {
        PackSpec s;
        preset_predict(s);
        s.active[0] = g.c0; s.active[1] = g.c1;
        s.tree_begin = tree_begin; s.tree_end = tree_end;
        g.err = pack_forest(f, s, g.pf);
    };
    {
        unsigned nt = std::thread::hardware_concurrency();
        if (nt == 0) nt = 1;
        if (nt > 32) nt = 32;
        if (groups.size() < 4) nt = 1;
        if (nt <= 1) for (Group &g : groups) run(g);
        else {
            std::atomic<size_t> next{0};
            std::vector<std::thread> pool;
            for (unsigned t = 0; t < nt; ++t)
                pool.emplace_back([&]() { for (size_t k; (k = next.fetch_add(1)) < groups.size();) run(groups[k]); });
            for (auto &th : pool) th.join();
        }
    }
    TableArena A;
    for (Group &g : groups) {
        if (!g.err.empty()) return fail(FMC_ERR_CAPACITY, "packing model " + std::to_string(id) + ": " + g.err);
        g.multi = g.pf.table_bytes() > kWindowBytes;
        g.table = A.place(g.pf, g.pl);
        std::vector<uint64_t>().swap(g.pf.slots);
    }
    const int no = f.n_outputs;
    double *d_rows = nullptr, *d_out = nullptr;
    std::vector<double> staged((size_t)n * kNumMax), outs((size_t)n * no);
    {
        size_t at = 0;
        for (const Group &g : groups)
            for (int64_t r : g.rows) { std::memcpy(&staged[at * kNumMax], rows_host + r * kNumMax, sizeof(double) * kNumMax); ++at; }
    }
    int rc = FMC_OK;
    cudaError_t e = cudaSuccess;
    do {
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) break;
        if ((e = A.upload(nullptr, true)) != cudaSuccess) break;
        if ((e = cudaMalloc(&d_rows, staged.size() * 8)) != cudaSuccess) break;
        if ((e = cudaMalloc(&d_out, outs.size() * 8)) != cudaSuccess) break;
        if ((e = cudaMemcpy(d_rows, staged.data(), staged.size() * 8, cudaMemcpyHostToDevice)) != cudaSuccess) break;
        size_t at = 0;
        for (const Group &g : groups) {
            const long long m = (long long)g.rows.size();
            PredictArgs a;
            std::memset(&a, 0, sizeof(a));
            a.rows = d_rows + at * kNumMax; a.out = d_out + at * no; a.n = m;
            const uint64_t w = A.window_addr(g.table);
            a.win_lo = (uint32_t)w; a.win_hi = (uint32_t)(w >> 32);
            a.stream = A.d_stream; a.consts = A.d_consts;
            for (int k = 0; k < 8; ++k) { a.stream_off[k] = g.pl.stream_off[k]; a.consts_off[k] = g.pl.consts_off[k]; a.n_groups[k] = g.pl.n_groups[k]; }
            a.n_outputs = no; a.n_num = f.n_num;
            a.multi_window = g.multi ? 1 : 0;
            a.zero_is_missing = (f.kind == FMC_KIND_XGB && f.zero_is_missing) ? 1 : 0;
            for (int k = 0; k < 8; ++k) a.base[k] = f.base[k];
            a.n_scaled = f.n_scaled;
            for (int j = 0; j < f.n_scaled; ++j) { a.scaler_cols[j] = f.scaler_cols[j]; a.scaler_mean[j] = f.scaler_mean[j]; a.scaler_scale[j] = f.scaler_scale[j]; }
            a.stats = c->d_pred_stats;
            long long blocks = (m + kPredThreads - 1) / kPredThreads;
            const long long cap = (long long)c->prop.multiProcessorCount * 8;
            if (blocks > cap) blocks = cap;
            if (f.kind == FMC_KIND_SKL) predict_kernel<true><<<(int)blocks, kPredThreads>>>(a);
            else predict_kernel<false><<<(int)blocks, kPredThreads>>>(a);
            at += (size_t)m;
        }
        if ((e = cudaGetLastError()) != cudaSuccess) break;
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) break;
        if ((e = cudaMemcpy(outs.data(), d_out, outs.size() * 8, cudaMemcpyDeviceToHost)) != cudaSuccess) break;
        at = 0;
        for (const Group &g : groups)
            for (int64_t r : g.rows) { std::memcpy(out_host + r * no, &outs[at * no], sizeof(double) * no); ++at; }
    } while (0);
    cudaFree(d_rows); cudaFree(d_out);
    A.release();
    if (e != cudaSuccess) rc = fail(FMC_ERR_CUDA, std::string("fmc_tree_predict_cols_host: ") + cudaGetErrorString(e));
    return rc;
}

// Diagnostics: number of out-of-range gathers / feature offsets seen by a library built with
// -DFMC_DEBUG_CHECKS (always 0 for the production build), counted since the last call.
extern "C" int64_t fmc_debug_errors(void) {
#ifdef FMC_DEBUG_CHECKS
    unsigned long long v = 0, z = 0;
    if (cudaMemcpyFromSymbol(&v, g_dbg_errors, 8) != cudaSuccess) return -1;
    cudaMemcpyToSymbol(g_dbg_errors, &z, 8);
    return (int64_t)v;
#else
    return 0;
#endif
}
// Node gathers of the fmc_tree_predict launches since the last reset: out[0] warp-level (one per warp and tree level,
// what the L1 data pipe sees), out[1] lane-level of live rows.  Synchronises the device.
extern "C" int fmc_predict_stats(fmc_ctx *c, uint64_t *out2, int32_t reset) {
    if (!c || !out2) return fail(FMC_ERR_INVALID, "fmc_predict_stats: bad argument");
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out2, c->d_pred_stats, 16, cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(c->d_pred_stats, 0, 16));
    return FMC_OK;
}

// Measurement helper: forget the specialised tables, so that the next fmc_simulate specialises, packs and uploads again.
extern "C" int fmc_invalidate_tables(fmc_ctx *c) {
    if (!c) return fail(FMC_ERR_INVALID, "ctx is NULL");
    c->tables_dirty = true;
    return FMC_OK;
}

extern "C" int fmc_sync(fmc_ctx *c) {
    if (!c) return fail(FMC_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    return FMC_OK;
}

// ---------------------------------------------------------------------------------------------
// Achievable gather bandwidth (the roofline denominator SURVEY 8(d) asks for): every lane runs
// kProbeChains dependent chains of 8-byte read-only gathers through a table of `table_bytes`
// (each slot holds the index of the next one: a random cyclic permutation), the access pattern of a
// tree walk with no arithmetic around it.  table_bytes well below the L1 size measures the L1 gather
// rate, a few MiB the L2 gather rate.
// ---------------------------------------------------------------------------------------------
constexpr int kProbeChains = 8;
__global__ void __launch_bounds__(1024, 1) gather_probe_kernel(const uint2 *__restrict__ tbl, uint32_t n_slots, int iters,
                                                              unsigned int *sink) {
    uint32_t idx[kProbeChains];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int c = 0; c < kProbeChains; ++c) idx[c] = (t * 2654435761u + (uint32_t)c * 40503u) % n_slots;
    uint32_t acc = 0;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int c = 0; c < kProbeChains; ++c) {
            const uint2 v = __ldg(tbl + idx[c]);
            idx[c] = v.x;
            acc ^= v.y;
        }
    }
    if (acc == 0x12345678u) atomicAdd(sink, 1u);
}

extern "C" int fmc_gather_probe(fmc_ctx *c, int64_t table_bytes, int32_t iters, double *gbytes_per_s) {
    if (!c || !gbytes_per_s || table_bytes < 1024 || iters <= 0) return fail(FMC_ERR_INVALID, "fmc_gather_probe: bad argument");
    CK(cudaSetDevice(c->device));
    const uint32_t n = (uint32_t)(table_bytes / 8);
    std::vector<uint2> h(n);
    // random cyclic permutation (Sattolo) so that every chain visits the whole table
    std::vector<uint32_t> perm(n);
    for (uint32_t i = 0; i < n; ++i) perm[i] = i;
    uint64_t s = 0x9E3779B97F4A7C15ull;
    for (uint32_t i = n - 1; i > 0; --i) {
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        const uint32_t j = (uint32_t)((s >> 33) % i);
        std::swap(perm[i], perm[j]);
    }
    for (uint32_t i = 0; i < n; ++i) h[i] = make_uint2(perm[i], i);
    uint2 *d = nullptr;
    unsigned int *sink = nullptr;
    CK(cudaMalloc(&d, (size_t)n * 8));
    cudaError_t e = cudaMalloc(&sink, 4);
    if (e != cudaSuccess) { cudaFree(d); return fail(FMC_ERR_CUDA, cudaGetErrorString(e)); }
    cudaMemcpy(d, h.data(), (size_t)n * 8, cudaMemcpyHostToDevice);
    cudaMemset(sink, 0, 4);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int grid = c->prop.multiProcessorCount;
    gather_probe_kernel<<<grid, 1024>>>(d, n, iters / 4 + 1, sink);      // warm-up
    float best = 1e30f;
    for (int r = 0; r < 3; ++r) {
        cudaEventRecord(e0);
        gather_probe_kernel<<<grid, 1024>>>(d, n, iters, sink);
        cudaEventRecord(e1);
        e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d); cudaFree(sink);
    if (e != cudaSuccess) return fail(FMC_ERR_CUDA, std::string("gather_probe_kernel: ") + cudaGetErrorString(e));
    const double loads = (double)grid * 1024.0 * kProbeChains * (double)iters;
    *gbytes_per_s = loads * 8.0 / ((double)best * 1e-3) / 1e9;
    return FMC_OK;
}

// Warp-coherent variant: the production walk is not a random gather -- at every level the 32 lanes of a warp sit inside
// ONE tree, i.e. inside a window of a few hundred bytes.  Here every warp follows kProbeChains chains of WINDOWS of
// `window_bytes` (a random cyclic permutation over the windows of the table, the same next window for all lanes) and
// each lane reads a data-dependent slot inside the current window: the access pattern of a tree level with nothing
// around it (no feature load, no compare).  This is the denominator a walk can be held against (< 1 by construction).
__global__ void __launch_bounds__(1024, 1) gather_probe_coherent_kernel(const uint2 *__restrict__ tbl, uint32_t n_windows,
                                                                       uint32_t slots_per_window, int iters, unsigned int *sink) {
    uint32_t win[kProbeChains], off[kProbeChains];
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int c = 0; c < kProbeChains; ++c) {
        win[c] = (warp * 2654435761u + (uint32_t)c * 40503u) % n_windows;
        off[c] = (lane * 7u + (uint32_t)c) & (slots_per_window - 1u);
    }
    uint32_t acc = 0;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int c = 0; c < kProbeChains; ++c) {
            const uint2 v = __ldg(tbl + (size_t)win[c] * slots_per_window + off[c]);
            win[c] = v.x;
            off[c] = (v.y + lane * 5u) & (slots_per_window - 1u);
            acc ^= v.y;
        }
    }
    if (acc == 0x12345678u) atomicAdd(sink, 1u);
}

extern "C" int fmc_gather_probe_coherent(fmc_ctx *c, int64_t table_bytes, int32_t window_bytes, int32_t iters, double *out3) {
    if (!c || !out3 || table_bytes < 1024 || iters <= 0 || window_bytes < 8 || (window_bytes & (window_bytes - 1)) ||
        window_bytes > table_bytes)
        return fail(FMC_ERR_INVALID, "fmc_gather_probe_coherent: bad argument (window_bytes must be a power of two)");
    CK(cudaSetDevice(c->device));
    const uint32_t spw = (uint32_t)(window_bytes / 8), nw = (uint32_t)(table_bytes / window_bytes);
    std::vector<uint32_t> perm(nw);
    for (uint32_t i = 0; i < nw; ++i) perm[i] = i;
    uint64_t s = 0x9E3779B97F4A7C15ull;
    for (uint32_t i = nw - 1; i > 0; --i) {        // Sattolo: one cycle through every window
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        const uint32_t j = (uint32_t)((s >> 33) % i);
        std::swap(perm[i], perm[j]);
    }
    std::vector<uint2> h((size_t)nw * spw);
    for (uint32_t w = 0; w < nw; ++w)
        for (uint32_t k = 0; k < spw; ++k) {
            s = s * 6364136223846793005ull + 1442695040888963407ull;
            h[(size_t)w * spw + k] = make_uint2(perm[w], (uint32_t)(s >> 35));
        }
    uint2 *d = nullptr;
    unsigned int *sink = nullptr;
    CK(cudaMalloc(&d, h.size() * 8));
    cudaError_t e = cudaMalloc(&sink, 4);
    if (e != cudaSuccess) { cudaFree(d); return fail(FMC_ERR_CUDA, cudaGetErrorString(e)); }
    cudaMemcpy(d, h.data(), h.size() * 8, cudaMemcpyHostToDevice);
    cudaMemset(sink, 0, 4);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int grid = c->prop.multiProcessorCount;
    gather_probe_coherent_kernel<<<grid, 1024>>>(d, nw, spw, iters / 4 + 1, sink);      // warm-up
    float best = 1e30f;
    for (int r = 0; r < 3; ++r) {
        cudaEventRecord(e0);
        gather_probe_coherent_kernel<<<grid, 1024>>>(d, nw, spw, iters, sink);
        cudaEventRecord(e1);
        e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d); cudaFree(sink);
    if (e != cudaSuccess) return fail(FMC_ERR_CUDA, std::string("gather_probe_coherent_kernel: ") + cudaGetErrorString(e));
    const double warp_gathers = (double)grid * 32.0 * kProbeChains * (double)iters;
    out3[0] = warp_gathers * 32.0 * 8.0 / ((double)best * 1e-3) / 1e9;    // GB/s of gathered slots (8 bytes x lanes)
    out3[1] = warp_gathers / ((double)best * 1e-3);                       // warp-level gather instructions per second
    out3[2] = (double)best;                                               // ms
    return FMC_OK;
}

// Host-only packing entry point: lets CPU tests inspect the specialised tables without a GPU.  It
// performs no evaluation -- tests walk the returned tables themselves.
//   mode 0 = simulation preset (timeouts + SP+ folded to `fold_value`), 1 = predict preset.
// Returns the number of node slots, or a negative status; fills up to the given capacities.
static int64_t pack_host_impl(const fmc_forest_desc *d, int32_t mode, int32_t col0, int32_t col1,
                              const double *fold_value17, int32_t n_scaled, const int32_t *scaler_cols,
                              const double *scaler_mean, const double *scaler_scale, int32_t tree_begin,
                              int32_t tree_end, int32_t n_dyn, const int32_t *dyn_cols, const int32_t *dyn_rows,
                              uint64_t *slots_out, int64_t slots_cap, uint64_t *stream_out,
                              int64_t stream_cap, uint64_t *consts_out, int64_t consts_cap, int32_t *info_out) {
    if (!d) return fail(FMC_ERR_INVALID, "fmc_pack_forest_host: desc is NULL");
    HostForest f;
    f.assign(*d);
    prescale(f);
    PackSpec s;
    if (mode == 0) preset_sim(s); else preset_predict(s);
    s.active[0] = col0; s.active[1] = col1;
    if (n_dyn < 0 || n_dyn > (int)(sizeof(s.dyn_col) / sizeof(s.dyn_col[0]))) return fail(FMC_ERR_INVALID, "fmc_pack_forest_host_dyn: bad n_dyn");
    s.n_dyn = n_dyn;
    for (int i = 0; i < n_dyn; ++i) { s.dyn_col[i] = dyn_cols[i]; s.dyn_row[i] = (int8_t)dyn_rows[i]; }
    if (fold_value17) for (int k = 0; k < kNumMax; ++k) s.fold_value[k] = fold_value17[k];
    if (n_scaled < 0 || n_scaled > 16) return fail(FMC_ERR_INVALID, "fmc_pack_forest_host: n_scaled must be 0..16");
    for (int j = 0; j < n_scaled; ++j)
        if (scaler_cols[j] < 0 || scaler_cols[j] >= kNumMax) return fail(FMC_ERR_INVALID, "fmc_pack_forest_host: scaler column outside the 17 numerics");
    s.n_scaled = n_scaled;
    for (int j = 0; j < n_scaled && j < 16; ++j) { s.scaler_cols[j] = scaler_cols[j]; s.scaler_mean[j] = scaler_mean[j]; s.scaler_scale[j] = scaler_scale[j]; }
    s.tree_begin = tree_begin; s.tree_end = tree_end;
    PackedForest pf;
    const std::string err = pack_forest(f, s, pf);
    if (!err.empty()) return fail(FMC_ERR_CAPACITY, err);
    if (info_out) {
        info_out[0] = pf.rounds; info_out[1] = pf.max_depth; info_out[2] = pf.n_outputs; info_out[3] = kIlp;
        info_out[4] = s.ninf_row; info_out[5] = (int32_t)pf.stream.size(); info_out[6] = (int32_t)pf.consts.size();
        info_out[7] = (int32_t)pf.constants;
        for (int k = 0; k < 8; ++k) {
            info_out[8 + k] = (int32_t)pf.stream_off[k]; info_out[16 + k] = (int32_t)pf.n_groups[k];
            info_out[24 + k] = (int32_t)pf.consts_off[k];
        }
    }
    if (slots_out && (int64_t)pf.slots.size() <= slots_cap) std::memcpy(slots_out, pf.slots.data(), pf.slots.size() * 8);
    if (stream_out && (int64_t)pf.stream.size() <= stream_cap) std::memcpy(stream_out, pf.stream.data(), pf.stream.size() * 8);
    if (consts_out && (int64_t)pf.consts.size() <= consts_cap) std::memcpy(consts_out, pf.consts.data(), pf.consts.size() * 8);
    return (int64_t)pf.slots.size();
}

// Host-only: the exact-memo key (fmc_memo.hpp) of n states on the forest specialised like fmc_set_matchups would
// specialise it -- the same build_rank_spec / memo_key code the kernel runs.  CPU tests use it to check, against the
// oracle, that states sharing a key share their margins bit for bit.
extern "C" int64_t fmc_memo_keys_host(const fmc_forest_desc *d, int32_t family, int32_t col0, int32_t col1,
                                      const double *fold_value17, int32_t n_scaled, const int32_t *scaler_cols,
                                      const double *scaler_mean, const double *scaler_scale, int64_t n,
                                      const double *states, uint64_t *keys_out, int32_t *info_out) {
    if (!d || family < 0 || family >= kMemoFams || n < 0 || (n > 0 && (!states || !keys_out)))
        return fail(FMC_ERR_INVALID, "fmc_memo_keys_host: bad argument");
    if (n_scaled < 0 || n_scaled > 16) return fail(FMC_ERR_INVALID, "fmc_memo_keys_host: n_scaled must be 0..16");
    HostForest f;
    f.assign(*d);
    prescale(f);
    PackSpec s;
    preset_sim(s);
    s.active[0] = col0; s.active[1] = col1;
    if (fold_value17) for (int k = 0; k < kNumMax; ++k) s.fold_value[k] = fold_value17[k];
    RankSpecInput in;
    in.xgb = f.kind == FMC_KIND_XGB;
    in.zm = in.xgb && f.zero_is_missing;
    in.play_model = family == FMC_PLAY_MODEL;
    s.n_scaled = n_scaled;
    for (int j = 0; j < n_scaled; ++j) {
        if (scaler_cols[j] < 0 || scaler_cols[j] >= kNumMax) return fail(FMC_ERR_INVALID, "fmc_memo_keys_host: scaler column outside the 17 numerics");
        s.scaler_cols[j] = scaler_cols[j]; s.scaler_mean[j] = scaler_mean[j]; s.scaler_scale[j] = scaler_scale[j];
        if (in.play_model && scaler_cols[j] < 6) { in.pm_scaled[scaler_cols[j]] = 1; in.pm_mean[scaler_cols[j]] = scaler_mean[j]; in.pm_scale[scaler_cols[j]] = scaler_scale[j]; }
    }
    PackedForest pf;
    const std::string err = pack_forest(f, s, pf);
    if (!err.empty()) return fail(FMC_ERR_CAPACITY, err);
    std::vector<RankSpec> rsv(1);
    RankSpec &rs = rsv[0];
    const std::string why = build_rank_spec(pf.row_thr, in, rs);
    if (info_out) {
        info_out[0] = (int32_t)rs.enabled; info_out[1] = (int32_t)rs.n_thr[0]; info_out[2] = (int32_t)rs.n_thr[1];
        info_out[3] = (int32_t)pf.constants;
    }
    if (!rs.enabled) { g_err = why; return 0; }
    for (int64_t i = 0; i < n; ++i) {
        const double *x = states + i * 5;
        const int down = (int)x[0], sd = (int)x[3], sec = (int)x[4];
        float v1 = (float)x[1], v2 = (float)x[2];
        if (in.play_model) {
            if (in.pm_scaled[1]) v1 = (float)((x[1] - in.pm_mean[1]) / in.pm_scale[1]);
            if (in.pm_scaled[2]) v2 = (float)((x[2] - in.pm_mean[2]) / in.pm_scale[2]);
        }
        keys_out[i] = in.xgb ? memo_key<true>(&rs, family, 0, 0, down, x[1], x[2], sd, sec, v1, v2)
                             : memo_key<false>(&rs, family, 0, 0, down, x[1], x[2], sd, sec, v1, v2);
    }
    return 1;
}

extern "C" int64_t fmc_pack_forest_host(const fmc_forest_desc *d, int32_t mode, int32_t col0, int32_t col1,
                                        const double *fold_value17, int32_t n_scaled, const int32_t *scaler_cols,
                                        const double *scaler_mean, const double *scaler_scale, int32_t tree_begin,
                                        int32_t tree_end, uint64_t *slots_out, int64_t slots_cap, uint64_t *stream_out,
                                        int64_t stream_cap, uint64_t *consts_out, int64_t consts_cap, int32_t *info_out) {
    return pack_host_impl(d, mode, col0, col1, fold_value17, n_scaled, scaler_cols, scaler_mean, scaler_scale, tree_begin,
                          tree_end, 0, nullptr, nullptr, slots_out, slots_cap, stream_out, stream_cap, consts_out,
                          consts_cap, info_out);
}

extern "C" int64_t fmc_pack_forest_host_dyn(const fmc_forest_desc *d, int32_t mode, int32_t col0, int32_t col1,
                                            const double *fold_value17, int32_t n_dyn, const int32_t *dyn_cols,
                                            const int32_t *dyn_rows, uint64_t *slots_out, int64_t slots_cap,
                                            uint64_t *stream_out, int64_t stream_cap, uint64_t *consts_out,
                                            int64_t consts_cap, int32_t *info_out) {
    return pack_host_impl(d, mode, col0, col1, fold_value17, 0, nullptr, nullptr, nullptr, 0, -1, n_dyn, dyn_cols, dyn_rows,
                          slots_out, slots_cap, stream_out, stream_cap, consts_out, consts_cap, info_out);
}
