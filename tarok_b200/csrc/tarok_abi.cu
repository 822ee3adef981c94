// C ABI of libtarok_b200.so (declared in include/tarok_b200.h): handle, device buffers, launches.
// No torch, no C++ types across the boundary.  Every launch goes to the caller's stream.
#include "../../include/tarok_b200.h"

#include <dlfcn.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "tarok_host.h"
#include "tarok_kernels.cuh"
#include "tarok_obs.cuh"

using tk::u64;
using tk::u32;

#define TK_MAX_CHUNKS 32
#define TK_GRAPH_MODES 20                       /* contracts 0..9, synthetic modes 16..18 */

struct tarok_env {
    int device;
    int sm_count;
    int step_impl;                             // 0 auto, 1 plain k_step, 2 persistent TMA-staged k_step_tma
    int pdl;                                   // chain play_step launches with programmatic dependent launch
    int lockstep;                              // pass the lock-step hint to play_step (specialised per trick position)
    int lock_plays;                            // plays made by every live game since the last deal, -1 = unknown
    uint32_t epoch;                            // draw-cache epoch (set_first_gid)
    int use_graph;                             // tarok_rollout_stepwise replays a captured CUDA graph (TAROK_OPT_GRAPH, default on)
    cudaGraphExec_t graphs[TK_GRAPH_MODES];    // one per rollout mode, captured on first use; dropped when an option changes
    cudaStream_t s_cap;                        // private stream the graphs are captured on
    tk::RunParams* run_dev;                    // {first_gid, rc_epoch} the GRAPH kernel variants read (rewritten before every replay)
    int capturing;                             // launch the GRAPH variants (set while a rollout graph is being captured)
    cudaGraphExec_t bucket_graph;              // tarok_obs_buckets_host: hist + scan + scatter + counts copy as one launch
    const void* bucket_key[5];                 // the arguments that graph was captured with
    int lazy_mask;                             // chains of random steps write legal masks in their last launch only (default on)
    int materialise;                           // tarok_score writes the materialised piles / talon back (default on)
    int chunks;                                // upload/compute/download pipeline depth of the host-buffer entries
    u32 flags;
    tk::Env e;
    // staging buffers of the host-buffer entry point
    uint8_t* st_perm; uint8_t* st_contract; uint8_t* st_declarer; uint8_t* st_king;
    int staging_ready;                         // set only after every stream / event / buffer below exists
    tk::u32* cta_hist;                         // scratch of tarok_obs_buckets: [n_alloc / 256][128]
    tarok_pack_pool* pool;                     // host threads of tarok_rollout_host_packed (lazily created)
    uint8_t* pin_rec;                          // pinned scratch: the records being uploaded [n_alloc x TAROK_RECORD_BYTES]
    int pack_used[TK_MAX_CHUNKS];              // chunk c of the pinned scratch has an upload recorded on ev_up[c]
    cudaStream_t s_up, s_down;                 // internal copy streams of the chunked host pipeline
    cudaEvent_t ev_fork, ev_join, ev_up[TK_MAX_CHUNKS], ev_done[TK_MAX_CHUNKS];
    std::atomic<int> exports;
    u64 launches;
    char err[512];
};

static thread_local char g_create_err[512] = "";

static int fail(tarok_env* h, int code, const char* fmt, ...) {
    char* dst = h ? h->err : g_create_err;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}

#define TK_CUDA(h, call)                                                                          \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(h, -2, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define TK_CHECK_HANDLE(h) do { if (!(h)) return fail(nullptr, -1, "null handle"); } while (0)
#define TK_LAUNCH_OK(h)                                                                            \
    do {                                                                                          \
        cudaError_t _e = cudaGetLastError();                                                      \
        if (_e != cudaSuccess) return fail(h, -3, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
        (h)->launches++;                                                                          \
    } while (0)

// Staging resources of the host-buffer entries: every member is null until created, so a partial set can be torn down.
static void free_staging(tarok_env* h) {
    if (h->s_up) cudaStreamDestroy(h->s_up);
    if (h->s_down) cudaStreamDestroy(h->s_down);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (int c = 0; c < TK_MAX_CHUNKS; c++) {
        if (h->ev_up[c]) cudaEventDestroy(h->ev_up[c]);
        if (h->ev_done[c]) cudaEventDestroy(h->ev_done[c]);
    }
    cudaFree(h->st_perm); cudaFree(h->st_contract); cudaFree(h->st_declarer); cudaFree(h->st_king);
    h->s_up = h->s_down = nullptr; h->ev_fork = h->ev_join = nullptr;
    memset(h->ev_up, 0, sizeof(h->ev_up)); memset(h->ev_done, 0, sizeof(h->ev_done));
    h->st_perm = h->st_contract = h->st_declarer = h->st_king = nullptr;
    h->staging_ready = 0;
}

// Every change of the first global game id starts a new epoch of the draw cache (tarok_kernels.cuh, step_lock): entries
// written under another id can never match a tag again.  28 bits of epoch, 4 bits of trick index.
static inline void set_first_gid(tarok_env* h, u64 first_gid) {
    h->e.first_gid = first_gid;
    h->epoch = (h->epoch % 0x0FFFFFFFu) + 1u;                 // 1 .. 2^28 - 1: never 0, the value of a cleared entry
    h->e.rc_epoch = h->epoch << 4;
}

// Draw cache policy: all three positions while the state a chain of steps touches stays inside the 126 MB L2 (the cache
// adds 12 B per game to it); beyond that the step kernels are HBM-bound, the extra 4-8 B per game and step cost more than
// the ten Philox rounds they save (8 M deals, uniform bids: 72.5 us per launch without, 74.9 us with rows 1-2), so it is off.
static inline u32 default_draw_cache_rows(u64 n_alloc) { return n_alloc <= (3ull << 20) ? 3u : 0u; }

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline unsigned grid1(u64 n_alloc) { return (unsigned)(n_alloc / tk::CTA); }        // one game per lane
static inline unsigned grid2(u64 n_alloc) { return (unsigned)(n_alloc / tk::TILE); }       // two games per lane

struct DeviceGuard {
    int prev; bool ok;
    explicit DeviceGuard(int dev) : prev(0), ok(false) {
        if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
    }
    ~DeviceGuard() { if (ok) cudaSetDevice(prev); }
};

// play_step launcher.  Default: the plain kernel, one 512-game tile per CTA, compiled per trick position for lock-step
// batches (the hint) with programmatic dependent launch; TAROK_OPT_STEP_IMPL=2 selects the persistent TMA-staged variant
// (one CTA per resident slot, 4 per SM), which measures slower on B200 and is kept for comparison (tools/step_ab.py).
template <bool RANDOM, bool MASK = true, bool GRAPH = false>
static void launch_step(tarok_env* h, const uint8_t* action, cudaStream_t s) {
    const unsigned tiles = grid2(h->e.n_alloc);
    const unsigned resident = (unsigned)h->sm_count * 4u;
    const bool tma = h->step_impl == 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(tma ? (tiles < resident ? tiles : resident) : tiles);
    cfg.blockDim = dim3(tk::CTA);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // PDL: overlap this launch with the previous tail
    at[0].val.programmaticStreamSerializationAllowed = h->pdl ? 1 : 0;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    // TAROK_OPT_STEP_IMPL = 3: the persistent prefetching kernel for what it covers -- interior launches (no masks) of a
    // lock-step chain of random steps with the draw cache on for all three positions; everything else takes the plain kernel
    const bool pp = h->step_impl == 3 && RANDOM && !MASK && h->lockstep && h->lock_plays >= 0 && h->e.rc_rows == 3u;
    if (pp) {
        const int hint = h->lock_plays;
        const int pos = hint & 3;
        const unsigned per_sm = pos == 3 ? TK_PP_BLOCKS_3 : TK_PP_BLOCKS_012;
        const unsigned slots = (unsigned)h->sm_count * per_sm;
        cfg.gridDim = dim3(tiles < slots ? tiles : slots);
        switch (pos) {
            case 0: cfg.dynamicSmemBytes = 2 * sizeof(tk::LockStage<0>); cudaLaunchKernelEx(&cfg, tk::k_step_pp<0, GRAPH>, h->e, hint); break;
            case 1: cfg.dynamicSmemBytes = 2 * sizeof(tk::LockStage<1>); cudaLaunchKernelEx(&cfg, tk::k_step_pp<1, GRAPH>, h->e, hint); break;
            case 2: cfg.dynamicSmemBytes = 2 * sizeof(tk::LockStage<2>); cudaLaunchKernelEx(&cfg, tk::k_step_pp<2, GRAPH>, h->e, hint); break;
            default: cfg.dynamicSmemBytes = 2 * sizeof(tk::LockStage<3>); cudaLaunchKernelEx(&cfg, tk::k_step_pp<3, GRAPH>, h->e, hint); break;
        }
    } else if (tma) cudaLaunchKernelEx(&cfg, tk::k_step_tma<RANDOM>, h->e, action);
    else {
        const int hint = h->lockstep ? h->lock_plays : -1;
        switch (hint >= 0 ? (hint & 3) : 4) {
            case 0: cudaLaunchKernelEx(&cfg, tk::k_step<RANDOM, 0, MASK, GRAPH>, h->e, action, hint); break;
            case 1: cudaLaunchKernelEx(&cfg, tk::k_step<RANDOM, 1, MASK, GRAPH>, h->e, action, hint); break;
            case 2: cudaLaunchKernelEx(&cfg, tk::k_step<RANDOM, 2, MASK, GRAPH>, h->e, action, hint); break;
            case 3: cudaLaunchKernelEx(&cfg, tk::k_step<RANDOM, 3, MASK, GRAPH>, h->e, action, hint); break;
            default: cudaLaunchKernelEx(&cfg, tk::k_step<RANDOM, -1, MASK, GRAPH>, h->e, action, hint); break;
        }
    }
    // lock-step bookkeeping (only a hint to the kernel, which verifies it per warp): every live game has made
    // `lock_plays` plays since the last deal; one more after this launch
    if (h->lock_plays >= 0) h->lock_plays = h->lock_plays < 47 ? h->lock_plays + 1 : -1;
}

// `count` back-to-back in-kernel random steps.  Only the last launch writes legal masks (nobody can observe the interior
// ones); with the TMA-staged implementation or the eager-mask option every launch does.
static int random_chain(tarok_env* h, uint32_t count, cudaStream_t s) {
    for (uint32_t t = 0; t < count; t++) {
        const bool lazy = t + 1 < count && h->lazy_mask && h->step_impl != 2;
        if (h->capturing) {                                // kernels of a rollout graph: run parameters from device memory
            if (lazy) launch_step<true, false, true>(h, nullptr, s);
            else launch_step<true, true, true>(h, nullptr, s);
        } else {
            if (lazy) launch_step<true, false>(h, nullptr, s);
            else launch_step<true, true>(h, nullptr, s);
        }
        TK_LAUNCH_OK(h);
    }
    return 0;
}

extern "C" {

// The captured graphs freeze every option (kernel variant, launch attributes, parameters): any change drops them.
static void drop_graphs(tarok_env* h) {
    if (h->bucket_graph) { cudaGraphExecDestroy(h->bucket_graph); h->bucket_graph = nullptr; }
    for (int m = 0; m < TK_GRAPH_MODES; m++)
        if (h->graphs[m]) { cudaGraphExecDestroy(h->graphs[m]); h->graphs[m] = nullptr; }
}

int tarok_set_option(tarok_t* h, int option, int64_t value) {
    TK_CHECK_HANDLE(h);
    drop_graphs(h);
    if (option == TAROK_OPT_GRAPH && value >= 0 && value <= 2) { h->use_graph = (int)value; return 0; }
    if (option == TAROK_OPT_STEP_IMPL && value >= 0 && value <= 3) { h->step_impl = (int)value; return 0; }
    if (option == TAROK_OPT_PDL && (value == 0 || value == 1)) { h->pdl = (int)value; return 0; }
    if (option == TAROK_OPT_LOCKSTEP && (value == 0 || value == 1)) { h->lockstep = (int)value; return 0; }
    if (option == TAROK_OPT_MATERIALISE && (value == 0 || value == 1)) { h->materialise = (int)value; return 0; }
    if (option == TAROK_OPT_LAZY_MASK && (value == 0 || value == 1)) { h->lazy_mask = (int)value; return 0; }
    if (option == TAROK_OPT_DRAW_CACHE && (value == -1 || value == 0 || value == 2 || value == 3)) {
        h->e.rc_rows = value >= 0 ? (u32)value : default_draw_cache_rows(h->e.n_alloc);
        return 0;
    }
    if (option == TAROK_OPT_CHUNKS && value >= 1 && value <= TK_MAX_CHUNKS) { h->chunks = (int)value; return 0; }
    return fail(h, -1, "unknown option %d / value %lld", option, (long long)value);
}

int tarok_create(int device, uint64_t n_games, uint64_t seed, uint32_t flags, tarok_t** out) {
    if (!out) return fail(nullptr, -1, "out is null");
    *out = nullptr;
    if (n_games == 0 || n_games > (1ull << 29)) return fail(nullptr, -1, "n_games must be in 1..2^29");
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0)
        return fail(nullptr, -2, "no CUDA device: %s (tarok_b200 has no CPU fallback)", cudaGetErrorString(ce));
    if (device < 0 || device >= count) return fail(nullptr, -1, "device %d out of range (0..%d)", device, count - 1);
    DeviceGuard dg(device);
    cudaDeviceProp prop;
    TK_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, -2, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    tarok_env* h = new (std::nothrow) tarok_env();
    if (!h) return fail(nullptr, -4, "out of host memory");
    memset(&h->e, 0, sizeof(h->e));
    h->device = device; h->sm_count = prop.multiProcessorCount; h->step_impl = 0; h->pdl = 1; h->lockstep = 1; h->lock_plays = -1; h->lazy_mask = 1; h->materialise = 1; h->chunks = 8; h->flags = flags; h->launches = 0; h->exports = 0; h->err[0] = 0;
    h->st_perm = h->st_contract = h->st_declarer = h->st_king = nullptr;
    h->s_up = h->s_down = nullptr; h->ev_fork = h->ev_join = nullptr; h->staging_ready = 0;
    memset(h->ev_up, 0, sizeof(h->ev_up)); memset(h->ev_done, 0, sizeof(h->ev_done));
    h->use_graph = 1; memset(h->graphs, 0, sizeof(h->graphs)); h->s_cap = nullptr; h->run_dev = nullptr; h->capturing = 0; h->e.run_ptr = nullptr; h->bucket_graph = nullptr;
    h->cta_hist = nullptr; h->pool = nullptr; h->pin_rec = nullptr; memset(h->pack_used, 0, sizeof(h->pack_used));
    const u64 na = (n_games + tk::TILE - 1) / tk::TILE * tk::TILE;
    h->e.n = n_games; h->e.n_alloc = na; h->epoch = 0; set_first_gid(h, 0);
    h->e.rc_rows = default_draw_cache_rows(na);
    tk::philox_keys_init(h->e.rng, seed);
#define TK_ALLOC(ptr, bytes)                                                       \
    do {                                                                           \
        cudaError_t _e = cudaMalloc((void**)&(ptr), (bytes));                      \
        if (_e != cudaSuccess) {                                                   \
            fail(nullptr, -4, "cudaMalloc(%llu B) failed: %s", (unsigned long long)(bytes), cudaGetErrorString(_e)); \
            tarok_destroy(h);                                                      \
            return -4;                                                             \
        }                                                                          \
    } while (0)
    TK_ALLOC(h->e.hands, 4 * na * 8);
    TK_ALLOC(h->e.piles, 4 * na * 8);
    TK_ALLOC(h->e.talon, na * 8);
    TK_ALLOC(h->e.torder, na * 8);
    TK_ALLOC(h->e.meta, na * 8);
    TK_ALLOC(h->e.mask, na * 8);
    TK_ALLOC(h->e.scores, na * 8);
    TK_ALLOC(h->e.stats, TAROK_STATS_LEN * 8);
    TK_ALLOC(h->e.tricklog, 12 * na * 4);
    cudaMemset(h->e.tricklog, 0, 12 * na * 4);
    TK_ALLOC(h->e.dpts, na);
    cudaMemset(h->e.dpts, 0, na);
    TK_ALLOC(h->run_dev, sizeof(tk::RunParams));
    h->e.run_ptr = h->run_dev;
    TK_ALLOC(h->e.rcache, 3 * (na / 2) * sizeof(uint2));
    cudaMemset(h->e.rcache, 0, 3 * (na / 2) * sizeof(uint2));
    if (flags & TAROK_FLAG_HISTORY) {
        TK_ALLOC(h->e.hist, 48 * na);
        TK_ALLOC(h->e.hands0, 4 * na * 8);
        TK_ALLOC(h->e.discard, na * 8);
        TK_ALLOC(h->e.qmax_hist, 48 * na * 4);
        cudaMemset(h->e.qmax_hist, 0, 48 * na * 4);
        cudaMemset(h->e.hist, 0xFF, 48 * na);
    }
#undef TK_ALLOC
    cudaMemset(h->e.stats, 0, TAROK_STATS_LEN * 8);
    cudaMemset(h->e.scores, 0, na * 8);
    cudaMemset(h->e.mask, 0, na * 8);
    // every game starts "finished/padded" until dealt
    {
        tk::Env e = h->e; e.n = 0;
        tk::k_deal<<<grid1(na), tk::CTA>>>(e);
        cudaError_t _e = cudaDeviceSynchronize();
        if (_e != cudaSuccess) {
            fail(nullptr, -3, "initial kernel failed: %s (is libtarok_b200.so built for this GPU?)", cudaGetErrorString(_e));
            tarok_destroy(h);
            return -3;
        }
    }
    *out = h;
    return 0;
}

int tarok_destroy(tarok_t* h) {
    if (!h) return 0;
    if (h->exports.load() != 0) return fail(h, -5, "%d exported tensors still alive", h->exports.load());
    DeviceGuard dg(h->device);
    cudaFree(h->e.hands); cudaFree(h->e.piles); cudaFree(h->e.talon); cudaFree(h->e.torder);
    cudaFree(h->e.meta); cudaFree(h->e.mask); cudaFree(h->e.scores); cudaFree(h->e.stats); cudaFree(h->e.tricklog);
    cudaFree(h->e.hist); cudaFree(h->e.hands0); cudaFree(h->e.discard); cudaFree(h->e.qmax_hist); cudaFree(h->e.dpts); cudaFree(h->e.rcache);
    free_staging(h);
    drop_graphs(h);
    if (h->s_cap) cudaStreamDestroy(h->s_cap);
    cudaFree(h->run_dev);
    cudaFree(h->cta_hist);
    tarok_pack_pool_destroy(h->pool);
    if (h->pin_rec) cudaFreeHost(h->pin_rec);
    delete h;
    return 0;
}

const char* tarok_last_error(const tarok_t* h) { return h ? h->err : g_create_err; }
uint64_t tarok_n_games(const tarok_t* h) { return h ? h->e.n : 0; }
uint64_t tarok_n_alloc(const tarok_t* h) { return h ? h->e.n_alloc : 0; }
uint64_t tarok_launch_count(const tarok_t* h) { return h ? h->launches : 0; }

// ---- deal ---------------------------------------------------------------------------------------

static void clear_hist(tarok_t* h, void* stream) {
    if (h->e.hist) cudaMemsetAsync(h->e.hist, 0xFF, 48 * h->e.n_alloc, S(stream));
}

int tarok_deal(tarok_t* h, uint64_t first_global_game_id, void* stream) {
    TK_CHECK_HANDLE(h);
    DeviceGuard dg(h->device);
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    clear_hist(h, stream);
    tk::k_deal<<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_set_deals(tarok_t* h, const uint8_t* perm_dev, uint64_t first_global_game_id, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!perm_dev) return fail(h, -1, "perm_dev is null");
    DeviceGuard dg(h->device);
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    clear_hist(h, stream);
    tk::k_set_deals<<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, perm_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_export_perm(tarok_t* h, uint8_t* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!out_dev) return fail(h, -1, "out_dev is null");
    DeviceGuard dg(h->device);
    tk::k_export_perm<<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, out_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

// ---- auction / contract -----------------------------------------------------------------------------

int tarok_auction(tarok_t* h, const uint8_t* intent_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!intent_dev) return fail(h, -1, "intent_dev is null");
    if (((uintptr_t)intent_dev) & 3u) return fail(h, -1, "intent_dev must be 4-byte aligned");
    DeviceGuard dg(h->device);
    tk::k_begin<tk::SRC_INTENTS><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, 0u, intent_dev, nullptr, nullptr);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_auction_synth(tarok_t* h, uint32_t mode, void* stream) {
    TK_CHECK_HANDLE(h);
    if (mode != TAROK_MODE_AUCTION_UNIFORM && mode != TAROK_MODE_AUCTION_BOT) return fail(h, -1, "bad auction mode %u", mode);
    DeviceGuard dg(h->device);
    tk::k_begin<tk::SRC_SYNTH><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, mode, nullptr, nullptr, nullptr);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_force_contract(tarok_t* h, const uint8_t* contract_dev, const uint8_t* declarer_dev, const uint8_t* king_dev,
                         void* stream) {
    TK_CHECK_HANDLE(h);
    if (!contract_dev || !declarer_dev) return fail(h, -1, "contract_dev/declarer_dev is null");
    DeviceGuard dg(h->device);
    tk::k_begin<tk::SRC_FORCED><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, 0u, contract_dev, declarer_dev, king_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_force_contract_synth(tarok_t* h, uint32_t mode, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!(mode <= TAROK_ODPRTI_BERAC || mode == TAROK_MODE_NAVADNA_MIX)) return fail(h, -1, "bad contract mode %u", mode);
    DeviceGuard dg(h->device);
    tk::k_begin<tk::SRC_SYNTH><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, mode, nullptr, nullptr, nullptr);
    TK_LAUNCH_OK(h);
    return 0;
}

// ---- exchange ---------------------------------------------------------------------------------------

int tarok_exchange(tarok_t* h, const uint8_t* group_dev, const uint64_t* discard_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!group_dev || !discard_dev) return fail(h, -1, "group_dev/discard_dev is null");
    DeviceGuard dg(h->device);
    tk::k_exchange<false><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, 0u, group_dev, (const u64*)discard_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_exchange_synth(tarok_t* h, uint32_t random_group, void* stream) {
    TK_CHECK_HANDLE(h);
    DeviceGuard dg(h->device);
    tk::k_exchange<true><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, random_group, nullptr, nullptr);
    TK_LAUNCH_OK(h);
    return 0;
}

// ---- play -------------------------------------------------------------------------------------------

int tarok_legal_mask(tarok_t* h, uint64_t* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!out_dev) return fail(h, -1, "out_dev is null");
    if (((uintptr_t)out_dev) & 15u) return fail(h, -1, "out_dev must be 16-byte aligned");
    DeviceGuard dg(h->device);
    tk::k_legal_mask<<<grid2(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, (u64*)out_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_hands_by_seat(tarok_t* h, uint64_t* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!out_dev) return fail(h, -1, "out_dev is null");
    DeviceGuard dg(h->device);
    tk::k_hands_by_seat<<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, (u64*)out_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_step(tarok_t* h, const uint8_t* card_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!card_dev) return fail(h, -1, "card_dev is null");
    if (((uintptr_t)card_dev) & 1u) return fail(h, -1, "card_dev must be 2-byte aligned");
    DeviceGuard dg(h->device);
    launch_step<false>(h, card_dev, S(stream));
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_step_random(tarok_t* h, void* stream) {
    TK_CHECK_HANDLE(h);
    DeviceGuard dg(h->device);
    launch_step<true>(h, nullptr, S(stream));
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_steps_random(tarok_t* h, uint32_t count, void* stream) {
    TK_CHECK_HANDLE(h);
    DeviceGuard dg(h->device);
    return random_chain(h, count, S(stream));
}

// ---- score / stats ----------------------------------------------------------------------------------

int tarok_score(tarok_t* h, int16_t* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (out_dev && (((uintptr_t)out_dev) & 15u)) return fail(h, -1, "out_dev must be 16-byte aligned");
    DeviceGuard dg(h->device);
    u64* out = out_dev ? (u64*)out_dev : h->e.scores;
    u64 out_n = out_dev ? h->e.n : h->e.n_alloc;
    if (h->materialise) tk::k_score<true><<<grid2(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, out, out_n);
    else tk::k_score<false><<<grid2(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, out, out_n);
    TK_LAUNCH_OK(h);
    return 0;
}

// A new run seed for an existing handle (the Philox key of every synthetic draw): what tarok_create(seed) sets, without
// giving the device buffers back -- a caller that plays batch after batch under fresh seeds (Tarok.start / paralel_start with no
// seed given) keeps one handle.  Work already enqueued keeps the old key (kernel parameters are copied at launch).
int tarok_reseed(tarok_t* h, uint64_t seed) {
    TK_CHECK_HANDLE(h);
    drop_graphs(h);                                        // the captured kernels carry the old round keys
    tk::philox_keys_init(h->e.rng, seed);
    set_first_gid(h, h->e.first_gid);                      // a new draw-cache epoch: cached lanes belong to the old key
    return 0;
}

int tarok_reset_stats(tarok_t* h, void* stream) {
    TK_CHECK_HANDLE(h);
    DeviceGuard dg(h->device);
    TK_CUDA(h, cudaMemsetAsync(h->e.stats, 0, TAROK_STATS_LEN * 8, S(stream)));
    return 0;
}

int tarok_read_stats(tarok_t* h, int64_t* out_host, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!out_host) return fail(h, -1, "out_host is null");
    DeviceGuard dg(h->device);
    TK_CUDA(h, cudaMemcpyAsync(out_host, h->e.stats, TAROK_STATS_LEN * 8, cudaMemcpyDeviceToHost, S(stream)));
    TK_CUDA(h, cudaStreamSynchronize(S(stream)));
    return 0;
}

// ---- the one collective: all-reduce of the statistics vector (NCCL over NVLink / NVSwitch) ------------------------
// libnccl is resolved at run time (the process that owns the communicator has it loaded already), so the library
// itself carries no link-time dependency on NCCL.
typedef int (*nccl_allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);

int tarok_allreduce_stats(tarok_t* h, void* nccl_comm, int64_t* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!nccl_comm || !out_dev) return fail(h, -1, "nccl_comm/out_dev is null");
    static nccl_allreduce_fn fn = nullptr;
    if (!fn) {
        void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW);
        if (!lib) return fail(h, -6, "libnccl.so.2 not found: %s", dlerror());
        fn = (nccl_allreduce_fn)dlsym(lib, "ncclAllReduce");
        if (!fn) return fail(h, -6, "ncclAllReduce not found in libnccl");
    }
    DeviceGuard dg(h->device);
    const int rc = fn(h->e.stats, out_dev, TAROK_STATS_LEN, /*ncclInt64*/ 4, /*ncclSum*/ 0, nccl_comm, S(stream));
    if (rc != 0) return fail(h, -6, "ncclAllReduce failed with code %d", rc);
    return 0;
}

// ---- whole deals --------------------------------------------------------------------------------------

static int play_out_stepwise(tarok_t* h, uint32_t random_group, void* stream) {
    tk::k_exchange<true><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, random_group, nullptr, nullptr);
    TK_LAUNCH_OK(h);
    if (int rc = random_chain(h, 48, S(stream))) return rc;
    if (h->materialise) tk::k_score<true><<<grid2(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, h->e.scores, h->e.n_alloc);
    else tk::k_score<false><<<grid2(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, h->e.scores, h->e.n_alloc);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_setup_synth(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!(mode <= TAROK_ODPRTI_BERAC || (mode >= TAROK_MODE_NAVADNA_MIX && mode <= TAROK_MODE_AUCTION_BOT)))
        return fail(h, -1, "bad mode %u", mode);
    DeviceGuard dg(h->device);
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    clear_hist(h, stream);
    tk::k_setup_synth<false><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, mode);
    TK_LAUNCH_OK(h);
    return 0;
}

// setup -> 48 x play_step -> score, enqueued on `s` with the environment `env` (h->e, or its copy that reads the run
// parameters from device memory while a graph is being captured).
static int enqueue_rollout_stepwise(tarok_t* h, uint32_t mode, cudaStream_t s) {
    h->lock_plays = 0;
    clear_hist(h, s);
    if (h->capturing) tk::k_setup_synth<true><<<grid1(h->e.n_alloc), tk::CTA, 0, s>>>(h->e, mode);
    else tk::k_setup_synth<false><<<grid1(h->e.n_alloc), tk::CTA, 0, s>>>(h->e, mode);
    TK_LAUNCH_OK(h);
    if (int rc = random_chain(h, 48, s)) return rc;
    const unsigned grid = grid2(h->e.n_alloc);
    if (h->capturing) {
        if (h->materialise) tk::k_score<true, true><<<grid, tk::CTA, 0, s>>>(h->e, h->e.scores, h->e.n_alloc);
        else tk::k_score<false, true><<<grid, tk::CTA, 0, s>>>(h->e, h->e.scores, h->e.n_alloc);
    } else {
        if (h->materialise) tk::k_score<true><<<grid, tk::CTA, 0, s>>>(h->e, h->e.scores, h->e.n_alloc);
        else tk::k_score<false><<<grid, tk::CTA, 0, s>>>(h->e, h->e.scores, h->e.n_alloc);
    }
    TK_LAUNCH_OK(h);
    return 0;
}

// Captures the rollout of `mode` once (on a private stream: the caller's may be the legacy default stream, which cannot be
// captured) with the GRAPH kernel variants, which read first_gid / the draw-cache epoch from h->run_dev.
static int capture_rollout_graph(tarok_t* h, uint32_t mode) {
    if (!h->s_cap) TK_CUDA(h, cudaStreamCreateWithFlags(&h->s_cap, cudaStreamNonBlocking));
    cudaGraph_t g = nullptr;
    const uint64_t launches0 = h->launches;
    TK_CUDA(h, cudaStreamBeginCapture(h->s_cap, cudaStreamCaptureModeThreadLocal));
    h->capturing = 1;
    const int rc = enqueue_rollout_stepwise(h, mode, h->s_cap);
    h->capturing = 0;
    const cudaError_t ce = cudaStreamEndCapture(h->s_cap, &g);
    h->launches = launches0;                               // nothing ran yet
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) return fail(h, -2, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
    const cudaError_t ie = cudaGraphInstantiate(&h->graphs[mode], g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) { h->graphs[mode] = nullptr; return fail(h, -2, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
    return 0;
}

int tarok_rollout_stepwise(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!(mode <= TAROK_ODPRTI_BERAC || (mode >= TAROK_MODE_NAVADNA_MIX && mode <= TAROK_MODE_AUCTION_BOT)))
        return fail(h, -1, "bad mode %u", mode);
    DeviceGuard dg(h->device);
    cudaStream_t s = S(stream);
    set_first_gid(h, first_global_game_id);
    // 50 launches cost more host time than a small batch takes on the GPU: the whole rollout is replayed as ONE graph
    // launch (+ a one-thread kernel that hands over this call's first_gid and draw-cache epoch).  Not while the caller is
    // capturing `stream` itself (the launches below are then captured as they are), nor with the TMA-staged variant.
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (h->use_graph && (h->use_graph == 2 || h->e.n_alloc <= (3ull << 20)) && h->step_impl != 2 && mode < TK_GRAPH_MODES
        && cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone) {
        if (!h->graphs[mode] && capture_rollout_graph(h, mode) != 0) {
            h->use_graph = 0;                              // e.g. another capture is open in this thread: plain launches from now on
            cudaGetLastError();
            return enqueue_rollout_stepwise(h, mode, s);
        }
        tk::k_set_run<<<1, 1, 0, s>>>(h->run_dev, h->e.first_gid, h->e.rc_epoch);
        TK_LAUNCH_OK(h);
        TK_CUDA(h, cudaGraphLaunch(h->graphs[mode], s));
        h->launches += 50;                                 // the graph's kernels: setup + 48 play_steps + score (+ k_set_run above)
        h->lock_plays = -1;
        return 0;
    }
    cudaGetLastError();                                    // a failed capture query must not stick
    return enqueue_rollout_stepwise(h, mode, s);
}

int tarok_rollout_fused(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!(mode <= TAROK_ODPRTI_BERAC || (mode >= TAROK_MODE_NAVADNA_MIX && mode <= TAROK_MODE_AUCTION_BOT)))
        return fail(h, -1, "bad mode %u", mode);
    DeviceGuard dg(h->device);
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    clear_hist(h, stream);
    tk::k_rollout_fused<tk::DEALS_PHILOX><<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, mode, nullptr, nullptr, nullptr, nullptr,
                                                                           h->e.scores, 1, 0ull);
    TK_LAUNCH_OK(h);
    return 0;
}

// Lazily created: the copy streams, events and device staging buffers of the host-buffer entries.  The handle is marked
// ready only once everything exists; a failure half-way frees what was created, so the next call starts from scratch.
static int create_staging(tarok_t* h) {
    TK_CUDA(h, cudaStreamCreateWithFlags(&h->s_up, cudaStreamNonBlocking));
    TK_CUDA(h, cudaStreamCreateWithFlags(&h->s_down, cudaStreamNonBlocking));
    TK_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    TK_CUDA(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    for (int c = 0; c < TK_MAX_CHUNKS; c++) {
        TK_CUDA(h, cudaEventCreateWithFlags(&h->ev_up[c], cudaEventDisableTiming));
        TK_CUDA(h, cudaEventCreateWithFlags(&h->ev_done[c], cudaEventDisableTiming));
    }
    TK_CUDA(h, cudaMalloc((void**)&h->st_perm, h->e.n_alloc * 54));
    TK_CUDA(h, cudaMalloc((void**)&h->st_contract, h->e.n_alloc));
    TK_CUDA(h, cudaMalloc((void**)&h->st_declarer, h->e.n_alloc));
    TK_CUDA(h, cudaMalloc((void**)&h->st_king, h->e.n_alloc));
    return 0;
}
static int ensure_staging(tarok_t* h) {
    if (h->staging_ready) return 0;
    const int rc = create_staging(h);
    if (rc) { free_staging(h); return rc; }
    h->staging_ready = 1;
    return 0;
}

// Chunked pipeline shared by the two host-buffer entries: upload chunk c+1 (copy stream) while chunk c plays (caller's
// stream) and chunk c-1's scores go back (download stream).  `row` = bytes per deal of the input format (54: permutation
// rows + three 1-byte arrays; 20: deal records, which carry the contract themselves).
static int rollout_host_fused(tarok_t* h, const uint8_t* deals_host, size_t row, const uint8_t* contract_host,
                              const uint8_t* declarer_host, const uint8_t* king_host, int16_t* scores_host,
                              int64_t* stats_host, cudaStream_t s) {
    const u64 n = h->e.n;
    uint64_t bounds[TK_MAX_CHUNKS + 1];
    const int nchunks = tarok_chunk_bounds(n, h->chunks, tarok_pack_block_rows(), bounds);   // tapered: short fill and drain
    TK_CUDA(h, cudaEventRecord(h->ev_fork, s));
    TK_CUDA(h, cudaStreamWaitEvent(h->s_up, h->ev_fork, 0));
    TK_CUDA(h, cudaStreamWaitEvent(h->s_down, h->ev_fork, 0));
    for (int c = 0; c < nchunks; c++) {
        const u64 b = bounds[c], e_ = bounds[c + 1], len = e_ - b;
        TK_CUDA(h, cudaMemcpyAsync(h->st_perm + b * row, deals_host + b * row, len * row, cudaMemcpyHostToDevice, h->s_up));
        if (c == 0 && contract_host) {   // the three 1-byte-per-game inputs go up whole, right behind the first chunk of deals
            TK_CUDA(h, cudaMemcpyAsync(h->st_contract, contract_host, n, cudaMemcpyHostToDevice, h->s_up));
            TK_CUDA(h, cudaMemcpyAsync(h->st_declarer, declarer_host, n, cudaMemcpyHostToDevice, h->s_up));
            if (king_host) TK_CUDA(h, cudaMemcpyAsync(h->st_king, king_host, n, cudaMemcpyHostToDevice, h->s_up));
        }
        TK_CUDA(h, cudaEventRecord(h->ev_up[c], h->s_up));
        TK_CUDA(h, cudaStreamWaitEvent(s, h->ev_up[c], 0));
        tk::Env ev = h->e;
        ev.n = e_;
        const unsigned grid = (unsigned)((len + tk::CTA - 1) / tk::CTA);
        if (row == 54)
            tk::k_rollout_fused<tk::DEALS_PERM><<<grid, tk::CTA, tk::CTA * 54, s>>>(
                ev, 0u, h->st_perm, h->st_contract, h->st_declarer, king_host ? h->st_king : nullptr, h->e.scores, 0, b);
        else
            tk::k_rollout_fused<tk::DEALS_RECORD><<<grid, tk::CTA, tk::CTA * TAROK_RECORD_BYTES, s>>>(ev, 0u, h->st_perm, nullptr, nullptr, nullptr,
                                                                          h->e.scores, 0, b);
        TK_LAUNCH_OK(h);
        if (scores_host) {
            TK_CUDA(h, cudaEventRecord(h->ev_done[c], s));
            TK_CUDA(h, cudaStreamWaitEvent(h->s_down, h->ev_done[c], 0));
            TK_CUDA(h, cudaMemcpyAsync((uint64_t*)scores_host + b, h->e.scores + b, len * 8, cudaMemcpyDeviceToHost, h->s_down));
        }
    }
    TK_CUDA(h, cudaEventRecord(h->ev_join, h->s_down));
    TK_CUDA(h, cudaStreamWaitEvent(s, h->ev_join, 0));
    if (stats_host) TK_CUDA(h, cudaMemcpyAsync(stats_host, h->e.stats, TAROK_STATS_LEN * 8, cudaMemcpyDeviceToHost, s));
    return 0;
}

int tarok_rollout_host(tarok_t* h, const uint8_t* perm_host, const uint8_t* contract_host, const uint8_t* declarer_host,
                       const uint8_t* king_host, uint64_t first_global_game_id, int fused, int16_t* scores_host,
                       int64_t* stats_host, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!perm_host || !contract_host || !declarer_host) return fail(h, -1, "perm/contract/declarer host pointers are required");
    DeviceGuard dg(h->device);
    const u64 n = h->e.n;
    if (int rc = ensure_staging(h)) return rc;
    cudaStream_t s = S(stream);
    TK_CUDA(h, cudaMemsetAsync(h->e.stats, 0, TAROK_STATS_LEN * 8, s));
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    if (fused) return rollout_host_fused(h, perm_host, 54, contract_host, declarer_host, king_host, scores_host, stats_host, s);
    TK_CUDA(h, cudaMemcpyAsync(h->st_perm, perm_host, n * 54, cudaMemcpyHostToDevice, s));
    TK_CUDA(h, cudaMemcpyAsync(h->st_contract, contract_host, n, cudaMemcpyHostToDevice, s));
    TK_CUDA(h, cudaMemcpyAsync(h->st_declarer, declarer_host, n, cudaMemcpyHostToDevice, s));
    if (king_host) TK_CUDA(h, cudaMemcpyAsync(h->st_king, king_host, n, cudaMemcpyHostToDevice, s));
    clear_hist(h, stream);
    tk::k_set_deals<<<grid1(h->e.n_alloc), tk::CTA, 0, s>>>(h->e, h->st_perm);
    TK_LAUNCH_OK(h);
    tk::k_begin<tk::SRC_FORCED><<<grid1(h->e.n_alloc), tk::CTA, 0, s>>>(h->e, 0u, h->st_contract, h->st_declarer,
                                                                         king_host ? h->st_king : nullptr);
    TK_LAUNCH_OK(h);
    if (int rc = play_out_stepwise(h, 0u, stream)) return rc;
    if (scores_host) TK_CUDA(h, cudaMemcpyAsync(scores_host, h->e.scores, n * 8, cudaMemcpyDeviceToHost, s));
    if (stats_host) TK_CUDA(h, cudaMemcpyAsync(stats_host, h->e.stats, TAROK_STATS_LEN * 8, cudaMemcpyDeviceToHost, s));
    return 0;
}

int tarok_rollout_records(tarok_t* h, const void* records_host, uint64_t first_global_game_id, int16_t* scores_host,
                          int64_t* stats_host, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!records_host) return fail(h, -1, "records_host is null");
    DeviceGuard dg(h->device);
    if (int rc = ensure_staging(h)) return rc;
    cudaStream_t s = S(stream);
    TK_CUDA(h, cudaMemsetAsync(h->e.stats, 0, TAROK_STATS_LEN * 8, s));
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    return rollout_host_fused(h, (const uint8_t*)records_host, TAROK_RECORD_BYTES, nullptr, nullptr, nullptr, scores_host,
                              stats_host, s);
}

// Upload / play / download of the chunks of tarok_rollout_host_packed, each as soon as the pool has packed it.
static int packed_pipeline(tarok_t* h, const uint64_t* bounds, int nchunks, int16_t* scores_host, int64_t* stats_host, cudaStream_t s) {
    TK_CUDA(h, cudaEventRecord(h->ev_fork, s));
    TK_CUDA(h, cudaStreamWaitEvent(h->s_up, h->ev_fork, 0));
    TK_CUDA(h, cudaStreamWaitEvent(h->s_down, h->ev_fork, 0));
    for (int c = 0; c < nchunks; c++) {
        const u64 b = bounds[c], e_ = bounds[c + 1], len = e_ - b;
        tarok_pack_pool_wait_chunk(h->pool, c);
        TK_CUDA(h, cudaMemcpyAsync(h->st_perm + b * TAROK_RECORD_BYTES, h->pin_rec + b * TAROK_RECORD_BYTES,
                                   len * TAROK_RECORD_BYTES, cudaMemcpyHostToDevice, h->s_up));
        TK_CUDA(h, cudaEventRecord(h->ev_up[c], h->s_up));
        h->pack_used[c] = 1;
        TK_CUDA(h, cudaStreamWaitEvent(s, h->ev_up[c], 0));
        tk::Env ev = h->e;
        ev.n = e_;
        tk::k_rollout_fused<tk::DEALS_RECORD><<<(unsigned)((len + tk::CTA - 1) / tk::CTA), tk::CTA, tk::CTA * TAROK_RECORD_BYTES, s>>>(
            ev, 0u, h->st_perm, nullptr, nullptr, nullptr, h->e.scores, 0, b);
        TK_LAUNCH_OK(h);
        if (scores_host) {
            TK_CUDA(h, cudaEventRecord(h->ev_done[c], s));
            TK_CUDA(h, cudaStreamWaitEvent(h->s_down, h->ev_done[c], 0));
            TK_CUDA(h, cudaMemcpyAsync((uint64_t*)scores_host + b, h->e.scores + b, len * 8, cudaMemcpyDeviceToHost, h->s_down));
        }
    }
    TK_CUDA(h, cudaEventRecord(h->ev_join, h->s_down));
    TK_CUDA(h, cudaStreamWaitEvent(s, h->ev_join, 0));
    if (stats_host) TK_CUDA(h, cudaMemcpyAsync(stats_host, h->e.stats, TAROK_STATS_LEN * 8, cudaMemcpyDeviceToHost, s));
    return 0;
}

// Third form of the host-buffer entry: the caller hands over permutation ROWS (what Igra.shuffle produces), the library
// serialises each chunk into 20-byte deal records with `threads` host threads right before that chunk's upload, so PCIe
// carries 20 instead of 57 bytes per deal and the packing of chunk c+1 overlaps the upload / play / download of chunk c.
int tarok_rollout_host_packed(tarok_t* h, const uint8_t* perm_host, const uint8_t* contract_host, const uint8_t* declarer_host,
                              const uint8_t* king_host, uint64_t first_global_game_id, int threads, int16_t* scores_host,
                              int64_t* stats_host, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!perm_host || !contract_host || !declarer_host) return fail(h, -1, "perm/contract/declarer host pointers are required");
    if (threads < 1 || threads > 256) return fail(h, -1, "threads must be in 1..256");
    DeviceGuard dg(h->device);
    if (int rc = ensure_staging(h)) return rc;
    if (!h->pin_rec) TK_CUDA(h, cudaHostAlloc((void**)&h->pin_rec, h->e.n_alloc * TAROK_RECORD_BYTES, cudaHostAllocDefault));
    if (h->pool && tarok_pack_pool_threads(h->pool) != threads) { tarok_pack_pool_destroy(h->pool); h->pool = nullptr; }
    if (!h->pool) h->pool = tarok_pack_pool_create(threads);
    if (!h->pool) return fail(h, -4, "could not create the pack pool");
    cudaStream_t s = S(stream);
    TK_CUDA(h, cudaMemsetAsync(h->e.stats, 0, TAROK_STATS_LEN * 8, s));
    h->lock_plays = 0;
    set_first_gid(h, first_global_game_id);
    const u64 n = h->e.n;
    // the previous call's uploads must have left the pinned scratch before it is overwritten
    for (int c = 0; c < TK_MAX_CHUNKS; c++)
        if (h->pack_used[c]) { TK_CUDA(h, cudaEventSynchronize(h->ev_up[c])); h->pack_used[c] = 0; }
    // the pool packs the whole batch block by block in the background; chunk c is uploaded as soon as its blocks are done
    uint64_t bounds[TK_MAX_CHUNKS + 1];
    const int nchunks = tarok_chunk_bounds(n, h->chunks, tarok_pack_block_rows(), bounds);
    tarok_pack_pool_begin(h->pool, perm_host, contract_host, declarer_host, king_host, n, bounds, nchunks, h->pin_rec);
    const int rc = packed_pipeline(h, bounds, nchunks, scores_host, stats_host, s);
    if (rc)                                                 // the workers still read the caller's rows: let them finish
        for (int c = 0; c < nchunks; c++) tarok_pack_pool_wait_chunk(h->pool, c);
    return rc;
}

// ---- observations (SURVEY 8f rank 1) ------------------------------------------------------------------------

int tarok_obs_shape(tarok_t* h, uint8_t* type_dev, uint8_t* rows_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!type_dev || !rows_dev) return fail(h, -1, "type_dev/rows_dev is null");
    DeviceGuard dg(h->device);
    tk::k_obs_shape<<<grid1(h->e.n_alloc), tk::CTA, 0, S(stream)>>>(h->e, type_dev, rows_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

static int enqueue_obs_buckets(tarok_t* h, int players, int32_t* sel_dev, uint32_t* counts_dev, uint8_t* selkey_dev,
                               uint32_t* counts_host, cudaStream_t s) {
    const unsigned n_cta = grid1(h->e.n_alloc);
    tk::k_bucket_hist<<<n_cta, tk::CTA, 0, s>>>(h->e, (u32)players, h->cta_hist);
    TK_LAUNCH_OK(h);
    tk::k_bucket_scan<<<1, tk::BUCKETS * tk::SCAN_PARTS, 0, s>>>(h->cta_hist, n_cta, counts_dev);
    TK_LAUNCH_OK(h);
    tk::k_bucket_scatter<<<n_cta, tk::CTA, 0, s>>>(h->e, (u32)players, h->cta_hist, counts_dev, (int*)sel_dev, selkey_dev);
    TK_LAUNCH_OK(h);
    if (counts_host) TK_CUDA(h, cudaMemcpyAsync(counts_host, counts_dev, 3 * tk::BUCKETS * sizeof(u32), cudaMemcpyDeviceToHost, s));
    return 0;
}

int tarok_obs_buckets(tarok_t* h, int players, int32_t* sel_dev, uint32_t* counts_dev, uint8_t* selkey_dev, void* stream) {
    return tarok_obs_buckets_host(h, players, sel_dev, counts_dev, selkey_dev, nullptr, stream);
}

// The same + the 1.5 KB of counts copied to (pinned) host memory.  This runs once per self-play step right after a
// synchronisation, i.e. on an empty stream, where every launch costs its full latency: the three kernels and the copy are
// replayed as ONE graph launch (captured per argument set on first use; dropped when an option changes).
int tarok_obs_buckets_host(tarok_t* h, int players, int32_t* sel_dev, uint32_t* counts_dev, uint8_t* selkey_dev,
                           uint32_t* counts_host, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!sel_dev || !counts_dev) return fail(h, -1, "sel_dev/counts_dev is null");
    if (players != 1 && players != 4) return fail(h, -1, "players must be 1 or 4");
    DeviceGuard dg(h->device);
    cudaStream_t s = S(stream);
    const unsigned n_cta = grid1(h->e.n_alloc);
    if (!h->cta_hist) TK_CUDA(h, cudaMalloc((void**)&h->cta_hist, (size_t)n_cta * tk::BUCKETS * sizeof(u32)));
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (h->use_graph && cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone) {
        const void* key[5] = {sel_dev, counts_dev, selkey_dev, counts_host, (const void*)(intptr_t)players};
        if (!h->bucket_graph || memcmp(key, h->bucket_key, sizeof(key)) != 0) {
            if (h->bucket_graph) { cudaGraphExecDestroy(h->bucket_graph); h->bucket_graph = nullptr; }
            if (!h->s_cap) TK_CUDA(h, cudaStreamCreateWithFlags(&h->s_cap, cudaStreamNonBlocking));
            cudaGraph_t g = nullptr;
            const uint64_t launches0 = h->launches;
            cudaError_t ie = cudaErrorUnknown;
            if (cudaStreamBeginCapture(h->s_cap, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const int rc = enqueue_obs_buckets(h, players, sel_dev, counts_dev, selkey_dev, counts_host, h->s_cap);
                const cudaError_t ce = cudaStreamEndCapture(h->s_cap, &g);
                if (!rc && ce == cudaSuccess) ie = cudaGraphInstantiate(&h->bucket_graph, g, 0);
            }
            h->launches = launches0;
            if (g) cudaGraphDestroy(g);
            if (ie != cudaSuccess) h->bucket_graph = nullptr;
            else memcpy(h->bucket_key, key, sizeof(key));
        }
        if (h->bucket_graph) {
            TK_CUDA(h, cudaGraphLaunch(h->bucket_graph, s));
            h->launches += 3;
            return 0;
        }
        cudaGetLastError();                                // capture failed: plain launches below
    }
    cudaGetLastError();
    return enqueue_obs_buckets(h, players, sel_dev, counts_dev, selkey_dev, counts_host, s);
}

int tarok_obs_expand_buckets(tarok_t* h, const int32_t* sel_dev, const uint8_t* selkey_dev, const uint32_t* counts_dev,
                             uint64_t n_total, float* opp_dev, float* hand_dev, float* talon_dev, float* talon_klop_dev,
                             float* king_dev, float* decl_dev, float* discard_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!h->e.hist) return fail(h, -1, "observations need TAROK_FLAG_HISTORY at tarok_create");
    if (!sel_dev || !selkey_dev || !counts_dev) return fail(h, -1, "sel_dev/selkey_dev/counts_dev is null");
    if (!opp_dev || !hand_dev || !talon_dev || !talon_klop_dev || !king_dev || !decl_dev || !discard_dev)
        return fail(h, -1, "every arena pointer is required");
    if ((((uintptr_t)opp_dev) | ((uintptr_t)hand_dev)) & 15u) return fail(h, -1, "opp_dev/hand_dev must be 16-byte aligned");
    if ((((uintptr_t)talon_dev) | ((uintptr_t)talon_klop_dev) | ((uintptr_t)discard_dev)) & 7u)
        return fail(h, -1, "talon/discard arenas must be 8-byte aligned");
    if (n_total == 0) return 0;
    if (n_total > h->e.n) return fail(h, -1, "n_total exceeds the number of games");
    DeviceGuard dg(h->device);
    tk::ObsArena a = {opp_dev, hand_dev, talon_dev, talon_klop_dev, king_dev, decl_dev, discard_dev};
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_obs_expand_all<<<(unsigned)((n_total + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, (const int*)sel_dev, selkey_dev, counts_dev, n_total, a);
    TK_LAUNCH_OK(h);
    return 0;
}

// random.random() < random_card as "Philox word < threshold" over 64 bits: random_card = 1 gives 2^32, above every word.
static inline u64 explore_threshold(float random_card) { return (u64)((double)random_card * 4294967296.0); }

int tarok_select_action_buckets(tarok_t* h, const float* const* q_ptrs_dev, const int32_t* sel_dev, const uint8_t* selkey_dev,
                                const uint32_t* counts_dev, uint64_t n_total, const float* random_card4, uint8_t* card_dev,
                                float* qmax_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!q_ptrs_dev || !sel_dev || !selkey_dev || !counts_dev || !card_dev || !random_card4)
        return fail(h, -1, "q_ptrs_dev/sel_dev/selkey_dev/counts_dev/card_dev/random_card4 is null");
    tk::Thresholds4 t4;
    for (int p = 0; p < 4; p++) {
        if (!(random_card4[p] >= 0.f && random_card4[p] <= 1.f)) return fail(h, -1, "random_card must be in [0,1]");
        t4.t[p] = explore_threshold(random_card4[p]);
    }
    if (n_total == 0) return 0;
    if (n_total > h->e.n) return fail(h, -1, "n_total exceeds the number of games");
    DeviceGuard dg(h->device);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_select_action_all<<<(unsigned)((n_total + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, q_ptrs_dev, (const int*)sel_dev, selkey_dev, counts_dev, n_total, t4, card_dev, qmax_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_select_action_buckets_tab(tarok_t* h, const float* const* q_ptrs_host, const int32_t* sel_dev, const uint8_t* selkey_dev,
                                    const uint32_t* counts_dev, uint64_t n_total, const float* random_card4, uint8_t* card_dev,
                                    float* qmax_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!q_ptrs_host || !sel_dev || !selkey_dev || !counts_dev || !card_dev || !random_card4)
        return fail(h, -1, "q_ptrs_host/sel_dev/selkey_dev/counts_dev/card_dev/random_card4 is null");
    tk::Thresholds4 t4;
    for (int p = 0; p < 4; p++) {
        if (!(random_card4[p] >= 0.f && random_card4[p] <= 1.f)) return fail(h, -1, "random_card must be in [0,1]");
        t4.t[p] = explore_threshold(random_card4[p]);
    }
    if (n_total == 0) return 0;
    if (n_total > h->e.n) return fail(h, -1, "n_total exceeds the number of games");
    DeviceGuard dg(h->device);
    tk::QTable qt;
    memcpy(qt.p, q_ptrs_host, sizeof(qt.p));
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_select_action_all_tab<<<(unsigned)((n_total + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, qt, (const int*)sel_dev, selkey_dev, counts_dev, n_total, t4, card_dev, qmax_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_obs_expand(tarok_t* h, int net_type, uint32_t rows, const int32_t* sel_dev, uint64_t n_sel, float* opp_dev,
                     float* hand_dev, float* talon_dev, float* king_dev, float* decl_dev, float* discard_dev,
                     float* mozne_dev, uint8_t* ok_dev, void* stream) {
    return tarok_obs_expand_at(h, -1, net_type, rows, sel_dev, n_sel, opp_dev, hand_dev, talon_dev, king_dev, decl_dev,
                               discard_dev, mozne_dev, ok_dev, stream);
}

int tarok_obs_expand_at(tarok_t* h, int play, int net_type, uint32_t rows, const int32_t* sel_dev, uint64_t n_sel,
                        float* opp_dev, float* hand_dev, float* talon_dev, float* king_dev, float* decl_dev,
                        float* discard_dev, float* mozne_dev, uint8_t* ok_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (play >= 48) return fail(h, -1, "play must be < 48");
    if (!h->e.hist) return fail(h, -1, "observations need TAROK_FLAG_HISTORY at tarok_create");
    if (net_type < 0 || net_type > 3) return fail(h, -1, "net_type must be 0..3");
    if (rows == 0 || (rows & 7u) || rows > 56) return fail(h, -1, "rows must be a multiple of 8 in 8..56");
    if (!opp_dev || !hand_dev) return fail(h, -1, "opp_dev/hand_dev is null");
    if ((((uintptr_t)opp_dev) | ((uintptr_t)hand_dev)) & 15u) return fail(h, -1, "opp_dev/hand_dev must be 16-byte aligned");
    if (n_sel == 0) return 0;
    DeviceGuard dg(h->device);
    tk::ObsOut o = {opp_dev, hand_dev, talon_dev, king_dev, decl_dev, discard_dev, mozne_dev, ok_dev};
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_obs_expand<<<(unsigned)((n_sel + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, net_type, rows, (const int*)sel_dev, n_sel, o, play < 0 ? -1 : play);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_select_action(tarok_t* h, const float* q_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                        uint8_t* card_dev, float* qmax_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!q_dev || !card_dev) return fail(h, -1, "q_dev/card_dev is null");
    if (!(random_card >= 0.f && random_card <= 1.f)) return fail(h, -1, "random_card must be in [0,1]");
    if (n_sel == 0) return 0;
    DeviceGuard dg(h->device);
    const u64 threshold = explore_threshold(random_card);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_select_action<<<(unsigned)((n_sel + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, q_dev, (const int*)sel_dev, n_sel, threshold, card_dev, qmax_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_obs_hands(tarok_t* h, float* out_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!out_dev) return fail(h, -1, "out_dev is null");
    DeviceGuard dg(h->device);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_obs_hands<<<(unsigned)((h->e.n + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(h->e, out_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_obs_exchange(tarok_t* h, const int32_t* sel_dev, uint64_t n_sel, float* hand_dev, float* talon_dev, float* game_dev,
                       uint8_t* ok_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!hand_dev || !talon_dev || !game_dev) return fail(h, -1, "hand_dev/talon_dev/game_dev is null");
    if (n_sel == 0) return 0;
    DeviceGuard dg(h->device);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_obs_exchange<<<(unsigned)((n_sel + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, (const int*)sel_dev, n_sel, hand_dev, talon_dev, game_dev, ok_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_select_exchange(tarok_t* h, const float* p_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                          uint8_t* group_dev, uint64_t* discard_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!p_dev || !group_dev || !discard_dev) return fail(h, -1, "p_dev/group_dev/discard_dev is null");
    if (!(random_card >= 0.f && random_card <= 1.f)) return fail(h, -1, "random_card must be in [0,1]");
    if (n_sel == 0) return 0;
    DeviceGuard dg(h->device);
    const u64 threshold = explore_threshold(random_card);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_select_exchange<<<(unsigned)((n_sel + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, p_dev, (const int*)sel_dev, n_sel, threshold, group_dev, (u64*)discard_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

int tarok_targets(tarok_t* h, const int32_t* sel_dev, uint64_t n_sel, float final_reword_factor, float* dy_dev,
                  uint8_t* seat_dev, uint8_t* rows_dev, void* stream) {
    TK_CHECK_HANDLE(h);
    if (!h->e.hist) return fail(h, -1, "replay targets need TAROK_FLAG_HISTORY at tarok_create");
    if (!dy_dev || !seat_dev) return fail(h, -1, "dy_dev/seat_dev is null");
    if (((uintptr_t)dy_dev) & 15u) return fail(h, -1, "dy_dev must be 16-byte aligned");
    if (n_sel == 0) return 0;
    DeviceGuard dg(h->device);
    const u64 warps_per_cta = tk::CTA / 32;
    tk::k_targets<<<(unsigned)((n_sel + warps_per_cta - 1) / warps_per_cta), tk::CTA, 0, S(stream)>>>(
        h->e, (const int*)sel_dev, n_sel, final_reword_factor, dy_dev, seat_dev, rows_dev);
    TK_LAUNCH_OK(h);
    return 0;
}

// ---- zero-copy views ------------------------------------------------------------------------------------

struct ExportCtx {
    DLManagedTensor t;
    int64_t shape[2];
    tarok_env* owner;
};

static void export_deleter(DLManagedTensor* self) {
    if (!self) return;
    ExportCtx* c = static_cast<ExportCtx*>(self->manager_ctx);
    c->owner->exports.fetch_sub(1);
    delete c;
}

static int field_desc(tarok_env* h, int field, void** ptr, int* ndim, int64_t shape[2], DLDataType* dt) {
    const int64_t na = (int64_t)h->e.n_alloc;
    // bitboards are lent as int64 (same bits; torch has no general uint64 support), bit 63 is never set
    DLDataType u64t = {0, 64, 1}, i16t = {0, 16, 1}, u8t = {1, 8, 1}, i64t = {0, 64, 1}, f32t = {2, 32, 1};
    switch (field) {
        case TAROK_F_HANDS: *ptr = h->e.hands; *ndim = 2; shape[0] = 4; shape[1] = na; *dt = u64t; break;
        case TAROK_F_PILES: *ptr = h->e.piles; *ndim = 2; shape[0] = 4; shape[1] = na; *dt = u64t; break;
        case TAROK_F_TALON: *ptr = h->e.talon; *ndim = 1; shape[0] = na; *dt = u64t; break;
        case TAROK_F_TALON_ORDER: *ptr = h->e.torder; *ndim = 1; shape[0] = na; *dt = u64t; break;
        case TAROK_F_META: *ptr = h->e.meta; *ndim = 1; shape[0] = na; *dt = u64t; break;
        case TAROK_F_MASK: *ptr = h->e.mask; *ndim = 1; shape[0] = na; *dt = u64t; break;
        case TAROK_F_SCORES: *ptr = h->e.scores; *ndim = 2; shape[0] = na; shape[1] = 4; *dt = i16t; break;
        case TAROK_F_HIST: *ptr = h->e.hist; *ndim = 2; shape[0] = 48; shape[1] = na; *dt = u8t; break;
        case TAROK_F_STATS: *ptr = h->e.stats; *ndim = 1; shape[0] = TAROK_STATS_LEN; *dt = i64t; break;
        case TAROK_F_HANDS0: *ptr = h->e.hands0; *ndim = 2; shape[0] = 4; shape[1] = na; *dt = u64t; break;
        case TAROK_F_DISCARD: *ptr = h->e.discard; *ndim = 1; shape[0] = na; *dt = u64t; break;
        case TAROK_F_QMAX_HIST: *ptr = h->e.qmax_hist; *ndim = 2; shape[0] = 48; shape[1] = na; *dt = f32t; break;
        default: return fail(h, -1, "unknown field %d", field);
    }
    if (!*ptr) return fail(h, -1, "field %d needs TAROK_FLAG_HISTORY at tarok_create", field);
    return 0;
}

int tarok_export(tarok_t* h, int field, DLManagedTensor** out) {
    TK_CHECK_HANDLE(h);
    if (!out) return fail(h, -1, "out is null");
    ExportCtx* c = new (std::nothrow) ExportCtx();
    if (!c) return fail(h, -4, "out of host memory");
    void* ptr; int ndim; DLDataType dt;
    int rc = field_desc(h, field, &ptr, &ndim, c->shape, &dt);
    if (rc) { delete c; return rc; }
    c->owner = h;
    c->t.dl_tensor.data = ptr;
    c->t.dl_tensor.device.device_type = 2;   // kDLCUDA
    c->t.dl_tensor.device.device_id = h->device;
    c->t.dl_tensor.ndim = ndim;
    c->t.dl_tensor.dtype = dt;
    c->t.dl_tensor.shape = c->shape;
    c->t.dl_tensor.strides = nullptr;        // compact row-major
    c->t.dl_tensor.byte_offset = 0;
    c->t.manager_ctx = c;
    c->t.deleter = export_deleter;
    h->exports.fetch_add(1);
    *out = &c->t;
    return 0;
}

void* tarok_field_ptr(tarok_t* h, int field) {
    if (!h) return nullptr;
    void* ptr = nullptr; int ndim; int64_t shape[2]; DLDataType dt;
    if (field_desc(h, field, &ptr, &ndim, shape, &dt)) return nullptr;
    return ptr;
}

}  // extern "C"
