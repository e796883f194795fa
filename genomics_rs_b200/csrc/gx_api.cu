// gx_api.cu -- C ABI of libgxalign (include/gxalign.h): context, plans, kernel dispatch.
// No CPU compute path exists in this file: every entry point needs a live sm_100 device.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gxalign.h"
#include "gx_fill.cuh"
#include "gx_lcs.cuh"
#include "gx_reads.cuh"
#include "gx_walk.cuh"

namespace gx {

static_assert(sizeof(DevResult) == sizeof(gx_result), "DevResult must mirror gx_result");
static_assert(sizeof(PairDesc) == 104, "PairDesc layout");
static_assert(warp_smem_bytes(2) % 16 == 0 && warp_smem_bytes(4) % 16 == 0 && warp_smem_bytes(8) % 16 == 0 && warp_smem_bytes(16) % 16 == 0,
              "per-warp smem must keep 16 B alignment");

// ------------------------------------------------------------------------------------------------
struct Block {
    void *ptr;
    size_t size;
    bool free;
};

struct Ctx {
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<Block> pool;
    // streamed score batches (gx_score_batch on large read sets): NLANES lanes of copy + kernel
    static constexpr int NLANES = 3;
    cudaStream_t lane_stream[NLANES] = {nullptr, nullptr, nullptr};
    cudaEvent_t lane_done[NLANES] = {nullptr, nullptr, nullptr};
    int *lane_scores_host[NLANES] = {nullptr, nullptr, nullptr};   // pinned
    uint4 *lane_rec_host[NLANES] = {nullptr, nullptr, nullptr};    // pinned: per-pair records of the chunk in flight
    size_t lane_scores_cap = 0;
    uint32_t *lane_cells_host[NLANES] = {nullptr, nullptr, nullptr};   // pinned: start cells (gx_score_batch_cells, local)
    size_t lane_cells_cap = 0;
    int host_threads = 1;                             // worker threads for the host passes over a chunk
    uint8_t *ops_stage = nullptr;                     // pinned D2H staging of op lists (grown on demand)
    size_t ops_stage_cap = 0;
    std::string last_error;
    size_t pool_bytes = 0;
};

static Ctx *g_ctx = nullptr;
static std::recursive_mutex g_mu;   // recursive: the gx_band_* entry points call the gx_plan_* ones
static thread_local std::string g_err;

static int fail_cuda(cudaError_t e, const char *what) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    g_err = buf;
    if (g_ctx) g_ctx->last_error = buf;
    return GX_ERR_CUDA;
}
// The C ABI never throws: entry points that allocate host memory are function-try-blocks ending in GX_GUARD_END.
#define GX_GUARD_END                                                  \
    catch (const std::bad_alloc &) {                                  \
        g_err = "host allocation failed";                             \
        return GX_ERR_NOMEM;                                          \
    }                                                                 \
    catch (...) {                                                     \
        g_err = "unexpected C++ exception inside libgxalign";         \
        return GX_ERR_INTERNAL;                                       \
    }
#define CK(call)                                        \
    do {                                                \
        cudaError_t e__ = (call);                       \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call); \
    } while (0)

// caching device allocator: plans are created per call by gx_align_pair/gx_align_batch
static int pool_alloc(Ctx *c, size_t bytes, void **out) {
    if (bytes == 0) bytes = 16;
    bytes = (bytes + 511) & ~size_t(511);
    int best = -1;
    for (size_t k = 0; k < c->pool.size(); ++k) {
        Block &b = c->pool[k];
        if (b.free && b.size >= bytes && b.size <= 2 * bytes + (1u << 20))
            if (best < 0 || b.size < c->pool[best].size) best = (int)k;
    }
    if (best >= 0) {
        c->pool[best].free = false;
        *out = c->pool[best].ptr;
        return GX_OK;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        // release cached blocks and retry once
        for (auto it = c->pool.begin(); it != c->pool.end();) {
            if (it->free) {
                cudaFree(it->ptr);
                c->pool_bytes -= it->size;
                it = c->pool.erase(it);
            } else ++it;
        }
        cudaGetLastError();
        e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            g_err = "device allocation of " + std::to_string(bytes) + " bytes failed";
            return GX_ERR_NOMEM;
        }
    }
    c->pool.push_back({p, bytes, false});
    c->pool_bytes += bytes;
    *out = p;
    return GX_OK;
}
static void pool_free(Ctx *c, void *p) {
    if (!p) return;
    for (auto &b : c->pool)
        if (b.ptr == p) {
            b.free = true;
            return;
        }
}

// ------------------------------------------------------------------------------------------------
// Debug / experiment switches (DESIGN.md 7a).  The environment is read ONCE per plan (gx_plan_create) or per streamed
// batch call, never on the execute path; -1 = not set.
struct Tunables {
    int r = -1, batch = -1, code_band = -1, band_resident = 1;
    int k = -1, chain1 = -1, tickets = -1, resident = -1, wpc = -1, grid_cap = -1, pad_keys = 0, poll_nap = 0, start_lead = 0,
        fill_stats = 0, walk_stats = 0, walk_rows = 0, no_stream = 0, reads32 = 0, test_abort = 0;
};
static int env_int(const char *name, int dflt) {
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}
static Tunables read_tunables() {
    Tunables t;
    t.k = env_int("GX_K", -1);
    t.r = env_int("GX_R", -1);
    t.batch = env_int("GX_BATCH", -1);
    t.band_resident = env_int("GX_BAND_RESIDENT", 1);   // 0: resident-strips plans keep codes in every tile
    t.code_band = env_int("GX_CODE_BAND", -1);   // 0: codes in every tile; > 0: half-width of the code band in columns
    t.chain1 = env_int("GX_CHAIN1", -1);
    t.tickets = getenv("GX_TICKETS") ? 1 : -1;
    t.resident = env_int("GX_RESIDENT", -1);
    t.wpc = env_int("GX_WPC", -1);
    t.grid_cap = env_int("GX_GRID_CAP", -1);
    t.pad_keys = getenv("GX_PAD_KEYS") ? 1 : 0;
    t.poll_nap = env_int("GX_POLL_NAP", 0);
    t.start_lead = env_int("GX_START_LEAD", 0);
    t.fill_stats = env_int("GX_FILL_STATS", 0);
    t.walk_stats = getenv("GX_WALK_STATS") ? 1 : 0;
    t.walk_rows = env_int("GX_WALK_ROWS", 0);          // 64..512, multiple of 64: rows of a code window of the walk
    t.no_stream = getenv("GX_NO_STREAM") ? 1 : 0;
    t.reads32 = getenv("GX_READS32") ? 1 : 0;
    t.test_abort = getenv("GX_TEST_ABORT") ? 1 : 0;
    return t;
}

enum PlanKind { KIND_WAVEFRONT = 0, KIND_READS = 1 };
typedef void (*FillKernel)(const FillParams);

}  // namespace gx

struct gx_band;
struct gx_plan {
    gx::Ctx *ctx = nullptr;
    int kind = gx::KIND_WAVEFRONT;
    uint64_t n_pairs = 0;
    gx_scores sc{};
    gx::Tunables tun;                  // debug switches as they were when the plan was created
    int is_local = 0, flags = 0;
    int K = 8, R = 1;                  // register tile of the fill: K columns x R rows per lane per step
    uint32_t cpb = 1;                  // code chunks per hand-off batch (batch = cpb * 64/(R*K) steps)
    bool chain1 = false;               // latency-optimised recurrence (gx_fill.cuh, CHAIN1)
    int track = 0;
    bool traceback = false;
    std::vector<gx::PairDesc> pairs;   // host copy (offsets filled at upload)
    std::vector<uint64_t> len1, len2;
    uint64_t n_tiles = 0;
    uint64_t n_strips = 0;             // strips of all pairs at the chosen K
    uint64_t cells = 0;
    uint64_t code_bytes = 0, ops_bytes = 0, colbuf_entries = 0, top_entries = 0, progress_entries = 0, best_entries = 0;
    uint64_t blob_cap = 0;
    uint64_t max_len = 0;
    // device
    uint8_t *d_blob = nullptr;
    uint8_t *d_blob_sym = nullptr;     // blob re-encoded to symbols 0..3 when the batch uses <= 4 distinct bytes
    uint8_t *d_lut = nullptr;
    unsigned long long *d_stats = nullptr;   // GX_FILL_STATS=1: wait/tile cycle counters of the last execute
    unsigned long long h_stats[8] = {0};
    unsigned long long *d_timeline = nullptr;   // GX_FILL_STATS=2: per-tile timestamps (debug)
    bool prof = false;
    gx::PairDesc *d_pairs = nullptr;
    gx::TileDesc *d_tiles = nullptr;
    gx::TileDesc *d_strips = nullptr;   // resident-strips mode (every strip has its own warp): tiles as [strip][panel]
    bool resident = false;
    uint32_t pmax = 0;
    uint32_t *d_ctrl = nullptr;  // [0] ticket, [16..] progress
    unsigned long long *d_colbuf = nullptr;
    int2 *d_top = nullptr;
    uint8_t *d_codes = nullptr;
    int4 *d_best = nullptr;
    // GX_FLAG_LCS_AT_MAX: first-maximum pass + bit-vector LCS (gx_lcs.cuh)
    bool lcs = false;
    int4 *d_first = nullptr;
    uint32_t *d_masks = nullptr, *d_carry = nullptr;
    uint32_t carry_words = 0;
    float lcs_ms = 0;
    gx::DevResult *d_results = nullptr;
    uint8_t *d_ops = nullptr;
    // reads kind
    uint64_t *d_off1 = nullptr, *d_off2 = nullptr;
    uint32_t *d_len1 = nullptr, *d_len2 = nullptr;
    int *d_scores = nullptr;
    uint32_t *d_cells = nullptr;       // local start-cell read plans: i << 16 | j per pair
    uint32_t parity = 0;
    bool uploaded = false, executed = false, colbuf_dirty = true;
    float fill_ms = 0, walk_ms = 0;
    int launches = 0;
    int retries = 0;                   // resident-strips executes that were repeated in ticket mode
    int reads_bits = 0;                // read plans: lane width of the kernel the last execute ran (16: s16x2, 32)
    bool code_band = false;            // global traceback plan in ticket mode: only tiles near the diagonal write direction codes
    uint8_t *d_tile_codes = nullptr;   // one flag per tile (indexed like tile_best)
    int band_fallbacks = 0;            // executes repeated with codes everywhere because a path left the band
    uint32_t left_band = 0;            // walks of the last execute that needed a tile outside the band
    double code_cell_frac = 1.0;       // share of the cells that lie in code-writing tiles
    uint64_t h2d_bytes = 0, d2h_bytes = 0, dev_bytes = 0;
    // band plans (gx_band_*): every "pair" is a column band of one wide table
    gx_band *band = nullptr;
};

// One process's share of a column-banded table: bands [first,last) of n_bands, linked left to right.
struct gx_band {
    gx_plan *plan = nullptr;
    uint64_t m = 0, n_total = 0;
    gx_scores sc{};
    int n_bands = 0, first = 0, last = 0;
    std::vector<uint64_t> col0, width;        // of the local bands
    uint8_t *link = nullptr;                  // own link block (plain cudaMalloc, exportable): [ack 256 B][inbox 8 B x m]
    std::vector<unsigned long long *> internal;   // inbox of local band q+1 == outbox of local band q
    void *left_base = nullptr, *right_base = nullptr;   // opened IPC mappings of the neighbours' link blocks
    uint32_t epoch = 0;                       // executes finished
    bool connected = false, poisoned = false, trivial = false;
    float fill_ms = 0;
};

namespace gx {

// (K, R) register tiles the library is built with: K columns x R rows per lane per step (gx_fill.cuh).  R > 1 (several
// rows per step) is supported by the kernels and was measured on every workload (profiles/r2a_sweep_kr_rowblock.jsonl):
// the fill is bound by instructions issued per cell, which R does not lower, and the pipeline ramp of a pair grows with R
// (31 steps of lane skew x R rows per strip), so only R = 1 is instantiated.  Add a pair here and in build.py to try one.
#define GX_COMBOS(X) X(4, 1) X(8, 1) X(16, 1)

// the fill kernels are instantiated in gx_fill_inst.cu, one translation unit per (K, R, CHAIN1) so that they build in parallel
#define GX_DECL(K, R)                                                  \
    FillKernel pick_fill_##K##_##R##_0(bool prof, bool L, bool C, int track); \
    FillKernel pick_fill_##K##_##R##_1(bool prof, bool L, bool C, int track);
GX_COMBOS(GX_DECL)
#undef GX_DECL

static bool combo_ok(int K, int R) {
#define GX_CHK(k, r) if (K == k && R == r) return true;
    GX_COMBOS(GX_CHK)
#undef GX_CHK
    return false;
}

static FillKernel pick_fill(int K, int R, bool prof, bool chain1, bool L, bool C, int track) {
#define GX_PICK(k, r) if (K == k && R == r) return chain1 ? pick_fill_##k##_##r##_1(prof, L, C, track) : pick_fill_##k##_##r##_0(prof, L, C, track);
    GX_COMBOS(GX_PICK)
#undef GX_PICK
    return nullptr;
}

static int launch_fill(gx_plan *pl, const FillParams &fp, int grid_cap, int track_override = -1) {
    Ctx *c = pl->ctx;
    const int K = pl->K;
    const bool L = pl->is_local != 0, C = pl->traceback;
    const bool banded = pl->code_band && track_override < 0 && C && !L;   // two-variant kernel + per-tile flags
    FillKernel kern = (track_override >= 0) ? pick_fill(K, pl->R, pl->prof, pl->chain1, L, false, track_override)
                      : banded              ? pick_fill(K, pl->R, pl->prof, pl->chain1, false, true, 4)
                                            : pick_fill(K, pl->R, pl->prof, pl->chain1, L, C, pl->track);
    if (!kern) {
        g_err = "no fill kernel for this (K, R)";
        return GX_ERR_INTERNAL;
    }
    // CTA shape: single-warp CTAs while the plan cannot fill half of the warp slots (see gx_common.cuh)
    int wpc = (pl->n_strips * 2 >= (uint64_t)c->sm_count * warps_per_sm(K)) ? WARPS_PER_CTA : 1;
    if (pl->tun.wpc >= 0) wpc = pl->tun.wpc == 1 ? 1 : WARPS_PER_CTA;
    if (pl->resident) wpc = 1;   // one strip per single-warp CTA, dealt round-robin over the SMs
    const size_t smem = (size_t)wpc * warp_smem_bytes(K);
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(WARPS_PER_CTA * warp_smem_bytes(K))));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, wpc * 32, smem));
    if (occ < 1) occ = 1;
    const bool codes_kernel = C && track_override < 0;
    occ = std::min(occ, (codes_kernel ? warps_per_sm(K) : GX_SCORE_CTAS * WARPS_PER_CTA) / wpc);
    uint64_t cap = (uint64_t)c->sm_count * occ;
    FillParams fq = fp;
    fq.tile_codes = banded ? pl->d_tile_codes : nullptr;
    if (pl->resident && pl->n_strips > cap) {
        g_err = "resident-strips plan does not fit the device (fewer than 16 single-warp CTAs per SM)";
        return GX_ERR_INTERNAL;
    }
    if (pl->resident) {   // every strip resident: static ownership, tiles as [strip][panel]
        fq.pmax = pl->pmax;
        fq.tiles = pl->d_strips;
        fq.n_tiles = (uint32_t)(pl->n_strips * pl->pmax);
    }
    uint64_t want = fq.pmax ? pl->n_strips : (pl->n_tiles + wpc - 1) / wpc;
    if (pl->tun.grid_cap >= 0) grid_cap = pl->tun.grid_cap;
    if (grid_cap > 0 && (uint64_t)grid_cap < cap) cap = grid_cap;
    int grid = (int)std::min<uint64_t>(want, cap);
    if (grid < 1) grid = 1;
    if (pl->resident) {
        // Resident strips wait for one another, so every CTA of the grid must be on the device at the same time:
        // a cooperative launch is the only way CUDA guarantees that (the grid fits: checked against the occupancy above).
        void *kargs[] = {(void *)&fq};
        CK(cudaLaunchCooperativeKernel((const void *)kern, dim3((unsigned)grid), dim3((unsigned)(wpc * 32)), kargs, smem, c->stream));
    } else {
        kern<<<grid, wpc * 32, smem, c->stream>>>(fq);
    }
    CK(cudaGetLastError());
    return GX_OK;
}

typedef void (*WalkKernel)(const WalkParams);
static int launch_walk(gx_plan *pl, WalkParams wp) {
    WalkKernel kern = nullptr;
#define GX_WALK(k, r) \
    if (pl->K == k && pl->R == r) kern = gx_walk_kernel<k, r>;
    GX_COMBOS(GX_WALK)
#undef GX_WALK
    if (!kern) {
        g_err = "no walk kernel for this (K, R)";
        return GX_ERR_INTERNAL;
    }
    // rows of a code window: 512 lets a diagonal path cross a whole strip (32*K <= 256 columns for K <= 8) inside one window;
    // fewer rows (three window buffers per CTA) keep every pair's walk CTA resident when there are many pairs -- the walk is a
    // latency chain per pair, so residency is its throughput; short sequences need no more rows than they have
    const uint32_t row_cap = (uint32_t)std::max<uint64_t>(64, std::min<uint64_t>(512, (pl->max_len + 63) / 64 * 64));
    uint32_t rows = 0;
    for (uint32_t cand : {512u, 384u, 256u, 192u, 128u, 64u}) {
        if (cand > 256u && pl->K > 8) continue;
        const uint32_t r_ = std::min(cand, row_cap);
        const uint32_t per_sm = std::min<uint32_t>(2048u / WALK_THREADS, (227u * 1024u) / (walk_smem_bytes(pl->K, pl->R, r_) + 1024u));
        if (pl->n_pairs <= (uint64_t)per_sm * (uint64_t)pl->ctx->sm_count) {
            rows = r_;
            break;
        }
    }
    if (!rows) rows = pl->max_len <= 256 ? 64u : 128u;     // more pairs than fit at once: many CTAs per SM
    if (pl->tun.walk_rows >= 64 && pl->tun.walk_rows <= 512 && pl->tun.walk_rows % 64 == 0) rows = (uint32_t)pl->tun.walk_rows;
    wp.win_rows = rows;
    const uint32_t smem = wp.traceback ? walk_smem_bytes(pl->K, pl->R, rows) : 0u;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_smem_bytes(pl->K, pl->R, 512u)));
    // one CTA per pair: path warp, loader warp and two emit warps with traceback; a single warp (start cell and score only) without
    kern<<<(unsigned)pl->n_pairs, wp.traceback ? WALK_THREADS : 32, smem, pl->ctx->stream>>>(wp);
    CK(cudaGetLastError());
    return GX_OK;
}

static int check_scores_impl(gx_scores sc, uint64_t m, uint64_t n, bool local) {
    if (!(sc.h <= 0 && sc.g < 0 && (long long)sc.h + sc.g < 0)) return GX_ERR_SCORES;
    long long mx = std::max({std::llabs((long long)sc.s_match), std::llabs((long long)sc.s_mismatch), std::llabs((long long)sc.g)});
    long long lim = 1ll << 29;
    if (m > (1ull << 28) || n > (1ull << 28)) return GX_ERR_RANGE;
    if ((long long)(m + n + 2) * mx + std::llabs((long long)sc.h) >= lim) return GX_ERR_RANGE;
    if (local) {
        long long vmax = (long long)std::min(m, n) * std::max<long long>(sc.s_match, 0);
        // start-cell keys, K <= 16: the classic form keys (V << log2 K) | k, which this bound keeps in int32; the CHAIN1
        // form keys (E << log2 K) | k with E = V + (h+g), which also needs -(h+g) < 2^(31 - log2 K): plan_create_locked
        // keeps local start-cell plans that break it on the classic form instead of refusing them
        if (vmax >= (1ll << 26)) return GX_ERR_RANGE;
    }
    return GX_OK;
}

static void plan_release(gx_plan *pl) {
    Ctx *c = pl->ctx;
    void *ptrs[] = {pl->d_tile_codes, pl->d_blob, pl->d_blob_sym, pl->d_lut, pl->d_stats, pl->d_timeline, pl->d_pairs, pl->d_tiles, pl->d_strips, pl->d_ctrl, pl->d_colbuf, pl->d_top, pl->d_codes, pl->d_best, pl->d_first, pl->d_masks, pl->d_carry,
                    pl->d_results, pl->d_ops, pl->d_off1, pl->d_off2, pl->d_len1, pl->d_len2, pl->d_scores, pl->d_cells};
    for (void *p : ptrs) pool_free(c, p);
}

}  // namespace gx

using namespace gx;

// ================================================================================================
extern "C" {

const char *gx_version(void) {
#ifdef GX_CHECKED
    return "gxalign 0.2 (sm_100a, checked build: device-side bounds assertions)";
#else
    return "gxalign 0.2 (sm_100a)";
#endif
}

const char *gx_strerror(int s) {
    switch (s) {
        case GX_OK: return "ok";
        case GX_ERR_ARG: return "invalid argument";
        case GX_ERR_SCORES: return "scores violate h <= 0, g < 0, h+g < 0";
        case GX_ERR_RANGE: return "sequence lengths x scores exceed the int32 cell range";
        case GX_ERR_OPS_CAP: return "ops buffer too small";
        case GX_ERR_NO_DEVICE: return "no sm_100 CUDA device (there is no CPU path)";
        case GX_ERR_CUDA: return "CUDA error";
        case GX_ERR_NOMEM: return "out of memory";
        case GX_ERR_NOT_INIT: return "gx_init not called";
        case GX_ERR_UNSUPPORTED: return "unsupported flag or mode";
        case GX_ERR_INTERNAL: return "internal error";
        default: return "unknown status";
    }
}

const char *gx_last_error(void) { return g_err.c_str(); }

int gx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

int gx_init(int device) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        g_err = "no CUDA device visible";
        return GX_ERR_NO_DEVICE;
    }
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) return GX_ERR_NO_DEVICE;
    }
    if (device >= n) return GX_ERR_ARG;
    int major = 0;
    CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) {
        g_err = "device is not compute capability 10.x; libgxalign carries sm_100a code only";
        return GX_ERR_NO_DEVICE;
    }
    if (g_ctx && g_ctx->device == device) return GX_OK;
    if (g_ctx) return GX_ERR_ARG;  // one context (one GPU) per process
    CK(cudaSetDevice(device));
    Ctx *c = new (std::nothrow) Ctx();
    if (!c) return GX_ERR_NOMEM;
    c->device = device;
    CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (auto &e : c->ev) CK(cudaEventCreate(&e));
    for (int k = 0; k < Ctx::NLANES; ++k) {
        CK(cudaStreamCreateWithFlags(&c->lane_stream[k], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&c->lane_done[k], cudaEventDisableTiming));
    }
    {
        // host passes of the streamed read path: a few threads per process (one process per GPU shares the host)
        int ndev = 1;
        cudaGetDeviceCount(&ndev);
        const unsigned hw = std::thread::hardware_concurrency();
        c->host_threads = (int)std::max(1u, std::min(8u, hw / (unsigned)std::max(1, ndev)));
        if (const char *e = getenv("GX_HOST_THREADS")) c->host_threads = std::max(1, atoi(e));
    }
    g_ctx = c;
    return GX_OK;
}
GX_GUARD_END

static void band_cache_drop();   // gx_nw_score_banded keeps its last band object
static void plan_cache_drop();   // gx_align_batch / gx_score_batch keep their last plan

void gx_shutdown(void) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!g_ctx) return;
    cudaSetDevice(g_ctx->device);
    cudaStreamSynchronize(g_ctx->stream);
    band_cache_drop();
    plan_cache_drop();
    for (auto &b : g_ctx->pool) cudaFree(b.ptr);
    for (auto &e : g_ctx->ev) cudaEventDestroy(e);
    for (int k = 0; k < Ctx::NLANES; ++k) {
        if (g_ctx->lane_stream[k]) cudaStreamDestroy(g_ctx->lane_stream[k]);
        if (g_ctx->lane_done[k]) cudaEventDestroy(g_ctx->lane_done[k]);
        if (g_ctx->lane_scores_host[k]) cudaFreeHost(g_ctx->lane_scores_host[k]);
        if (g_ctx->lane_rec_host[k]) cudaFreeHost(g_ctx->lane_rec_host[k]);
        if (g_ctx->lane_cells_host[k]) cudaFreeHost(g_ctx->lane_cells_host[k]);
    }
    if (g_ctx->ops_stage) cudaFreeHost(g_ctx->ops_stage);
    cudaStreamDestroy(g_ctx->stream);
    delete g_ctx;
    g_ctx = nullptr;
}

int gx_check_scores(gx_scores sc, uint64_t m, uint64_t n) { return check_scores_impl(sc, m, n, true); }

int gx_replay_ops(const uint8_t *ops, uint64_t n_ops, uint64_t start_i, uint64_t start_j, uint32_t *ops_i, uint32_t *ops_j) {
    if ((!ops && n_ops) || !ops_i || !ops_j) return GX_ERR_ARG;
    uint64_t i = start_i, j = start_j;
    for (uint64_t k = 0; k < n_ops; ++k) {
        ops_i[k] = (uint32_t)i;
        ops_j[k] = (uint32_t)j;
        switch (ops[k]) {
            case GX_MATCH:
            case GX_MISMATCH:
                i = i ? i - 1 : 0;
                j = j ? j - 1 : 0;
                break;
            case GX_INSERT:
            case GX_OPEN_INSERT: j = j ? j - 1 : 0; break;
            case GX_DELETE:
            case GX_OPEN_DELETE: i = i ? i - 1 : 0; break;
            default: return GX_ERR_ARG;
        }
    }
    return GX_OK;
}

// ------------------------------------------------------------------------------------------------
}  // extern "C"


// Ticket order of the fill kernel's tiles: key(p,s) = p*4096 + (strip_base+s)*64, ties by pair, then panel -- every
// dependency of (p,s), i.e. (p,s-1) and (p-1,s) (and, for column bands, the last strip of the band to the left), gets a
// smaller ticket, so a waiting warp only ever waits for tiles that were handed out before its own.  Generated in order
// without a sort: v = key / 64 = 64 p + strip_base + s.   S, P: strips / panels per pair; sbase: first global strip.
static void build_ticket_order(const std::vector<uint32_t> &S, const std::vector<uint32_t> &P, const std::vector<uint64_t> &sbase,
                               std::vector<TileDesc> &tiles) {
    const size_t n_pairs = S.size();
    constexpr uint64_t TS = PANEL_H / 64;   // strips a panel step is worth in the key (64 for 4096-row panels)
    uint64_t vmax = 0;
    std::vector<uint32_t> live;   // pairs that still have tiles at or after v: the sweep costs O(tiles + live pairs x v)
    for (size_t q = 0; q < n_pairs; ++q)
        if (S[q] && P[q]) {
            vmax = std::max<uint64_t>(vmax, (uint64_t)(P[q] - 1) * TS + sbase[q] + S[q] - 1);
            live.push_back((uint32_t)q);
        }
    for (uint64_t v = 0; v <= vmax && !live.empty(); ++v) {
        size_t keep = 0;
        for (size_t li = 0; li < live.size(); ++li) {
            const uint32_t q = live[li];
            const uint64_t last = (uint64_t)(P[q] - 1) * TS + sbase[q] + S[q] - 1;
            if (v <= last) live[keep++] = q;
            if (v < sbase[q]) continue;
            const uint64_t sv = v - sbase[q];
            const uint64_t p_hi = std::min<uint64_t>(P[q] - 1, sv / TS);
            const uint64_t p_lo = (sv >= S[q]) ? (sv - S[q] + 1 + TS - 1) / TS : 0;
            for (uint64_t p2 = p_lo; p2 <= p_hi; ++p2) tiles.push_back({q, (uint32_t)p2, (uint32_t)(sv - TS * p2), 0});
        }
        live.resize(keep);
    }
}

// band_col0 != null: the "pairs" are consecutive column bands of one table (band q starts at column band_col0[q]);
// their strips are ticketed as one left-to-right sequence and the short-read kernel is never chosen.
static int plan_create_locked(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local, int flags,
                              const uint64_t *band_col0, gx_plan **out) {
    if (!out) return GX_ERR_ARG;
    *out = nullptr;
    if (!g_ctx) return GX_ERR_NOT_INIT;
    if ((!len1 || !len2) && n_pairs) return GX_ERR_ARG;
    if (n_pairs >= (1ull << 31)) return GX_ERR_RANGE;
    Ctx *c = g_ctx;
    CK(cudaSetDevice(c->device));
    uint64_t max_len = 0;
    for (uint64_t q = 0; q < n_pairs; ++q) {
        int rc = check_scores_impl(sc, len1[q], len2[q], is_local != 0);
        if (rc) return rc;
        max_len = std::max({max_len, len1[q], len2[q]});
    }
    if (n_pairs == 0) {
        int rc = check_scores_impl(sc, 0, 0, is_local != 0);
        if (rc) return rc;
    }
    gx_plan *pl = new (std::nothrow) gx_plan();
    if (!pl) return GX_ERR_NOMEM;
    pl->ctx = c;
    pl->n_pairs = n_pairs;
    pl->sc = sc;
    pl->tun = read_tunables();
    pl->is_local = is_local ? 1 : 0;
    pl->flags = flags;
    pl->traceback = (flags & GX_FLAG_TRACEBACK) != 0;
    pl->track = is_local ? ((pl->traceback || (flags & GX_FLAG_START_CELL)) ? 2 : 1) : 0;
    pl->len1.assign(len1, len1 + n_pairs);
    pl->len2.assign(len2, len2 + n_pairs);
    pl->max_len = max_len;
    for (uint64_t q = 0; q < n_pairs; ++q) pl->cells += (len1[q] + 1) * (len2[q] + 1);

    // short-read batches without traceback go to the inter-task kernel (K4), local start-cell plans included
    pl->lcs = (flags & GX_FLAG_LCS_AT_MAX) != 0 && !band_col0;
    if (pl->lcs) {
        // the first-maximum keys are (V << log2 K) | k in int32 for every cell, global mode included
        long long mx = std::max({std::llabs((long long)sc.s_match), std::llabs((long long)sc.s_mismatch), std::llabs((long long)sc.g)});
        if (n_pairs > 65536 || (long long)(2 * max_len + 2) * mx + std::llabs((long long)sc.h) >= (1ll << 26)) {
            delete pl;
            return n_pairs > 65536 ? GX_ERR_UNSUPPORTED : GX_ERR_RANGE;
        }
    }
    const bool reads = !pl->lcs && !band_col0 && !pl->traceback && n_pairs >= 1024 && max_len <= (uint64_t)READS_MAX_LEN &&
                       (!is_local || sc.s_mismatch < 0);
    pl->kind = reads ? KIND_READS : KIND_WAVEFRONT;
    int rc = GX_OK;
    auto A = [&](size_t bytes, void **p) {
        if (rc == GX_OK) {
            rc = pool_alloc(c, bytes, p);
            if (rc == GX_OK) pl->dev_bytes += (bytes + 511) & ~size_t(511);
        }
    };
    if (pl->kind == KIND_READS) {
        A(n_pairs * 8, (void **)&pl->d_off1);
        A(n_pairs * 8, (void **)&pl->d_off2);
        A(n_pairs * 4, (void **)&pl->d_len1);
        A(n_pairs * 4, (void **)&pl->d_len2);
        A(n_pairs * 4, (void **)&pl->d_scores);
        if (pl->track == 2) A(n_pairs * 4, (void **)&pl->d_cells);
        if (rc == GX_OK) {
            std::vector<uint32_t> l1(n_pairs), l2(n_pairs);
            for (uint64_t q = 0; q < n_pairs; ++q) {
                l1[q] = (uint32_t)len1[q];
                l2[q] = (uint32_t)len2[q];
            }
            cudaError_t e = cudaMemcpyAsync(pl->d_len1, l1.data(), n_pairs * 4, cudaMemcpyHostToDevice, c->stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_len2, l2.data(), n_pairs * 4, cudaMemcpyHostToDevice, c->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
            if (e != cudaSuccess) rc = fail_cuda(e, "upload lengths");
        }
        if (rc != GX_OK) {
            plan_release(pl);
            delete pl;
            return rc;
        }
        *out = pl;
        return GX_OK;
    }

    // ---- wavefront geometry: K columns per lane.  Larger K amortises the per-step hand-off over more cells,
    // smaller K gives more strips (warps) for batches that cannot fill the GPU otherwise.
    {
        const uint64_t resident = (uint64_t)c->sm_count * warps_per_sm(16);   // thresholds below were tuned against 16 warps per SM
        uint64_t strips16 = 0, strips8 = 0;
        for (uint64_t q = 0; q < n_pairs; ++q)
            if (len1[q] && len2[q]) {
                strips16 += (len2[q] + 511) / 512;
                strips8 += (len2[q] + 255) / 256;
            }
        // measured on corona shards (tools/timeline_wl.py): 45 pairs K=16 ~ K=8; 23 pairs K=8 ~ K=4 << K=16;
        // 11 pairs K=4 6.1 ms vs K=8 8.5 ms; 6 pairs K=4 5.5 vs K=8 7.0 -- shorter strips win until the warp slots are full
        // round 2 (32-step batches in ticket mode, profiles/r2e_sweep_batch_b32.jsonl): K=8 beats K=16 wherever both fill the
        // warp slots (45 pairs 16.7 vs 17.3 ms, 1 Mbp x 1 Mbp 282 vs 340 ms), so K=16 is no longer picked by itself
        (void)strips16;
        pl->K = (strips8 * 10 >= resident * 12 || max_len < 2048) ? 8 : 4;
        if (combo_ok(pl->tun.k, 1)) pl->K = pl->tun.k;
        pl->R = 1;
        if (pl->tun.r > 0 && combo_ok(pl->K, pl->tun.r)) pl->R = pl->tun.r;
        // latency-optimised recurrence (one more ALU op per cell, 1-op row chain) when warps are too few to hide the
        // classic 3-op chain: measured win below ~1/4 of the resident warps, loss at full occupancy
        {
            uint64_t strips = 0;
            for (uint64_t q = 0; q < n_pairs; ++q)
                if (len1[q] && len2[q]) strips += (len2[q] + 32 * pl->K - 1) / (32 * pl->K);
            pl->chain1 = strips * 4 < resident;
            pl->n_strips = strips;
        }
        if (pl->tun.chain1 >= 0) pl->chain1 = pl->tun.chain1 != 0;
        // CHAIN1 takes the start-cell keys of a local plan in E-space, ((V + (h+g)) << log2 K) | k.  The score contract
        // bounds V but not h+g against 2^(31 - log2 K): from there the key of a small V wraps.  Such plans take the
        // classic form, whose keys (V << log2 K) | k fit every valid scoring.  Applied after the GX_K / GX_CHAIN1
        // overrides, so that no switch selects a form that cannot represent the keys.
        const int kb = pl->K == 16 ? 4 : pl->K == 8 ? 3 : 2;
        if (pl->track == 2 && pl->chain1 && -((long long)sc.h + sc.g) >= (1ll << (31 - kb))) pl->chain1 = false;
    }
    const int K = pl->K, R = pl->R, W = 32 * K;
    // resident-strips mode: every strip of the plan fits a warp slot of its own (single-warp CTAs, 16 per SM: the
    // launch bounds cap the registers at 128 and 16 x (per-warp shared memory + 1 KB) fits the SM for every K)
    {
        const uint64_t ns = pl->n_strips;
        // measured: 41 % of the warp slots (980 strips) 96 -> 76 ms, 60 % (6 corona pairs) 5.5 -> 4.6 ms, 83 % (1954 strips)
        // 352 -> 357 ms: with most slots busy the ticket order's interleaving of panels does as well, so stop at 70 %
        pl->resident = ns > 0 && ns * 10 <= (uint64_t)c->sm_count * warps_per_sm(K) * 7 && pl->tun.tickets < 0;
        if (pl->tun.resident >= 0 && ns <= (uint64_t)c->sm_count * warps_per_sm(K)) pl->resident = pl->tun.resident != 0;
    }
    // hand-off batch length (gx_fill.cuh, Geo): 32 steps when the plan keeps every warp slot busy (ticket mode: the per-batch
    // glue is what is left to amortise), short batches when the pipeline ramp of a pair -- strips x (31 + batch) steps --
    // is where the time goes (resident strips).  profiles/r2e_sweep_batch_*.jsonl.
    const uint32_t SPC = 64u / (uint32_t)(R * K), CPB_MAX = std::max(1u, 32u / (SPC * (uint32_t)R));
    {
        // (measured after the batch length became a run-time parameter, profiles/r2f_sweep_shards_batch.jsonl: 32 steps is
        // also as good or better for resident strips -- BRCA2 1.08 -> 1.00 ms, one 30 kb pair 2.93 -> 2.74 ms, the 6-pair shard
        // 4.74 -> 4.69 ms -- so every plan uses the longest batch; GX_BATCH forces another length)
        uint32_t steps = 32u;
        if (pl->tun.batch > 0) steps = (uint32_t)pl->tun.batch;
        uint32_t cpb = std::max(1u, steps / SPC);
        while (cpb & (cpb - 1)) cpb &= cpb - 1;          // power of two
        pl->cpb = std::min(cpb, CPB_MAX);
    }
    const uint32_t CPB = pl->cpb, BATCH = CPB * SPC;
    pl->pairs.resize(n_pairs);
    std::vector<TileDesc> tiles;
    std::vector<uint64_t> sbase(n_pairs, 0);
    uint64_t n_tiles_total = 0;
    uint64_t colbuf = 0, top = 0, codes = 0, ops = 0, progress = 0, best = 0;
    uint64_t strip_base = 0;   // band plans: strips of all bands form one sequence
    for (uint64_t q = 0; q < n_pairs; ++q) {
        PairDesc &pd = pl->pairs[q];
        memset(&pd, 0, sizeof pd);
        const uint64_t m = len1[q], n = len2[q];
        pd.m = (uint32_t)m;
        pd.n = (uint32_t)n;
        const bool interior = m > 0 && n > 0;
        pd.S = interior ? (uint32_t)((n + W - 1) / W) : 0;
        pd.P = interior ? (uint32_t)((m + PANEL_H - 1) / PANEL_H) : 0;
        pd.colbuf_off = colbuf;
        pd.top_off = top;
        pd.codes_off = codes;
        pd.ops_off = ops;
        pd.progress_off = (uint32_t)progress;
        pd.tile_base = (uint32_t)best;
        const uint32_t rows_max = (uint32_t)std::min<uint64_t>(m, PANEL_H);
        pd.tile_code_bytes = interior ? tile_batches(rows_max, (uint32_t)R, BATCH) * CPB * 32 * 16 : 0;
        pd.col0 = band_col0 ? (uint32_t)band_col0[q] : 0u;
        if (interior) {
            colbuf += (uint64_t)(pd.S - 1) * m;
            top += n;
            progress += pd.S;
            if (progress >= (1ull << 32) || best + (uint64_t)pd.S * pd.P >= (1ull << 32)) {
                delete pl;
                return GX_ERR_RANGE;
            }
            best += (uint64_t)pd.S * pd.P;
            if (pl->traceback) codes += (uint64_t)pd.S * pd.P * pd.tile_code_bytes;
        }
        if (pl->traceback) ops += ((m + n + 1) + 31) & ~uint64_t(31);
        sbase[q] = strip_base;
        n_tiles_total += (uint64_t)pd.S * pd.P;
        if (band_col0) strip_base += pd.S;
    }
    if (n_tiles_total >= (1ull << 32) - 65536) {
        delete pl;
        return GX_ERR_RANGE;
    }
    if (!pl->resident) {
        std::vector<uint32_t> Sv(n_pairs), Pv(n_pairs);
        for (uint64_t q = 0; q < n_pairs; ++q) {
            Sv[q] = pl->pairs[q].S;
            Pv[q] = pl->pairs[q].P;
        }
        tiles.reserve(n_tiles_total);
        build_ticket_order(Sv, Pv, sbase, tiles);
    }
    pl->n_tiles = n_tiles_total;
    std::vector<TileDesc> strips;
    {
        if (pl->resident) {
            for (uint64_t q = 0; q < n_pairs; ++q) pl->pmax = std::max(pl->pmax, pl->pairs[q].P);
            for (uint64_t q = 0; q < n_pairs; ++q)
                for (uint32_t s2 = 0; s2 < pl->pairs[q].S; ++s2)
                    for (uint32_t p2 = 0; p2 < pl->pmax; ++p2)
                        strips.push_back(p2 < pl->pairs[q].P ? TileDesc{(uint32_t)q, p2, s2, 0u} : TileDesc{0xffffffffu, 0u, 0u, 0u});
        }
    }
    pl->code_bytes = codes;
    pl->ops_bytes = ops;
    pl->colbuf_entries = colbuf;
    pl->top_entries = top;
    pl->progress_entries = progress;
    pl->best_entries = best;

    A(n_pairs * sizeof(PairDesc), (void **)&pl->d_pairs);
    A(tiles.size() * sizeof(TileDesc), (void **)&pl->d_tiles);
    if (pl->resident) A(strips.size() * sizeof(TileDesc), (void **)&pl->d_strips);
    A((16 + progress) * 4, (void **)&pl->d_ctrl);
    A(colbuf * 8, (void **)&pl->d_colbuf);
    A(top * 8, (void **)&pl->d_top);
    if (pl->traceback) A(codes, (void **)&pl->d_codes);
    if (pl->is_local) A(best * 16, (void **)&pl->d_best);
    if (pl->lcs) {
        pl->carry_words = (uint32_t)((max_len + 31) / 32 + 1);
        A(best * 16 + 16, (void **)&pl->d_first);
        A((size_t)n_pairs * 256 * LCS_BLOCK_WORDS * 4, (void **)&pl->d_masks);
        A((size_t)n_pairs * 2 * pl->carry_words * 4 + 16, (void **)&pl->d_carry);
    }
    A(n_pairs * sizeof(DevResult), (void **)&pl->d_results);
    // code band (see gx_common.cuh): global traceback plans.  A global alignment's path runs along the scaled diagonal
    // j = i*n/m (all 45 coronavirus pairs stay within 316 columns of it): default half-width 1024 + |m - n| columns.
    // (6-pair shard, resident strips: fill 4.67 -> 4.07 ms; a single pair gains nothing -- its chain of strips runs at the
    // pace of the strips that do write codes -- and loses nothing.)
    std::vector<uint8_t> tile_codes;
    if (pl->traceback && !is_local && !band_col0 && (!pl->resident || pl->tun.band_resident != 0) && pl->tun.code_band != 0 && best > 0) {
        tile_codes.assign(best, 1);
        double with = 0, all = 0;
        for (uint64_t q = 0; q < n_pairs; ++q) {
            const PairDesc &pd = pl->pairs[q];
            const uint64_t dmn = pd.m > pd.n ? pd.m - pd.n : pd.n - pd.m;
            const uint64_t cw = pl->tun.code_band > 0 ? (uint64_t)pl->tun.code_band : 1024 + dmn;
            for (uint32_t p2 = 0; p2 < pd.P; ++p2) {
                const double rows = (double)std::min<uint64_t>(PANEL_H, pd.m - (uint64_t)p2 * PANEL_H);
                for (uint32_t s2 = 0; s2 < pd.S; ++s2) {
                    const double cols = (double)std::min<uint64_t>((uint64_t)W, pd.n - (uint64_t)s2 * W);
                    const bool in = tile_in_code_band(pd.m, pd.n, p2, s2, (uint32_t)W, cw);
                    tile_codes[pd.tile_base + (uint64_t)p2 * pd.S + s2] = in ? 1 : 0;
                    all += rows * cols;
                    if (in) with += rows * cols;
                }
            }
        }
        pl->code_cell_frac = all > 0 ? with / all : 1.0;
        pl->code_band = pl->code_cell_frac < 0.9;     // not worth a second kernel variant otherwise
        if (!pl->code_band) pl->code_cell_frac = 1.0;
        if (pl->code_band) A(best, (void **)&pl->d_tile_codes);
    }
    if (pl->traceback) A(ops, (void **)&pl->d_ops);
    if (rc == GX_OK && pl->code_band) {
        cudaError_t e = cudaMemcpyAsync(pl->d_tile_codes, tile_codes.data(), best, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail_cuda(e, "upload tile code flags");
    }
    if (rc == GX_OK && (!tiles.empty() || !strips.empty())) {
        cudaError_t e = cudaSuccess;
        if (!tiles.empty()) e = cudaMemcpyAsync(pl->d_tiles, tiles.data(), tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess && pl->resident)
            e = cudaMemcpyAsync(pl->d_strips, strips.data(), strips.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail_cuda(e, "upload tiles");
    }
    if (rc != GX_OK) {
        plan_release(pl);
        delete pl;
        return rc;
    }
    *out = pl;
    return GX_OK;
}


// ------------------------------------------------------------------------------------------------
// Streamed score batch: large read sets (BASELINE config 4: 10 M x 150 bp) are cut into chunks of 2^18 pairs that flow
// through NLANES lanes (stream + device buffers each): while chunk c runs on the SMs, chunks c+1, c+2 cross PCIe and the
// scores of chunk c-1 come back.  The caller's arrays are used as they are (64-bit offsets and lengths, byte blob): the
// only host work is one validating pass and one pass that packs 16-byte records straight into pinned memory, both
// split over a few threads.  Returns GX_ERR_UNSUPPORTED when the batch does not qualify (the caller falls back to a plan).
template <class F>
static void host_parallel(int threads, uint64_t n, F &&f) {   // f(tid, lo, hi) over [0, n) in `threads` contiguous slices
    if (threads <= 1 || n < (1u << 15)) {
        f(0, (uint64_t)0, n);
        return;
    }
    std::vector<std::thread> th;
    th.reserve(threads - 1);
    const uint64_t per = (n + threads - 1) / threads;
    for (int t = 1; t < threads; ++t) {
        const uint64_t lo = std::min<uint64_t>(n, per * t), hi = std::min<uint64_t>(n, per * (t + 1));
        th.emplace_back([&f, t, lo, hi] { f(t, lo, hi); });
    }
    f(0, (uint64_t)0, std::min<uint64_t>(n, per));
    for (auto &t : th) t.join();
}

// start_i / start_j (both or neither): also each pair's start cell -- the read kernels' for local batches, (m, n) for global.
static int score_batch_streamed(const uint8_t *blob, uint64_t blob_len, const uint64_t *off1, const uint64_t *len1,
                                const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local,
                                int64_t *scores, uint64_t *start_i, uint64_t *start_j, bool force32) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!g_ctx) return GX_ERR_NOT_INIT;
    Ctx *c = g_ctx;
    if (n_pairs < (1u << 18) || (is_local && sc.s_mismatch >= 0)) return GX_ERR_UNSUPPORTED;
    int rc = check_scores_impl(sc, READS_MAX_LEN, READS_MAX_LEN, is_local != 0);
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    constexpr int NL = Ctx::NLANES;
    const uint64_t CH = 1u << 18;   // pairs per chunk: ~80 MB of 150 bp reads, ~1.5 ms of PCIe, ~1.5 ms of kernel
    const int T = std::min(c->host_threads, 16);
    if (c->lane_scores_cap < CH) {
        for (int k = 0; k < NL; ++k) {
            if (c->lane_scores_host[k]) cudaFreeHost(c->lane_scores_host[k]);
            c->lane_scores_host[k] = nullptr;
            if (c->lane_rec_host[k]) cudaFreeHost(c->lane_rec_host[k]);
            c->lane_rec_host[k] = nullptr;
            if (cudaHostAlloc((void **)&c->lane_scores_host[k], CH * sizeof(int), cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&c->lane_rec_host[k], CH * sizeof(uint4), cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                c->lane_scores_cap = 0;
                return GX_ERR_NOMEM;
            }
        }
        c->lane_scores_cap = CH;
    }
    const bool cells = start_i && is_local;   // global start cells are (m, n): written by the host in drain()
    if (cells && c->lane_cells_cap < CH) {
        for (int k = 0; k < NL; ++k) {
            if (c->lane_cells_host[k]) cudaFreeHost(c->lane_cells_host[k]);
            c->lane_cells_host[k] = nullptr;
            if (cudaHostAlloc((void **)&c->lane_cells_host[k], CH * sizeof(uint32_t), cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                c->lane_cells_cap = 0;
                return GX_ERR_NOMEM;
            }
        }
        c->lane_cells_cap = CH;
    }
    struct Lane {
        uint8_t *blob = nullptr;
        size_t blob_cap = 0;
        uint4 *rec = nullptr;
        int *scores = nullptr;
        uint32_t *cells = nullptr;
        uint64_t first = 0, count = 0;
        bool busy = false;
    } lane[NL];
    auto release = [&]() {
        for (auto &L : lane) {
            void *ptrs[] = {L.blob, L.rec, L.scores, L.cells};
            for (void *p : ptrs) pool_free(c, p);
        }
    };
    auto drain = [&](int k) -> int {   // scores (and start cells) of the chunk that ran on lane k -> caller's arrays
        Lane &L = lane[k];
        if (!L.busy) return GX_OK;
        cudaError_t e = cudaEventSynchronize(c->lane_done[k]);
        if (e != cudaSuccess) return fail_cuda(e, "cudaEventSynchronize(lane_done)");
        const int *src = c->lane_scores_host[k];
        int64_t *dst = scores + L.first;
        for (uint64_t q = 0; q < L.count; ++q) dst[q] = src[q];
        if (cells) {
            const uint32_t *cs = c->lane_cells_host[k];
            for (uint64_t q = 0; q < L.count; ++q) {
                start_i[L.first + q] = cs[q] >> 16;
                start_j[L.first + q] = cs[q] & 0xffffu;
            }
        } else if (start_i) {
            for (uint64_t q = L.first; q < L.first + L.count; ++q) {
                start_i[q] = len1[q];
                start_j[q] = len2[q];
            }
        }
        L.busy = false;
        return GX_OK;
    };
    for (int k = 0; k < NL && rc == GX_OK; ++k) {
        Lane &L = lane[k];
        rc = pool_alloc(c, CH * sizeof(uint4), (void **)&L.rec);
        if (!rc) rc = pool_alloc(c, CH * 4, (void **)&L.scores);
        if (!rc && cells) rc = pool_alloc(c, CH * 4, (void **)&L.cells);
    }
    struct Part {
        uint64_t lo = UINT64_MAX, hi = 0, maxlen = 0, sum = 0, bad = 0;
    };
    std::vector<Part> parts((size_t)std::max(T, 1));
    // errors inside the chunk loop leave through `break`: the lanes are drained and their pool blocks released below
#define CKB(call)                                   \
    {                                               \
        cudaError_t e__ = (call);                   \
        if (e__ != cudaSuccess) {                   \
            rc = fail_cuda(e__, #call);             \
            break;                                  \
        }                                           \
    }
    for (uint64_t first = 0, ci = 0; first < n_pairs && rc == GX_OK; first += CH, ++ci) {
        const int k = (int)(ci % NL);
        Lane &L = lane[k];
        const uint64_t count = std::min<uint64_t>(CH, n_pairs - first);
        const uint64_t *o1 = off1 + first, *o2 = off2 + first, *l1 = len1 + first, *l2 = len2 + first;
        // host pass 1 over the chunk: bounds, longest sequence, byte span of the chunk in the blob (branch-free: vectorises)
        for (auto &p : parts) p = Part();
        host_parallel(T, count, [&](int tid, uint64_t a, uint64_t b) {
            Part p;
            for (uint64_t q = a; q < b; ++q) {
                const uint64_t a0 = o1[q], a1 = a0 + l1[q], b0 = o2[q], b1 = b0 + l2[q];
                p.bad |= (uint64_t)(a1 > blob_len) | (uint64_t)(b1 > blob_len) | (uint64_t)(a1 < a0) | (uint64_t)(b1 < b0);
                p.lo = std::min(p.lo, std::min(a0, b0));
                p.hi = std::max(p.hi, std::max(a1, b1));
                p.maxlen = std::max(p.maxlen, std::max(l1[q], l2[q]));
                p.sum += l1[q] + l2[q];
            }
            parts[(size_t)tid] = p;
        });
        uint64_t lo = UINT64_MAX, hi = 0, maxlen = 0, sum = 0, badbits = 0;
        for (const auto &p : parts) {
            lo = std::min(lo, p.lo);
            hi = std::max(hi, p.hi);
            maxlen = std::max(maxlen, p.maxlen);
            sum += p.sum;
            badbits |= p.bad;
        }
        if (badbits) {
            rc = GX_ERR_ARG;
            break;
        }
        if (maxlen > (uint64_t)READS_MAX_LEN || hi - lo > 4 * sum + (1u << 20) || hi - lo >= (1ull << 32)) {
            rc = GX_ERR_UNSUPPORTED;   // long pairs or a scattered blob: not a read stream
            break;
        }
        rc = drain(k);                 // the chunk that used this lane NLANES rounds ago
        if (rc) break;
        const uint64_t span = hi > lo ? hi - lo : 0;
        if (L.blob_cap < span + 64) {
            pool_free(c, L.blob);
            L.blob = nullptr;
            L.blob_cap = 0;
            rc = pool_alloc(c, span + span / 4 + 64, (void **)&L.blob);
            if (rc) break;
            L.blob_cap = span + span / 4 + 64;
        }
        cudaStream_t st = c->lane_stream[k];
        if (span) CKB(cudaMemcpyAsync(L.blob, blob + lo, span, cudaMemcpyHostToDevice, st));
        // host pass 2: 16-byte records relative to the chunk's first byte, written straight into pinned memory
        // (lane k's record buffer is free: drain(k) above waited for the chunk that used it)
        {
            uint4 *rec = c->lane_rec_host[k];
            host_parallel(T, count, [&](int, uint64_t a, uint64_t b) {
                for (uint64_t q = a; q < b; ++q)
                    rec[q] = make_uint4((uint32_t)(o1[q] - lo), (uint32_t)(o2[q] - lo), (uint32_t)l1[q], (uint32_t)l2[q]);
            });
        }
        CKB(cudaMemcpyAsync(L.rec, c->lane_rec_host[k], count * sizeof(uint4), cudaMemcpyHostToDevice, st));
        ReadsParams rp;
        rp.blob = L.blob;
        rp.off1 = rp.off2 = nullptr;
        rp.len1 = rp.len2 = nullptr;
        rp.rec = L.rec;
        rp.n_pairs = (uint32_t)count;
        rp.scores = L.scores;
        rp.results = nullptr;
        rp.a = sc.s_match;
        rp.b = sc.s_mismatch;
        rp.g = sc.g;
        rp.h = sc.h;
        rp.is_local = is_local ? 1 : 0;
        rp.cells = cells ? L.cells : nullptr;
        if (launch_reads(rp, (int)maxlen, c->sm_count, st, force32) != 0) {
            rc = GX_ERR_UNSUPPORTED;
            break;
        }
        CKB(cudaGetLastError());
        CKB(cudaMemcpyAsync(c->lane_scores_host[k], L.scores, count * 4, cudaMemcpyDeviceToHost, st));
        if (cells) CKB(cudaMemcpyAsync(c->lane_cells_host[k], L.cells, count * 4, cudaMemcpyDeviceToHost, st));
        CKB(cudaEventRecord(c->lane_done[k], st));
        L.first = first;
        L.count = count;
        L.busy = true;
    }
#undef CKB
    for (int k = 0; k < NL && rc == GX_OK; ++k) rc = drain(k);
    if (rc != GX_OK) {
        for (int k = 0; k < NL; ++k) cudaStreamSynchronize(c->lane_stream[k]);
        cudaGetLastError();
    }
    release();
    return rc;
}

extern "C" {

int gx_plan_create(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local, int flags,
                   gx_plan **out) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    return plan_create_locked(len1, len2, n_pairs, sc, is_local, flags, nullptr, out);
}
GX_GUARD_END

int gx_plan_upload(gx_plan *pl, const uint8_t *blob, uint64_t blob_len, const uint64_t *off1, const uint64_t *off2) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl || (!blob && blob_len) || ((!off1 || !off2) && pl->n_pairs)) return GX_ERR_ARG;
    Ctx *c = pl->ctx;
    CK(cudaSetDevice(c->device));
    for (uint64_t q = 0; q < pl->n_pairs; ++q)   // written so that a huge offset cannot wrap around
        if (off1[q] > blob_len || pl->len1[q] > blob_len - off1[q] || off2[q] > blob_len || pl->len2[q] > blob_len - off2[q])
            return GX_ERR_ARG;
    if (!pl->d_blob || pl->blob_cap < blob_len + 64) {
        pool_free(c, pl->d_blob);
        pl->d_blob = nullptr;
        int rc = pool_alloc(c, blob_len + 64, (void **)&pl->d_blob);
        if (rc) return rc;
        pl->blob_cap = blob_len + 64;
        pl->dev_bytes += blob_len + 64;
    }
    if (blob_len) CK(cudaMemcpyAsync(pl->d_blob, blob, blob_len, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(pl->d_blob + blob_len, 0, 64, c->stream));
    pl->h2d_bytes = blob_len;
    if (pl->kind == KIND_READS) {
        if (pl->n_pairs) {
            CK(cudaMemcpyAsync(pl->d_off1, off1, pl->n_pairs * 8, cudaMemcpyHostToDevice, c->stream));
            CK(cudaMemcpyAsync(pl->d_off2, off2, pl->n_pairs * 8, cudaMemcpyHostToDevice, c->stream));
            pl->h2d_bytes += pl->n_pairs * 16;
        }
    } else {
        // alphabet of the batch: with <= 4 distinct bytes (and scores that fit a byte) the fill uses the one-hot / IDP.4A path:
        // the sequences are re-encoded to SHIFT AMOUNTS 8 * symbol (gx_fill.cuh, run_batch)
        bool seen[256] = {false};
        int nsym = 0;
        uint8_t lut[256];
        memset(lut, 255, sizeof lut);
        {
            // every distinct (offset, length) segment once -- all-vs-all batches reuse the same few sequences many times
            std::vector<std::pair<uint64_t, uint64_t>> segs;
            segs.reserve(2 * pl->n_pairs);
            for (uint64_t q = 0; q < pl->n_pairs; ++q) {
                segs.push_back({off1[q], pl->len1[q]});
                segs.push_back({off2[q], pl->len2[q]});
            }
            std::sort(segs.begin(), segs.end());
            segs.erase(std::unique(segs.begin(), segs.end()), segs.end());
            uint64_t done_to = 0;   // bytes below this offset have been scanned (segments sorted by offset)
            for (size_t k = 0; k < segs.size() && nsym <= 4; ++k) {
                uint64_t lo = std::max(segs[k].first, done_to), hi = segs[k].first + segs[k].second;
                for (uint64_t x = lo; x < hi; ++x) {
                    const uint8_t ch = blob[x];
                    if (!seen[ch]) {
                        seen[ch] = true;
                        if (nsym < 4) lut[ch] = (uint8_t)(8 * nsym);
                        nsym++;
                    }
                }
                done_to = std::max(done_to, hi);
            }
        }
        {
            // both forms of the recurrence put (score - (h+g)) resp. the raw score into one signed byte
            const long long hg = (long long)pl->sc.h + pl->sc.g;
            const long long v[4] = {pl->sc.s_match - hg, pl->sc.s_mismatch - hg, pl->sc.s_match, pl->sc.s_mismatch};
            bool fits = true;
            for (long long x : v) fits = fits && x >= -128 && x <= 127;
            pl->prof = nsym <= 4 && fits && pl->n_tiles > 0;
        }
        if (pl->prof) {
            for (int x = 0; x < 256; ++x)
                if (lut[x] == 255) lut[x] = 0;   // bytes outside the pairs' segments (over-read slack): any valid shift amount
            if (!pl->d_lut) {
                int rc = pool_alloc(c, 256, (void **)&pl->d_lut);
                if (rc) return rc;
            }
            pool_free(c, pl->d_blob_sym);
            pl->d_blob_sym = nullptr;
            int rc = pool_alloc(c, blob_len + 64, (void **)&pl->d_blob_sym);
            if (rc) return rc;
            pl->dev_bytes += blob_len + 64;
            CK(cudaMemcpyAsync(pl->d_lut, lut, 256, cudaMemcpyHostToDevice, c->stream));
            const int grid = (int)std::min<uint64_t>((blob_len + 64 + 255) / 256, (uint64_t)c->sm_count * 8);
            gx_encode_kernel<<<grid, 256, 0, c->stream>>>(pl->d_blob, pl->d_blob_sym, (size_t)blob_len + 64, pl->d_lut);
            CK(cudaGetLastError());
        }
        for (uint64_t q = 0; q < pl->n_pairs; ++q) {
            pl->pairs[q].s1_off = off1[q];
            pl->pairs[q].s2_off = off2[q];
        }
        if (pl->n_pairs) {
            CK(cudaMemcpyAsync(pl->d_pairs, pl->pairs.data(), pl->n_pairs * sizeof(PairDesc), cudaMemcpyHostToDevice, c->stream));
            pl->h2d_bytes += pl->n_pairs * sizeof(PairDesc);
        }
    }
    CK(cudaStreamSynchronize(c->stream));
    pl->uploaded = true;
    return GX_OK;
}
GX_GUARD_END

static int plan_execute_once(gx_plan *pl, bool *aborted);

// Ticket-ordered tile list of a plan (built at creation for ticket plans, on demand when a resident-strips plan falls back)
static int plan_build_tickets(gx_plan *pl) {
    Ctx *c = pl->ctx;
    const size_t np = pl->pairs.size();
    std::vector<uint32_t> Sv(np), Pv(np);
    std::vector<uint64_t> sbase(np, 0);
    uint64_t base = 0;
    for (size_t q = 0; q < np; ++q) {
        Sv[q] = pl->pairs[q].S;
        Pv[q] = pl->pairs[q].P;
        sbase[q] = base;
        if (pl->band) base += Sv[q];
    }
    std::vector<TileDesc> tiles;
    tiles.reserve(pl->n_tiles);
    build_ticket_order(Sv, Pv, sbase, tiles);
    if (tiles.size() != pl->n_tiles) return GX_ERR_INTERNAL;
    if (tiles.empty()) return GX_OK;
    pool_free(c, pl->d_tiles);
    pl->d_tiles = nullptr;
    int rc = pool_alloc(c, tiles.size() * sizeof(TileDesc), (void **)&pl->d_tiles);
    if (rc) return rc;
    CK(cudaMemcpyAsync(pl->d_tiles, tiles.data(), tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return GX_OK;
}

int gx_plan_execute(gx_plan *pl) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl) return GX_ERR_ARG;
    if (!pl->uploaded) return GX_ERR_ARG;
    bool aborted = false;
    int rc = plan_execute_once(pl, &aborted);
    // A resident-strips fill that gave up waiting (SPIN_LIMIT: the device was shared with something that kept its strips
    // from running together, or was lost) is repeated ONCE in ticket mode, where a waiting warp only ever waits for
    // warps that hold earlier tickets.  Band plans that span processes cannot be rewound: they stay failed (poisoned).
    if (rc == GX_ERR_INTERNAL && aborted && pl->resident && !(pl->band && pl->band->n_bands > pl->band->last - pl->band->first)) {
        pl->resident = false;
        pl->retries++;
        int rb = plan_build_tickets(pl);
        if (rb) return rb;
        pl->colbuf_dirty = true;     // the aborted execute left the LL parity words in an unknown state
        rc = plan_execute_once(pl, &aborted);
    }
    // A path left the code band (a walk needed a tile that wrote no codes): repeat with codes in every tile.  The band is
    // an optimisation of where traceback pointers are STORED, never of what is computed, so this keeps every result exact;
    // the time of the discarded attempt stays in fill_ms / walk_ms.
    if (rc == GX_OK && pl->code_band && pl->left_band != 0) {
        const float f0 = pl->fill_ms, w0 = pl->walk_ms;
        const int l0 = pl->launches;
        pl->code_band = false;
        pl->code_cell_frac = 1.0;
        pl->band_fallbacks++;
        rc = plan_execute_once(pl, &aborted);
        pl->fill_ms += f0;
        pl->walk_ms += w0;
        pl->launches += l0;
    }
    return rc;
}
GX_GUARD_END

static int plan_execute_once(gx_plan *pl, bool *aborted) {
    Ctx *c = pl->ctx;
    CK(cudaSetDevice(c->device));
    pl->launches = 0;
    pl->fill_ms = pl->walk_ms = 0;
    const gx_scores sc = pl->sc;
    if (pl->n_pairs == 0) {
        pl->executed = true;
        return GX_OK;
    }
    if (pl->kind == KIND_READS) {
        ReadsParams rp;
        rp.blob = pl->d_blob;
        rp.off1 = pl->d_off1;
        rp.off2 = pl->d_off2;
        rp.len1 = pl->d_len1;
        rp.len2 = pl->d_len2;
        rp.rec = nullptr;
        rp.n_pairs = (uint32_t)pl->n_pairs;
        rp.scores = pl->d_scores;
        rp.results = nullptr;
        rp.a = sc.s_match;
        rp.b = sc.s_mismatch;
        rp.g = sc.g;
        rp.h = sc.h;
        rp.is_local = pl->is_local;
        rp.cells = pl->d_cells;
        CK(cudaEventRecord(c->ev[0], c->stream));
        int rc = launch_reads(rp, (int)pl->max_len, c->sm_count, c->stream, pl->tun.reads32 != 0, &pl->reads_bits);
        if (rc == -1) return GX_ERR_UNSUPPORTED;
        CK(cudaGetLastError());
        CK(cudaEventRecord(c->ev[1], c->stream));
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaEventElapsedTime(&pl->fill_ms, c->ev[0], c->ev[1]));
        pl->launches = 1;
        pl->executed = true;
        return GX_OK;
    }

    gx_band *bd = pl->band;
    if (bd && bd->poisoned) {
        g_err = "band plan is unusable after a failed execute (neighbouring bands are out of step): create it again";
        return GX_ERR_INTERNAL;
    }
    CK(cudaEventRecord(c->ev[0], c->stream));   // the step's device time includes its own control-word reset
    if (pl->colbuf_dirty) {
        if (pl->colbuf_entries) CK(cudaMemsetAsync(pl->d_colbuf, 0xff, pl->colbuf_entries * 8, c->stream));  // parity bit 1 everywhere
        if (bd) {
            if (bd->epoch != 0 && bd->n_bands > bd->last - bd->first) {   // a remote neighbour cannot be rewound
                bd->poisoned = true;
                return GX_ERR_INTERNAL;
            }
            for (auto *lk : bd->internal) CK(cudaMemsetAsync(lk, 0xff, bd->m * 8, c->stream));
        }
        pl->parity = 0;
    }
    pl->colbuf_dirty = true;  // until this execute completes
    CK(cudaMemsetAsync(pl->d_ctrl, 0, (16 + pl->progress_entries) * 4, c->stream));
    FillParams fp;
    fp.blob = pl->d_blob;
    fp.blob_sym = pl->prof ? pl->d_blob_sym : nullptr;
    fp.one = 1u;
    fp.stats = nullptr;
    fp.timeline = nullptr;
    fp.pad_keys = (sc.s_mismatch >= 0 || pl->tun.pad_keys) ? 1u : 0u;
    fp.poll_nap = (uint32_t)pl->tun.poll_nap;
    fp.start_lead = (uint32_t)pl->tun.start_lead;
    if (pl->tun.fill_stats) {
        if (!pl->d_stats) {
            int rc = pool_alloc(c, 64, (void **)&pl->d_stats);
            if (rc) return rc;
        }
        CK(cudaMemsetAsync(pl->d_stats, 0, 64, c->stream));
        fp.stats = pl->d_stats;
        if (pl->tun.fill_stats >= 2) {
            if (!pl->d_timeline) {
                int rc = pool_alloc(c, (std::max<uint64_t>(pl->n_tiles, pl->n_strips * pl->pmax) + 1) * 32, (void **)&pl->d_timeline);
                if (rc) return rc;
            }
            fp.timeline = pl->d_timeline;
        }
    }
    fp.pairs = pl->d_pairs;
    fp.n_pairs = (uint32_t)pl->n_pairs;
    fp.code_bytes = pl->code_bytes;
    fp.tiles = pl->d_tiles;
    fp.n_tiles = (uint32_t)pl->n_tiles;
    fp.pmax = 0;   // launch_fill switches to the [strip][panel] list when every strip gets a warp
    fp.parity = pl->parity;
    fp.cpb = pl->cpb;
    fp.epoch = bd ? bd->epoch + 1 : 0;
    fp.ticket = pl->d_ctrl;
    fp.progress = pl->d_ctrl + 16;
    fp.colbuf = pl->d_colbuf;
    fp.top = pl->d_top;
    fp.codes = pl->d_codes;
    fp.tile_best = pl->d_best;
    fp.g = sc.g;
    fp.h = sc.h;
    fp.hg = sc.h + sc.g;
    fp.ap = sc.s_match - fp.hg;
    fp.bp = sc.s_mismatch - fp.hg;
    if (pl->n_tiles) {
        int rc = launch_fill(pl, fp, 0);
        if (rc) return rc;
        pl->launches++;
    }
    CK(cudaEventRecord(c->ev[1], c->stream));
    if (bd && bd->left_base) {   // our inbox is consumed: the left neighbour may start its next execute
        gx_band_ack_kernel<<<1, 1, 0, c->stream>>>(reinterpret_cast<uint32_t *>(bd->left_base), bd->epoch + 1);
        CK(cudaGetLastError());
        pl->launches++;
    }
    WalkParams wp;
    wp.blob = pl->d_blob;
    wp.pairs = pl->d_pairs;
    wp.n_pairs = (uint32_t)pl->n_pairs;
    wp.top = pl->d_top;
    wp.codes = pl->d_codes;
    wp.tile_best = pl->d_best;
    wp.results = pl->d_results;
    wp.ops = pl->d_ops;
    wp.g = sc.g;
    wp.h = sc.h;
    wp.hg = fp.hg;
    wp.kcols_log2 = pl->K == 16 ? 4 : pl->K == 4 ? 2 : 3;
    wp.is_local = pl->is_local;
    wp.traceback = pl->traceback ? 1 : 0;
    wp.have_best = pl->track == 2 ? 1 : 0;
    wp.debug = pl->tun.walk_stats;
    wp.check = pl->d_ctrl + 2;
    wp.left_band = pl->d_ctrl + 3;
    wp.tile_codes = pl->code_band ? pl->d_tile_codes : nullptr;
    wp.code_bytes = pl->code_bytes;
    wp.ops_bytes = pl->ops_bytes;
    {
        int rc = launch_walk(pl, wp);
        if (rc) return rc;
        pl->launches++;
    }
    CK(cudaEventRecord(c->ev[2], c->stream));
    uint32_t ctrl_words[3] = {0, 0, 0};   // [0] abort word, [1] checked build: site of a failed bounds check, [2] walks outside the code band
    CK(cudaMemcpyAsync(ctrl_words, pl->d_ctrl + 1, 12, cudaMemcpyDeviceToHost, c->stream));
    uint32_t ctrl2[2] = {0, 0};
    if (pl->lcs) {
        // alignment_table's second return value: a score-only fill pass that tracks the FIRST maximum, then the LCS
        // length of the two prefixes that end there (gx_lcs.cuh)
        if (pl->n_tiles) {
            CK(cudaMemsetAsync(pl->d_ctrl, 0, (16 + pl->progress_entries) * 4, c->stream));
            FillParams fq = fp;
            fq.parity = pl->parity ^ 1u;
            fq.codes = nullptr;
            fq.tile_best = pl->d_first;
            fq.stats = nullptr;
            fq.timeline = nullptr;
            int rc = launch_fill(pl, fq, 0, 3);
            if (rc) return rc;
            pl->launches++;
            CK(cudaMemcpyAsync(ctrl2, pl->d_ctrl + 1, 8, cudaMemcpyDeviceToHost, c->stream));
        }
        LcsParams lp;
        lp.blob = pl->d_blob;
        lp.pairs = pl->d_pairs;
        lp.n_pairs = (uint32_t)pl->n_pairs;
        lp.tile_first = pl->d_first;
        lp.masks = pl->d_masks;
        lp.carry = pl->d_carry;
        lp.carry_words = pl->carry_words;
        lp.results = pl->d_results;
        gx_lcs_kernel<<<(unsigned)pl->n_pairs, 32, 0, c->stream>>>(lp);
        CK(cudaGetLastError());
        pl->launches++;
        CK(cudaEventRecord(c->ev[3], c->stream));
    }
    if (fp.stats) CK(cudaMemcpyAsync(pl->h_stats, pl->d_stats, 64, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    uint32_t abort_word = ctrl_words[0];
    const uint32_t abort_word2 = ctrl2[0];
    if (ctrl_words[1] || ctrl2[1]) {
        g_err = "checked build: device bounds check failed at site " + std::to_string(ctrl_words[1] ? ctrl_words[1] : ctrl2[1]);
        return GX_ERR_INTERNAL;
    }
    if (pl->tun.test_abort && pl->resident && pl->retries == 0) abort_word = 1;   // test hook: exercise the ticket-mode retry
    if (abort_word || abort_word2) {
        g_err = "fill kernel aborted: a tile waited > SPIN_LIMIT polls for a dependency";
        if (bd && bd->n_bands > bd->last - bd->first) bd->poisoned = true;
        *aborted = true;
        return GX_ERR_INTERNAL;
    }
    if (bd) bd->epoch++;
    pl->left_band = ctrl_words[2];
    CK(cudaEventElapsedTime(&pl->fill_ms, c->ev[0], c->ev[1]));
    CK(cudaEventElapsedTime(&pl->walk_ms, c->ev[1], c->ev[2]));
    if (pl->lcs) CK(cudaEventElapsedTime(&pl->lcs_ms, c->ev[2], c->ev[3]));
    if (!(pl->lcs && pl->n_tiles)) pl->parity ^= 1u;   // with the first-maximum pass the fill ran twice: parity is back
    pl->colbuf_dirty = false;
    pl->executed = true;
    return GX_OK;
}

int gx_plan_fetch(gx_plan *pl, gx_result *out, uint8_t *ops_blob, const uint64_t *ops_off) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl || (!out && pl->n_pairs)) return GX_ERR_ARG;
    if (!pl->executed) return GX_ERR_ARG;
    if (pl->traceback && pl->n_pairs && (!ops_blob || !ops_off)) return GX_ERR_ARG;
    Ctx *c = pl->ctx;
    CK(cudaSetDevice(c->device));
    if (pl->n_pairs == 0) return GX_OK;
    if (pl->kind == KIND_READS) {
        std::vector<int> sc32(pl->n_pairs);
        std::vector<uint32_t> cells(pl->d_cells ? pl->n_pairs : 0);
        CK(cudaMemcpyAsync(sc32.data(), pl->d_scores, pl->n_pairs * 4, cudaMemcpyDeviceToHost, c->stream));
        if (pl->d_cells) CK(cudaMemcpyAsync(cells.data(), pl->d_cells, pl->n_pairs * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        pl->d2h_bytes = pl->n_pairs * (pl->d_cells ? 8 : 4);
        for (uint64_t q = 0; q < pl->n_pairs; ++q) {
            gx_result r;
            memset(&r, 0, sizeof r);
            r.score = sc32[q];
            // start cell = end cell, as gx_walk_kernel reports it for score-only plans; (m, n) without start cells
            r.start_i = r.end_i = pl->d_cells ? cells[q] >> 16 : pl->len1[q];
            r.start_j = r.end_j = pl->d_cells ? cells[q] & 0xffffu : pl->len2[q];
            r.fill_ms = pl->fill_ms;
            out[q] = r;
        }
        return GX_OK;
    }
    CK(cudaMemcpyAsync(out, pl->d_results, pl->n_pairs * sizeof(gx_result), cudaMemcpyDeviceToHost, c->stream));
    pl->d2h_bytes = pl->n_pairs * sizeof(gx_result);
    if (pl->traceback) {
        if (c->ops_stage_cap < pl->ops_bytes) {
            if (c->ops_stage) cudaFreeHost(c->ops_stage);
            c->ops_stage = nullptr;
            c->ops_stage_cap = 0;
            const size_t want = pl->ops_bytes + pl->ops_bytes / 4 + 4096;
            if (cudaHostAlloc((void **)&c->ops_stage, want, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return GX_ERR_NOMEM;
            }
            c->ops_stage_cap = want;
        }
        CK(cudaMemcpyAsync(c->ops_stage, pl->d_ops, pl->ops_bytes, cudaMemcpyDeviceToHost, c->stream));
        pl->d2h_bytes += pl->ops_bytes;
    }
    CK(cudaStreamSynchronize(c->stream));
    int rc = GX_OK;
    const bool walk_dbg = pl->tun.walk_stats != 0;
    for (uint64_t q = 0; q < pl->n_pairs; ++q) {
        if (!walk_dbg) out[q].fill_ms = pl->fill_ms;
        if (!walk_dbg) out[q].walk_ms = pl->walk_ms;
        if (pl->traceback) {
            const uint64_t cap = ops_off[q + 1] - ops_off[q];
            if (out[q].n_ops > cap) {
                rc = GX_ERR_OPS_CAP;
                continue;
            }
            memcpy(ops_blob + ops_off[q], c->ops_stage + pl->pairs[q].ops_off, out[q].n_ops);
        }
    }
    return rc;
}
GX_GUARD_END

int gx_plan_fetch_scores(gx_plan *pl, int64_t *scores) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl || (!scores && pl->n_pairs)) return GX_ERR_ARG;
    if (!pl->executed) return GX_ERR_ARG;
    Ctx *c = pl->ctx;
    CK(cudaSetDevice(c->device));
    if (pl->n_pairs == 0) return GX_OK;
    if (pl->kind == KIND_READS) {
        // int32 on the wire (4 B per pair), widened on the host
        std::vector<int> sc32(pl->n_pairs);
        CK(cudaMemcpyAsync(sc32.data(), pl->d_scores, pl->n_pairs * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        pl->d2h_bytes = pl->n_pairs * 4;
        for (uint64_t q = 0; q < pl->n_pairs; ++q) scores[q] = sc32[q];
        return GX_OK;
    }
    std::vector<gx_result> res(pl->n_pairs);
    CK(cudaMemcpyAsync(res.data(), pl->d_results, pl->n_pairs * sizeof(gx_result), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    pl->d2h_bytes = pl->n_pairs * sizeof(gx_result);
    for (uint64_t q = 0; q < pl->n_pairs; ++q) scores[q] = res[q].score;
    return GX_OK;
}
GX_GUARD_END

int gx_plan_debug_timeline(gx_plan *pl, uint64_t *out, uint64_t cap_words) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl || !out || !pl->d_timeline || cap_words < pl->n_tiles * 4) return GX_ERR_ARG;
    CK(cudaSetDevice(pl->ctx->device));
    CK(cudaMemcpy(out, pl->d_timeline, pl->n_tiles * 32, cudaMemcpyDeviceToHost));
    return GX_OK;
}

// Pure host arithmetic (no device): the ticket order plan_create would use for these pairs at register blocking K
// (bands != 0: the pairs are consecutive column bands of one table).  out = {pair, panel, strip} triples.
int gx_debug_tile_order(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs, int K, int bands, uint32_t *out,
                        uint64_t cap_tiles, uint64_t *n_tiles) try {
    if ((!len1 || !len2) && n_pairs) return GX_ERR_ARG;
    if (!n_tiles || (K != 2 && K != 4 && K != 8 && K != 16)) return GX_ERR_ARG;
    std::vector<uint32_t> S(n_pairs), P(n_pairs);
    std::vector<uint64_t> sbase(n_pairs, 0);
    uint64_t base = 0, total = 0;
    for (uint64_t q = 0; q < n_pairs; ++q) {
        const bool interior = len1[q] > 0 && len2[q] > 0;
        S[q] = interior ? (uint32_t)((len2[q] + 32 * K - 1) / (32 * K)) : 0;
        P[q] = interior ? (uint32_t)((len1[q] + PANEL_H - 1) / PANEL_H) : 0;
        sbase[q] = base;
        if (bands) base += S[q];
        total += (uint64_t)S[q] * P[q];
    }
    *n_tiles = total;
    if (!out) return GX_OK;
    if (cap_tiles < total) return GX_ERR_ARG;
    std::vector<TileDesc> tiles;
    tiles.reserve(total);
    build_ticket_order(S, P, sbase, tiles);
    if (tiles.size() != total) return GX_ERR_INTERNAL;
    for (size_t k = 0; k < tiles.size(); ++k) {
        out[3 * k + 0] = tiles[k].pair;
        out[3 * k + 1] = tiles[k].p;
        out[3 * k + 2] = tiles[k].s;
    }
    return GX_OK;
}
GX_GUARD_END

double gx_plan_stat(const gx_plan *pl, int what) {
    if (!pl) return -1.0;
    switch (what) {
        case 0: return pl->fill_ms;
        case 1: return pl->walk_ms;
        case 2: return pl->launches;
        case 3: return (double)pl->cells;
        case 4: return (double)pl->code_bytes;
        case 5: return (double)pl->dev_bytes;
        case 6: return (double)pl->h2d_bytes;
        case 7: return (double)pl->d2h_bytes;
        case 8: return (double)pl->n_tiles;
        case 9: return (double)pl->kind;
        case 15: return (double)pl->K;
        case 19: return (double)pl->R;
        case 20: return (double)pl->retries;
        case 23: return pl->code_cell_frac;
        case 24: return (double)pl->band_fallbacks;
        case 22: return (double)(pl->cpb * (64u / (uint32_t)(pl->R * pl->K)));   // steps per hand-off batch
        case 21: return pl->resident ? 1.0 : 0.0;
        case 17: return pl->chain1 ? 1.0 : 0.0;
        case 18: return pl->lcs_ms;
        case 25: return pl->prof ? 1.0 : 0.0;
        case 26: return (double)pl->reads_bits;
        case 10: case 11: case 12: case 13: case 14: return (double)pl->h_stats[what - 10];
        default: return -1.0;
    }
}

void gx_plan_destroy(gx_plan *pl) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!pl) return;
    plan_release(pl);
    delete pl;
}


// ================================================================================================
// Column-banded single pair (BASELINE config 5): SURVEY.md 8e.  Score only, global.
// ================================================================================================
int gx_band_range(uint64_t n_total, int n_bands, int band, uint64_t *col0, uint64_t *width) {
    if (n_bands < 1 || band < 0 || band >= n_bands || !col0 || !width) return GX_ERR_ARG;
    // wide tables: band edges on multiples of 512 columns (a whole strip for every K); narrow ones: even split
    uint64_t lo, hi;
    if (n_total / (uint64_t)n_bands >= std::max<uint64_t>(4096, 512ull * n_bands)) {
        const uint64_t base = ((n_total + n_bands - 1) / n_bands + 511) / 512 * 512;
        lo = std::min<uint64_t>(n_total, base * band);
        hi = std::min<uint64_t>(n_total, base * (band + 1));
    } else {
        const uint64_t q = n_total / n_bands, r = n_total % n_bands;
        lo = q * band + std::min<uint64_t>(band, r);
        hi = lo + q + ((uint64_t)band < r ? 1 : 0);
    }
    *col0 = lo;
    *width = hi - lo;
    return GX_OK;
}

static void band_free(gx_band *b) {
    if (!b) return;
    if (b->plan) gx_plan_destroy(b->plan);
    if (g_ctx) {
        for (auto *p : b->internal) pool_free(g_ctx, p);
        if (b->left_base) cudaIpcCloseMemHandle(b->left_base);
        if (b->right_base) cudaIpcCloseMemHandle(b->right_base);
        if (b->link) cudaFree(b->link);
        cudaGetLastError();
    }
    delete b;
}

int gx_band_create(uint64_t m, uint64_t n_total, int n_bands, int first_band, int last_band, gx_scores sc, gx_band **out) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!out) return GX_ERR_ARG;
    *out = nullptr;
    if (!g_ctx) return GX_ERR_NOT_INIT;
    if (n_bands < 1 || first_band < 0 || last_band <= first_band || last_band > n_bands) return GX_ERR_ARG;
    int rc = check_scores_impl(sc, m, n_total, false);
    if (rc) return rc;
    if (m > 0 && n_total > 0 && n_total < (uint64_t)n_bands) return GX_ERR_ARG;   // every band needs a column
    Ctx *c = g_ctx;
    CK(cudaSetDevice(c->device));
    gx_band *b = new (std::nothrow) gx_band();
    if (!b) return GX_ERR_NOMEM;
    b->m = m;
    b->n_total = n_total;
    b->sc = sc;
    b->n_bands = n_bands;
    b->first = first_band;
    b->last = last_band;
    b->trivial = (m == 0 || n_total == 0);   // boundary-only table: the score is a formula (algo.rs:204-220)
    if (b->trivial) {
        *out = b;
        return GX_OK;
    }
    const int nl = last_band - first_band;
    std::vector<uint64_t> l1(nl, m), l2(nl);
    b->col0.resize(nl);
    b->width.resize(nl);
    for (int q = 0; q < nl; ++q) {
        gx_band_range(n_total, n_bands, first_band + q, &b->col0[q], &b->width[q]);
        l2[q] = b->width[q];
        if (l2[q] == 0) {
            delete b;
            return GX_ERR_ARG;
        }
    }
    rc = plan_create_locked(l1.data(), l2.data(), (uint64_t)nl, sc, 0, 0, b->col0.data(), &b->plan);
    if (rc) {
        delete b;
        return rc;
    }
    b->plan->band = b;
    for (int q = 0; q + 1 < nl && rc == GX_OK; ++q) {
        unsigned long long *p = nullptr;
        rc = pool_alloc(c, m * 8, (void **)&p);
        if (rc == GX_OK) b->internal.push_back(p);
    }
    if (rc == GX_OK && nl < n_bands) {
        // remote neighbours: our link block holds the inbox of our first band and the ack word of our last band
        cudaError_t e = cudaMalloc((void **)&b->link, 256 + m * 8);
        if (e == cudaSuccess) e = cudaMemsetAsync(b->link, 0xff, 256 + m * 8, c->stream);   // parity bit 1 everywhere
        if (e == cudaSuccess) e = cudaMemsetAsync(b->link, 0, 256, c->stream);              // ack = 0 executes finished
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            cudaGetLastError();
            rc = (e == cudaErrorMemoryAllocation) ? GX_ERR_NOMEM : fail_cuda(e, "band link block");
        }
    }
    if (rc != GX_OK) {
        band_free(b);
        return rc;
    }
    // pointers known now: internal links; remote ones are patched in by gx_band_connect
    for (int q = 0; q < nl; ++q) {
        PairDesc &pd = b->plan->pairs[q];
        pd.inbox = (q > 0) ? b->internal[q - 1] : nullptr;
        pd.outbox = (q + 1 < nl) ? b->internal[q] : nullptr;
        pd.ack = nullptr;
    }
    b->connected = (nl == n_bands);
    *out = b;
    return GX_OK;
}
GX_GUARD_END

int gx_band_export(gx_band *b, void *handle, uint64_t handle_cap) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!b || !handle || handle_cap < GX_BAND_HANDLE_BYTES) return GX_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) <= GX_BAND_HANDLE_BYTES, "handle size");
    memset(handle, 0, GX_BAND_HANDLE_BYTES);
    if (!b->link) return GX_OK;   // nothing to share (all bands local, or a boundary-only table)
    CK(cudaSetDevice(g_ctx->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, b->link));
    memcpy(handle, &h, sizeof h);
    return GX_OK;
}

int gx_band_connect(gx_band *b, const void *left_handle, const void *right_handle) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!b) return GX_ERR_ARG;
    if (b->trivial) return GX_OK;
    const bool need_left = b->first > 0, need_right = b->last < b->n_bands;
    if ((need_left && !left_handle) || (need_right && !right_handle)) return GX_ERR_ARG;
    if (b->connected) return GX_OK;
    CK(cudaSetDevice(g_ctx->device));
    const int nl = b->last - b->first;
    if (need_left) {
        cudaIpcMemHandle_t h;
        memcpy(&h, left_handle, sizeof h);
        CK(cudaIpcOpenMemHandle(&b->left_base, h, cudaIpcMemLazyEnablePeerAccess));
        b->plan->pairs[0].inbox = reinterpret_cast<const unsigned long long *>(b->link + 256);
    }
    if (need_right) {
        cudaIpcMemHandle_t h;
        memcpy(&h, right_handle, sizeof h);
        CK(cudaIpcOpenMemHandle(&b->right_base, h, cudaIpcMemLazyEnablePeerAccess));
        b->plan->pairs[nl - 1].outbox = reinterpret_cast<unsigned long long *>(static_cast<uint8_t *>(b->right_base) + 256);
        b->plan->pairs[nl - 1].ack = reinterpret_cast<const uint32_t *>(b->link);
    }
    b->connected = true;
    if (b->plan->uploaded) {
        CK(cudaMemcpyAsync(b->plan->d_pairs, b->plan->pairs.data(), nl * sizeof(PairDesc), cudaMemcpyHostToDevice, g_ctx->stream));
        CK(cudaStreamSynchronize(g_ctx->stream));
    }
    return GX_OK;
}
GX_GUARD_END

int gx_band_upload(gx_band *b, const uint8_t *s1, const uint8_t *s2) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!b) return GX_ERR_ARG;
    if (b->trivial) return GX_OK;
    if (!s1 || !s2) return GX_ERR_ARG;
    const int nl = b->last - b->first;
    const uint64_t c_lo = b->col0[0], c_hi = b->col0[nl - 1] + b->width[nl - 1];
    std::vector<uint8_t> blob(b->m + (c_hi - c_lo));
    memcpy(blob.data(), s1, b->m);
    memcpy(blob.data() + b->m, s2 + c_lo, c_hi - c_lo);
    std::vector<uint64_t> off1(nl, 0), off2(nl);
    for (int q = 0; q < nl; ++q) off2[q] = b->m + (b->col0[q] - c_lo);
    return gx_plan_upload(b->plan, blob.data(), blob.size(), off1.data(), off2.data());
}
GX_GUARD_END

int gx_band_execute(gx_band *b) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!b) return GX_ERR_ARG;
    if (b->trivial) return GX_OK;
    if (!b->connected) return GX_ERR_ARG;
    int rc = gx_plan_execute(b->plan);
    b->fill_ms = b->plan->fill_ms;
    return rc;
}
GX_GUARD_END

int gx_band_score(gx_band *b, int64_t *score, int *valid) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!b || !score || !valid) return GX_ERR_ARG;
    *valid = (b->last == b->n_bands) ? 1 : 0;
    *score = 0;
    if (!*valid) return GX_OK;
    if (b->trivial) {   // algo.rs:195-220: only boundary cells exist
        const uint64_t len = b->m + b->n_total;
        *score = len ? (int64_t)b->sc.h + (int64_t)len * b->sc.g : 0;
        return GX_OK;
    }
    if (!b->plan->executed) return GX_ERR_ARG;
    const int nl = b->last - b->first;
    std::vector<int64_t> sc(nl);
    int rc = gx_plan_fetch_scores(b->plan, sc.data());
    if (rc) return rc;
    *score = sc[nl - 1];
    return GX_OK;
}
GX_GUARD_END

double gx_band_stat(const gx_band *b, int what) {
    if (!b) return -1.0;
    if (what == 16) return (double)b->epoch;
    if (!b->plan) return what == 3 ? (double)((b->m + 1) * (b->n_total + 1)) : 0.0;
    return gx_plan_stat(b->plan, what);
}

void gx_band_destroy(gx_band *b) {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    band_free(b);
}

// The band object of the last gx_nw_score_banded call is kept (geometry, tile lists, device buffers): a caller that
// scores a stream of equally shaped pairs pays for plan creation once.  Released by gx_shutdown or by a call with
// another shape; its device memory comes from the context's caching pool either way.
static gx_band *g_band_cache = nullptr;
static void band_cache_drop() {
    if (g_band_cache) band_free(g_band_cache);
    g_band_cache = nullptr;
}

int gx_nw_score_banded(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n, gx_scores sc, int n_bands, int64_t *score) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!score || (!s1 && m) || (!s2 && n)) return GX_ERR_ARG;
    gx_band *b = g_band_cache;
    const bool hit = b && b->m == m && b->n_total == n && b->n_bands == n_bands && b->first == 0 && b->last == n_bands &&
                     memcmp(&b->sc, &sc, sizeof sc) == 0 && !b->poisoned;
    if (!hit) {
        band_cache_drop();
        b = nullptr;
        int rc = gx_band_create(m, n, n_bands, 0, n_bands, sc, &b);
        if (rc) return rc;
        g_band_cache = b;
    }
    int valid = 0;
    int rc = gx_band_upload(b, s1, s2);
    if (!rc) rc = gx_band_execute(b);
    if (!rc) rc = gx_band_score(b, score, &valid);
    if (rc) band_cache_drop();
    return rc;
}
GX_GUARD_END

// ------------------------------------------------------------------------------------------------
// small-table visualiser support: display.rs:131-220 prints the path grid and the three score planes
int gx_debug_planes(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n, gx_scores sc, int is_local, int64_t *ins,
                    int64_t *del, int64_t *sub) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (!ins || !del || !sub || (!s1 && m) || (!s2 && n)) return GX_ERR_ARG;
    if (!g_ctx) return GX_ERR_NOT_INIT;
    if (!(m < 200 && n < 2000)) return GX_ERR_RANGE;     // display.rs:139: "Sequence table too large to visualize"
    int rc = check_scores_impl(sc, m, n, is_local != 0);
    if (rc) return rc;
    Ctx *c = g_ctx;
    CK(cudaSetDevice(c->device));
    const size_t cells = (size_t)(m + 1) * (n + 1);
    uint8_t *d_seq = nullptr;
    long long *d_planes = nullptr;
    rc = pool_alloc(c, m + n + 16, (void **)&d_seq);
    if (!rc) rc = pool_alloc(c, 3 * cells * 8, (void **)&d_planes);
    if (!rc) {
        cudaError_t e = cudaSuccess;
        if (m) e = cudaMemcpyAsync(d_seq, s1, m, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess && n) e = cudaMemcpyAsync(d_seq + m, s2, n, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) {
            PlanesParams pp;
            pp.s1 = d_seq;
            pp.s2 = d_seq + m;
            pp.m = (uint32_t)m;
            pp.n = (uint32_t)n;
            pp.a = sc.s_match;
            pp.b = sc.s_mismatch;
            pp.g = sc.g;
            pp.h = sc.h;
            pp.is_local = is_local ? 1 : 0;
            pp.pi = d_planes;
            pp.pd = d_planes + cells;
            pp.ps = d_planes + 2 * cells;
            gx_planes_kernel<<<1, 256, 0, c->stream>>>(pp);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(ins, d_planes, cells * 8, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(del, d_planes + cells, cells * 8, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(sub, d_planes + 2 * cells, cells * 8, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail_cuda(e, "gx_debug_planes");
    }
    pool_free(c, d_seq);
    pool_free(c, d_planes);
    return rc;
}
GX_GUARD_END

// The one-shot batch calls keep the plan of their previous call (geometry, tile order, device buffers): a caller that
// aligns a stream of equally shaped batches -- or bench.py's end-to-end loop -- pays for plan creation once (0.4 ms of the
// 19 ms of the 45-pair batch).  A call with other lengths / scores / flags replaces it; gx_shutdown releases it.
static gx_plan *g_plan_cache = nullptr;
static void plan_cache_drop() {
    if (g_plan_cache) gx_plan_destroy(g_plan_cache);
    g_plan_cache = nullptr;
}
static int cached_plan(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local, int flags, gx_plan **out) {
    gx_plan *pl = g_plan_cache;
    const Tunables now = read_tunables();
    if (pl && pl->n_pairs == n_pairs && pl->is_local == (is_local ? 1 : 0) && pl->flags == flags && memcmp(&pl->sc, &sc, sizeof sc) == 0 &&
        memcmp(&pl->tun, &now, sizeof now) == 0 && (n_pairs == 0 || (len1 && len2 && memcmp(pl->len1.data(), len1, n_pairs * 8) == 0 &&
                                                                     memcmp(pl->len2.data(), len2, n_pairs * 8) == 0))) {
        *out = pl;
        return GX_OK;
    }
    plan_cache_drop();
    int rc = gx_plan_create(len1, len2, n_pairs, sc, is_local, flags, &pl);
    if (rc) return rc;
    g_plan_cache = pl;
    *out = pl;
    return GX_OK;
}

int gx_align_batch(const uint8_t *seq_blob, uint64_t blob_len, const uint64_t *off1, const uint64_t *len1, const uint64_t *off2,
                   const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local, int flags, gx_result *out,
                   uint8_t *ops_blob, const uint64_t *ops_off) try {
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    gx_plan *pl = nullptr;
    int rc = cached_plan(len1, len2, n_pairs, sc, is_local, flags, &pl);
    if (rc) return rc;
    rc = gx_plan_upload(pl, seq_blob, blob_len, off1, off2);
    if (!rc) rc = gx_plan_execute(pl);
    if (!rc) rc = gx_plan_fetch(pl, out, ops_blob, ops_off);
    if (rc) plan_cache_drop();      // never keep a plan that failed
    return rc;
}
GX_GUARD_END

int gx_score_batch(const uint8_t *seq_blob, uint64_t blob_len, const uint64_t *off1, const uint64_t *len1, const uint64_t *off2,
                   const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local, int64_t *scores) try {
    if ((!seq_blob && blob_len) || ((!off1 || !len1 || !off2 || !len2 || !scores) && n_pairs)) return GX_ERR_ARG;
    // large read sets stream through two copy/compute lanes; everything else goes through a plan
    if (!getenv("GX_NO_STREAM")) {   // debug switch, read once per batch call
        const int rcs = score_batch_streamed(seq_blob, blob_len, off1, len1, off2, len2, n_pairs, sc, is_local, scores,
                                             nullptr, nullptr, getenv("GX_READS32") != nullptr);
        if (rcs != GX_ERR_UNSUPPORTED) return rcs;
    }
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    gx_plan *pl = nullptr;
    int rc = cached_plan(len1, len2, n_pairs, sc, is_local, 0, &pl);
    if (rc) return rc;
    rc = gx_plan_upload(pl, seq_blob, blob_len, off1, off2);
    if (!rc) rc = gx_plan_execute(pl);
    if (!rc) rc = gx_plan_fetch_scores(pl, scores);
    if (rc) plan_cache_drop();
    return rc;
}
GX_GUARD_END

int gx_score_batch_cells(const uint8_t *seq_blob, uint64_t blob_len, const uint64_t *off1, const uint64_t *len1,
                         const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs, gx_scores sc, int is_local,
                         int64_t *scores, uint64_t *start_i, uint64_t *start_j) try {
    if ((!seq_blob && blob_len) || ((!off1 || !len1 || !off2 || !len2 || !scores || !start_i || !start_j) && n_pairs))
        return GX_ERR_ARG;
    if (!getenv("GX_NO_STREAM")) {
        const int rcs = score_batch_streamed(seq_blob, blob_len, off1, len1, off2, len2, n_pairs, sc, is_local, scores,
                                             start_i, start_j, getenv("GX_READS32") != nullptr);
        if (rcs != GX_ERR_UNSUPPORTED) return rcs;
    }
    // everything the streamed path declines: a plan with start cells (read kernels when the batch qualifies, else the
    // wavefront fill and its start-cell reduction)
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    gx_plan *pl = nullptr;
    int rc = cached_plan(len1, len2, n_pairs, sc, is_local, GX_FLAG_START_CELL, &pl);
    if (rc) return rc;
    std::vector<gx_result> res(n_pairs);
    rc = gx_plan_upload(pl, seq_blob, blob_len, off1, off2);
    if (!rc) rc = gx_plan_execute(pl);
    if (!rc) rc = gx_plan_fetch(pl, res.data(), nullptr, nullptr);
    if (rc) {
        plan_cache_drop();
        return rc;
    }
    for (uint64_t q = 0; q < n_pairs; ++q) {
        scores[q] = res[q].score;
        start_i[q] = res[q].start_i;
        start_j[q] = res[q].start_j;
    }
    return GX_OK;
}
GX_GUARD_END

int gx_align_pair(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n, gx_scores sc, int is_local, int flags,
                  gx_result *out, uint8_t *ops, uint64_t ops_cap) try {
    if (!out || (!s1 && m) || (!s2 && n)) return GX_ERR_ARG;
    if (m > (1ull << 28) || n > (1ull << 28)) return GX_ERR_RANGE;   // before anything is sized from the caller's numbers
    if ((flags & GX_FLAG_TRACEBACK) && (!ops || ops_cap < m + n + 1)) return (!ops) ? GX_ERR_ARG : GX_ERR_OPS_CAP;
    std::vector<uint8_t> blob(m + n);
    if (m) memcpy(blob.data(), s1, m);
    if (n) memcpy(blob.data() + m, s2, n);
    uint64_t off1 = 0, off2 = m, l1 = m, l2 = n;
    uint64_t ops_off[2] = {0, ops_cap};
    return gx_align_batch(blob.data(), m + n, &off1, &l1, &off2, &l2, 1, sc, is_local, flags, out, ops, ops_off);
}
GX_GUARD_END

}  // extern "C"
