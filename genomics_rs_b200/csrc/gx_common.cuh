// gx_common.cuh -- shared device/host definitions of libgxalign (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gx {

// "minus infinity" of the int32 cell state (SURVEY.md 3.4); the reference uses i64::MIN + |g+h| (algo.rs:166)
constexpr int NEG32 = -(1 << 30);

// Rows of one panel: a tile is (panel p, strip s) = PANEL_H rows x 32*K columns, owned by one warp.
constexpr int PANEL_H_LOG2 = 12;
constexpr int PANEL_H = 1 << PANEL_H_LOG2;
// The fill kernel has no CTA-level cooperation (per-warp shared memory, no __syncthreads), so the same code runs as
// 8-warp CTAs (2 per SM) or as single-warp CTAs (16 per SM).  Single-warp CTAs let the block scheduler spread a small
// number of busy warps over all SMs instead of packing the first tickets onto the few SMs whose CTAs started first;
// with every warp slot busy the 8-warp shape is a few per cent faster.  gx_api.cu picks the shape per plan.
constexpr int WARPS_PER_CTA = 8;
constexpr int CTA_THREADS = WARPS_PER_CTA * 32;
// 8-warp CTAs per SM: 2 (16 warps, 128 registers per thread) for every K and every instance.  Tried: 3 CTAs (24 warps,
// 80 registers) for K <= 8 to have more warps covering the ones that wait for their left neighbour -- slower everywhere
// (corona45 K=8 18.2 -> 20.9 ms, 1 Mbp x 1 Mbp 322 -> 373 ms): the register cap costs more than the occupancy gives.
constexpr int CTAS_PER_SM = 2;
constexpr int WARPS_PER_SM = WARPS_PER_CTA * CTAS_PER_SM;

// per-warp shared memory: s1 panel segment (+32: 16 B alignment slack in front, 16 B over-read behind),
// the left-boundary in-ring and right-boundary out-ring (2 x 32 rows x 8 B each) and one mbarrier.
constexpr int WARP_SMEM_S1 = PANEL_H + 32;
constexpr int WARP_SMEM_BYTES = WARP_SMEM_S1 + 512 + 512 + 16;

// Checked build (-DGX_CHECKED, `GX_BUILD_TAG=chk`): every shared-memory ring / staging index, code-chunk offset,
// boundary-buffer row and op index the kernels form is range-checked on the device; a violation records its site number
// in the plan's control block (word 2) and the execute returns GX_ERR_INTERNAL naming it.  compute-sanitizer is closed on
// the B200 pool this was developed on; the GPU test-suite is run against this build instead (tools/gpu_checked.sh).
#ifdef GX_CHECKED
#define GX_CHECK(word, cond, site)                                   \
    do {                                                             \
        if (!(cond)) atomicMax(reinterpret_cast<unsigned int *>(word), (unsigned int)(site)); \
    } while (0)
#else
#define GX_CHECK(word, cond, site) ((void)0)
#endif

struct PairDesc {
    uint64_t s1_off, s2_off;   // byte offsets of the two sequences in the device blob
    uint64_t colbuf_off;       // u64 entries: strip s (< S-1) right boundary column, row i (1..m) at colbuf_off + s*m + (i-1)
    uint64_t top_off;          // int2 entries: column j (1..n) at top_off + (j-1): (E,D) of the last finished panel row
    uint64_t codes_off;        // bytes: tile (p,s) at codes_off + (p*S+s)*tile_code_bytes
    uint64_t ops_off;          // bytes in the device ops blob
    uint32_t m, n;
    uint32_t S, P;             // strips, panels
    uint32_t progress_off;     // u32 entries: progress[s] = panels finished by strip s
    uint32_t tile_base;        // tile_best index of tile (0,0); tile (p,s) at tile_base + p*S + s
    uint32_t tile_code_bytes;
    uint32_t col0;             // column band (config 5): this "pair" is columns col0+1 .. col0+n of a wider table
    // band links: strip 0 takes its left boundary from `inbox` (rows 1..m at [i-1]) instead of the column-0
    // formula; the last strip publishes its right boundary to `outbox`, which may be peer-GPU memory (NVLink).
    const unsigned long long *inbox;
    unsigned long long *outbox;
    // flow control of a remote outbox: the consumer stores the number of executes it has finished here (our memory);
    // execute e may overwrite the consumer's inbox only once *ack >= e-1.  Null when the outbox is local or absent.
    const uint32_t *ack;
};

// Code band (global traceback plans, and local ones with compact storage): direction codes are only WRITTEN by tiles
// within `code_w` columns of a line from (a0,b0) to the path's end cell (a1,b1) -- for a global alignment the table's
// scaled diagonal (0,0)-(m,n); for a local one the slope-1 line back from its start cell (i*,j*) to the table's edge,
// (i*-d, j*-d) with d = min(i*,j*), found by a score-only pass first.  Above row a0 the line's column is b0; tiles
// that start at or beyond the end cell are out (the path moves only up and left from it); tile (0,0) is always in.
// Every other tile runs the score-only cell (5 instead of 9 instructions).  One flag byte per tile (FillParams / WalkParams::tile_codes, indexed like tile_best;
// null = every tile has codes), written by the host, read by the fill (which variant to run) and by the walk, which
// verifies that every tile it enters has codes; if a path ever leaves the band the execute is repeated (gx_plan_execute),
// so results stay exact: with codes everywhere, or -- compact storage -- with a wider band for the pairs that left it.
// Compact storage (pairs whose codes would not fit the device for every tile): only in-band tiles have memory for codes.
// A slot table (FillParams / WalkParams::tile_slot, indexed like tile_best) maps tile (p,s) to its slot, its codes are at
// codes_off + slot * tile_code_bytes; an out-of-band tile maps to slot 0 of its pair (tile (0,0) is always in the band),
// so that every address the kernels form lies inside the codes buffer although nothing is read or written there.
__host__ inline bool tile_in_code_band(uint64_t a0, uint64_t b0, uint64_t a1, uint64_t b1, uint64_t m, uint32_t p, uint32_t s,
                                       uint32_t W, uint64_t code_w) {
    const uint64_t i0 = (uint64_t)p << PANEL_H_LOG2;
    const uint64_t i1 = (i0 + PANEL_H < m) ? i0 + PANEL_H : m;
    const uint64_t c0 = (uint64_t)s * W, c1 = c0 + W;   // the tile's columns [c0, c1)
    if (p == 0 && s == 0) return true;
    if (i0 >= a1 || c0 >= b1) return false;
    auto col = [&](uint64_t i) { return (i <= a0 || a1 == a0) ? b0 : b0 + (i - a0) * (b1 - b0) / (a1 - a0); };
    const uint64_t lo = col(i0), hi = col(i1);          // the line's columns at the tile's first / last row
    return c1 + code_w > lo && c0 < hi + code_w + 1;
}

struct TileDesc {
    uint32_t pair, p, s, pad_;
};

// device copy of gx_result (include/gxalign.h) -- identical layout, checked by static_assert in gx_api.cu
struct DevResult {
    long long score;
    unsigned long long start_i, start_j, end_i, end_j, n_ops, matches, mismatches, gap_extensions, opening_gaps, lcs_at_first_max;
    double fill_ms, walk_ms;
};

struct FillParams {
    const uint8_t *blob;
    const uint8_t *blob_sym;         // blob re-encoded to shift amounts 8*symbol (one-hot / IDP.4A path), else null
    uint32_t one;                    // the constant 1, opaque to ptxas (keeps code-bit IMADs on the FMA pipe)
    const PairDesc *pairs;
    const TileDesc *tiles;
    uint32_t n_pairs;                // pairs in `pairs` (checked build)
    uint32_t n_tiles;
    uint32_t pmax;                   // resident-strips mode: tiles are laid out [strip][panel] with pmax entries per strip; else 0
    uint32_t parity;                 // LL parity bit of this execute (SURVEY "boundary hand-off")
    uint32_t cpb;                    // code chunks per hand-off batch (batch = cpb * SPC steps <= 32 rows)
    uint32_t epoch;                  // 1-based execute number of a band plan (see PairDesc::ack), else 0
    uint32_t *ticket;
    uint32_t *progress;
    unsigned long long *colbuf;
    int2 *top;
    uint8_t *codes;
    const uint8_t *tile_codes;       // code band: one flag per tile (1 = this tile writes codes), or null (all do)
    uint64_t code_bytes;             // size of `codes` (checked build)
    int4 *tile_best;
    uint32_t pad_keys;               // 1: padded columns of a pair's last strip could reach the maximum (s_mismatch >= 0): mask their keys
    int g, hg, ap, bp, h;            // ap = s_match - (h+g), bp = s_mismatch - (h+g): S is formed in E-space (E = V + h + g)
    const uint32_t *tile_slot;       // compact code storage: slot of each tile's codes (code band, above), or null (dense)
};

struct WalkParams {
    const uint8_t *blob;
    const PairDesc *pairs;
    uint32_t n_pairs;
    const int2 *top;
    const uint8_t *codes;
    const int4 *tile_best;
    DevResult *results;
    uint8_t *ops;
    int g, hg, h;
    int is_local, traceback, have_best;
    uint32_t *left_band;             // control block word 3: walks that needed a tile outside the code band
    const uint8_t *tile_codes;       // code band: one flag per tile, or null (every tile has codes)
    uint32_t *check;                 // checked build: where a failed bounds check records its site (control block word 2)
    uint64_t code_bytes, ops_bytes;  // sizes of the codes / ops buffers (checked build)
    uint32_t win_rows;               // rows of a code window of the walk (256 or 512)
    const uint32_t *tile_slot;       // compact code storage: slot of each tile's codes, or null (tile (p,s) at p*S+s)
    uint2 *left_cell;                // compact code storage: per pair, the cell whose tile was outside the band, or null
};

// ---------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t phase) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// system-scope variants: band hand-off between GPUs (peer memory over NVLink); data and flag share one word
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int2 ld_cg_int2(const int2 *p) {
    int2 v;
    asm volatile("ld.global.cg.v2.s32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_cg_int2(int2 *p, int2 v) {
    asm volatile("st.global.cg.v2.s32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_cs_uint4(uint4 *p, uint4 v) {
    // streaming store: traceback codes are written once and read only along the path
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// shared-memory load the compiler may not move or merge (pins the issue point of a deliberately early load)
__device__ __forceinline__ uint2 lds_volatile_uint2(const uint2 *p) {
    uint2 v;
    asm volatile("ld.volatile.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(smem_u32(p)) : "memory");
    return v;
}

template <int N>
struct Log2 {
    static constexpr int value = 1 + Log2<N / 2>::value;
};
template <>
struct Log2<1> {
    static constexpr int value = 0;
};

}  // namespace gx
