// gx_reads.cuh -- K4: inter-task batch kernel for many short pairs (score, and on request the local start cell).
//
// Same recurrences as gx_fill.cuh (reference: /root/reference/src/alignment/algo.rs:191-268), but the
// unit of parallelism is the PAIR: a group of G lanes owns one pair, each lane K register-blocked
// columns (G*K >= n), rows flow through the group as a systolic skew with two shuffles per step.
// No shared memory, no inter-warp traffic, no traceback storage.
//
// Local mode needs no masking at all: rows above/below the table and columns right of it are fed a
// never-matching character, which (for s_mismatch < 0) makes every such cell strictly smaller than a
// real cell it derives from, so the running maximum is unaffected.  Global mode freezes a lane's
// state outside rows 0..m-1 (two selects per cell) and reads E[m][n] from the lane that owns column n.
//
// TRACK (local only): also the start cell, the last cell in row-major order that attains the table maximum
// (algo.rs:306-323), (m, n) when that maximum is 0.  By the argument above no cell outside the table can tie a
// positive maximum, so only the zero rule needs handling.  Output: one uint32 per pair, i << 16 | j.
#pragma once
#include <cstdlib>

#include "gx_common.cuh"

namespace gx {

constexpr int READS_MAX_LEN = 640;

struct ReadsParams;

struct ReadsParams {
    const uint8_t *blob;
    const uint64_t *off1, *off2;
    const uint32_t *len1, *len2;       // lengths as 32-bit words (plans), or null:
    const uint4 *rec;                  // streamed chunks: one 16-byte record per pair {off1, off2, len1, len2} relative to
                                       // `blob` (packed by the host while it validates the chunk); overrides off*/len*
    uint32_t n_pairs;
    int *scores;
    DevResult *results;   // may be null
    int a, b, g, h, is_local;
    uint32_t *cells;      // local start cells (i << 16 | j), or null: score only
};

// start cell of a local pair from its best (V, i, j): the zero rule of gx_walk.cuh applies to an empty table too
__device__ __forceinline__ uint32_t reads_cell(int v, uint32_t i, uint32_t j, int m, int n) {
    return (v <= 0 || m == 0 || n == 0) ? ((uint32_t)m << 16 | (uint32_t)n) : (i << 16 | j);
}

// geometry of pair q: sequence pointers and lengths (have == false: an empty pair at the blob's start)
__device__ __forceinline__ void reads_pair(const ReadsParams &P, uint64_t q, bool have, const uint8_t *&s1, const uint8_t *&s2, int &m,
                                           int &n) {
    if (P.rec) {
        const uint4 r = have ? __ldg(P.rec + q) : make_uint4(0u, 0u, 0u, 0u);
        s1 = P.blob + r.x;
        s2 = P.blob + r.y;
        m = (int)r.z;
        n = (int)r.w;
    } else {
        s1 = P.blob + (have ? P.off1[q] : 0);
        s2 = P.blob + (have ? P.off2[q] : 0);
        m = have ? (int)P.len1[q] : 0;
        n = have ? (int)P.len2[q] : 0;
    }
}

template <int G, int K, bool LOCAL, bool TRACK>
__global__ void __launch_bounds__(256) gx_reads_kernel(const ReadsParams P) {
    static_assert(!TRACK || (LOCAL && K <= 32), "start cells: local only, column index in 5 bits");
    constexpr unsigned FULLM = 0xffffffffu;
    constexpr int GPW = 32 / G;  // groups per warp
    const int lane = threadIdx.x & 31;
    const int lg = lane % G;     // lane in group
    const int gw = lane / G;     // group in warp
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const int g = P.g, hg = P.h + P.g, h = P.h;
    const int ap = P.a - hg, bp = P.b - hg;

    for (uint64_t base = (uint64_t)warp_global * GPW; base < P.n_pairs; base += (uint64_t)n_warps * GPW) {
        const uint64_t q = base + gw;
        const bool have = q < P.n_pairs;
        int m, n;
        const uint8_t *s1, *s2;
        reads_pair(P, q, have, s1, s2, m, n);
        const int jl = lg * K;
        int c2[K], eu[K], du[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            c2[k] = (jl + k < n) ? (int)__ldg(s2 + jl + k) : 256;
            eu[k] = (LOCAL ? 0 : h + (jl + k + 1) * g) + hg;
            du[k] = NEG32;
        }
        int vd = ((jl == 0) ? 0 : (LOCAL ? 0 : h + jl * g)) + hg;  // E of (row 0, column jl)
        // every lane of the group must finish row m-1; the warp runs the longest group's step count
        const int lstar = (n > 0) ? (n - 1) / K : 0;
        int steps = (m > 0 && n > 0) ? m + G - 1 : 0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) steps = max(steps, __shfl_xor_sync(FULLM, steps, off));

        // local: lanes that have not reached row 0 yet must see "V = 0, I = 0" from their left neighbour
        int elast = LOCAL ? hg : 0, ilast = 0, best = 0;
        int brow = 0;   // TRACK: best holds the key (V << 5) | k of the lane's best cell, brow its row
        int c1n = (m > 0 && lg == 0) ? (int)__ldg(s1) : -1;
        for (int t = 0; t < steps; ++t) {
            const int r = t - lg;
            const int c1 = c1n;
            {   // prefetch next row's character (address independent of the DP state)
                const int rn = r + 1;
                c1n = (rn >= 0 && rn < m) ? (int)__ldg(s1 + rn) : -1;
            }
            int el = __shfl_up_sync(FULLM, elast, 1);
            int il = __shfl_up_sync(FULLM, ilast, 1);
            if (lg == 0) {
                el = (LOCAL ? 0 : h + (r + 1) * g) + hg;  // column 0: V = delete_score (algo.rs:204-211)
                il = NEG32;
            }
            const bool active = LOCAL ? true : (r >= 0 && r < m);  // global: state is frozen outside rows 0..m-1
            int e = el, irun = il, ed = vd;
            int rkey = 0;   // TRACK: largest (V << 5) | k of this row: the last column that attains the row's maximum
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int In = LOCAL ? __viaddmax_s32_relu(irun, g, e) : __viaddmax_s32(irun, g, e);
                const int Dn = LOCAL ? __viaddmax_s32_relu(du[k], g, eu[k]) : __viaddmax_s32(du[k], g, eu[k]);
                const int Sn = ed + ((c1 == c2[k]) ? ap : bp);
                const int Vn = LOCAL ? __vimax3_s32_relu(In, Dn, Sn) : __vimax3_s32(In, Dn, Sn);
                ed = eu[k];
                const int En = Vn + hg;
                if (LOCAL) {
                    eu[k] = En;
                    du[k] = Dn;
                    // The key cannot wrap: the score contract (check_scores_impl) refuses every local scoring with
                    // min(m, n) * max(s_match, 0) >= 2^26, so 0 <= V < 2^26 and (V << 5) | 31 < 2^31.
                    if (TRACK) rkey = max(rkey, Vn * 32 + k);
                    else best = max(best, Vn);
                } else {
                    eu[k] = active ? En : eu[k];
                    du[k] = active ? Dn : du[k];
                }
                e = En;
                irun = In;
            }
            vd = active ? el : vd;
            elast = e;
            ilast = irun;
            if (TRACK && rkey >= (best & ~31)) {   // V of the row >= the lane's best V: later rows win ties
                best = rkey;
                brow = r;
            }
        }
        int score;
        if (TRACK) {
            // (V, i, j) of the group's best cell: the largest 64-bit key V << 32 | i << 16 | j.  A cell outside the table
            // (r < 0, r >= m or column >= n) may be a lane's best but never ties a positive table maximum, so it can
            // only win the reduction when that maximum is 0, which the zero rule replaces.
            unsigned long long key = (unsigned long long)(best >> 5) << 32 |
                                     ((uint32_t)(brow + 1) & 0xffffu) << 16 | (uint32_t)(jl + (best & 31) + 1);
#pragma unroll
            for (int off = G / 2; off > 0; off >>= 1) key = max(key, __shfl_xor_sync(FULLM, key, off));
            score = (m == 0 || n == 0) ? 0 : (int)(key >> 32);
            if (have && lg == 0) P.cells[q] = reads_cell(score, (uint32_t)key >> 16, (uint32_t)key & 0xffffu, m, n);
        } else if (LOCAL) {
            score = best;
#pragma unroll
            for (int off = G / 2; off > 0; off >>= 1) score = max(score, __shfl_xor_sync(FULLM, score, off));
            if (m == 0 || n == 0) score = 0;
        } else {
            // the owner of column n holds E[m][n] in eu[(n-1)%K] (frozen after row m-1)
            int v = 0;
            const int kk = (n > 0) ? (n - 1) % K : 0;
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (k == kk) v = eu[k];
            v = __shfl_sync(FULLM, v, gw * G + lstar);
            score = v - hg;
            if (m == 0 && n == 0) score = 0;
            else if (m == 0) score = h + n * g;
            else if (n == 0) score = h + m * g;
        }
        if (have && lg == 0) {
            P.scores[q] = score;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// s16x2 variant (local, score only): TWO pairs per lane group, one in each 16-bit half of every register.
// Frame: V is kept as is (>= 0); I and D are carried unclamped and biased by beta = -(h+g) > 0
// (Ihat = I + beta, Dhat = D + beta -- clamping I and D at 0 does not change V, see DESIGN.md), so that
//     Ihat' = max(Ihat + g, V_left)           one VIADDMNMX.S16x2, no separate "V + h + g"
//     Dhat' = max(Dhat + g, V_up)             one VIADDMNMX.S16x2
//     Shat  = V_diag + (eq ? a : b) + beta    plain 32-bit add: both halves non-negative, no borrow
//     Vhat  = max3(Ihat', Dhat', Shat)        one VIMNMX3.S16x2
//     V     = max(Vhat - beta, 0)             one VIADDMNMX.S16x2.RELU
// match/mismatch: x = c1 ^ c2 (halves 0 iff equal), ne = min_u16x2(x, 1), sub = (a+beta) - ne*(a-b)  (IMAD).
// Needs s_mismatch < 0, s_mismatch + beta >= 0 and min(m,n)*s_match + beta < 2^15 (host checks).
//
// TRACK: no (V, k) key fits a 16-bit half, so the running maximum becomes a per-row maximum; once per step each half
// compares it with the lane's best (Vhat frame: for V > 0, Vhat = V + beta, so ties on Vhat are ties on V), and only on
// steps where some lane of the warp improves does it search its K columns for the last one that attains the row maximum.
template <int G, int K, bool TRACK>
__global__ void __launch_bounds__(256, 2) gx_reads16_kernel(const ReadsParams P) {
    constexpr unsigned FULLM = 0xffffffffu;
    constexpr int GPW = 32 / G;  // groups per warp; each group aligns 2 pairs
    const int lane = threadIdx.x & 31;
    const int lg = lane % G;
    const int gw = lane / G;
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const int beta = -(P.h + P.g);
    const uint32_t g2 = ((uint32_t)(P.g & 0xffff)) * 0x00010001u;
    const uint32_t hg2 = ((uint32_t)((P.h + P.g) & 0xffff)) * 0x00010001u;
    const uint32_t ap2 = ((uint32_t)(P.a + beta)) * 0x00010001u;      // match + beta, both halves (>= 0)
    const int negd = -(P.a - P.b);                                    // sub = ap2 + ne * negd  (halves stay >= 0)
    const uint32_t ninf2 = ((uint32_t)((-16000) & 0xffff)) * 0x00010001u;
    const uint64_t n_dual = ((uint64_t)P.n_pairs + 1) / 2;

    for (uint64_t base = (uint64_t)warp_global * GPW; base < n_dual; base += (uint64_t)n_warps * GPW) {
        const uint64_t dq = base + gw;
        const uint64_t qa = 2 * dq, qb = 2 * dq + 1;
        const bool ha = dq < n_dual && qa < P.n_pairs, hb = dq < n_dual && qb < P.n_pairs;
        int ma, na, mb, nb;
        const uint8_t *s1a, *s2a, *s1b, *s2b;
        reads_pair(P, qa, ha, s1a, s2a, ma, na);
        reads_pair(P, qb, hb, s1b, s2b, mb, nb);
        const int jl = lg * K;
        uint32_t c2[K], vu[K], du[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t ca = (jl + k < na) ? (uint32_t)__ldg(s2a + jl + k) : 0x200u;   // padding never matches
            const uint32_t cb = (jl + k < nb) ? (uint32_t)__ldg(s2b + jl + k) : 0x200u;
            c2[k] = ca | (cb << 16);
            vu[k] = 0u;        // V of row 0
            du[k] = ninf2;     // Dhat of row 0
        }
        uint32_t vd = 0u;      // V of (row 0, column jl)
        const int mm = max(ma, mb);
        int steps = (mm > 0) ? mm + G - 1 : 0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) steps = max(steps, __shfl_xor_sync(FULLM, steps, off));

        uint32_t vlast = 0u, ilast = 0u, best = 0u;
        uint32_t brow = 0u, bcol = 0u;   // TRACK, per half: row + 1 and k + 1 of the lane's best cell
        auto row_chars = [&](int r) -> uint32_t {
            const uint32_t ca = (r >= 0 && r < ma) ? (uint32_t)__ldg(s1a + r) : 0x100u;
            const uint32_t cb = (r >= 0 && r < mb) ? (uint32_t)__ldg(s1b + r) : 0x100u;
            return ca | (cb << 16);
        };
        uint32_t c1n = row_chars(-lg);
        for (int t = 0; t < steps; ++t) {
            const uint32_t c1 = c1n;
            c1n = row_chars(t + 1 - lg);   // prefetch: independent of the DP state
            uint32_t vl = __shfl_up_sync(FULLM, vlast, 1);
            uint32_t il = __shfl_up_sync(FULLM, ilast, 1);
            if (lg == 0) {
                vl = 0u;         // column 0: V = 0
                il = ninf2;      // I = -inf
            }
            uint32_t v = vl, irun = il, dg = vd;
            uint32_t rmax = 0u;   // TRACK: Vhat maximum of the row
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint32_t ne = __vminu2(c1 ^ c2[k], 0x00010001u);
                const uint32_t sub = ap2 + ne * (uint32_t)negd;
                const uint32_t In = __viaddmax_s16x2(irun, g2, v);
                const uint32_t Dn = __viaddmax_s16x2(du[k], g2, vu[k]);
                const uint32_t Sn = dg + sub;
                const uint32_t Vh = __vimax3_s16x2(In, Dn, Sn);
                const uint32_t Vn = __viaddmax_s16x2_relu(Vh, hg2, 0u);
                if (TRACK) rmax = (k == 0) ? Vh : __vmaxs2(rmax, Vh);
                else best = __vmaxs2(best, Vh);
                dg = vu[k];
                vu[k] = Vn;
                du[k] = Dn;
                v = Vn;
                irun = In;
            }
            vd = vl;
            vlast = v;
            ilast = irun;
            if (TRACK) {
                const uint32_t ge = __vcmpges2(rmax, best);   // 0xffff in the halves whose row reaches the lane's best
                if (__any_sync(FULLM, ge != 0u)) {
                    // last column of the row whose V equals the row maximum: d = rmaxV - V >= 0 in both halves (no
                    // borrow), ne = 0 where equal; the largest (1 - ne) * (k + 1) is the last such k, plus one
                    const uint32_t rv = __viaddmax_s16x2_relu(rmax, hg2, 0u);
                    uint32_t col = 0u;
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        const uint32_t ne = __vminu2(rv - vu[k], 0x00010001u);
                        col = __vmaxu2(col, (uint32_t)(k + 1) * 0x00010001u - ne * (uint32_t)(k + 1));
                    }
                    const uint32_t row2 = ((uint32_t)(t - lg + 1) & 0xffffu) * 0x00010001u;
                    best = (rmax & ge) | (best & ~ge);
                    bcol = (col & ge) | (bcol & ~ge);
                    brow = (row2 & ge) | (brow & ~ge);
                }
            }
        }
        if constexpr (TRACK) {
            // per half, the group's best (Vhat, i, j) as one 64-bit key (Vhat biased to unsigned); cells outside a
            // pair's table never tie its positive maximum, and a maximum of 0 takes the zero rule (see gx_reads_kernel)
            auto half_key = [&](int sh) -> unsigned long long {
                const uint32_t vh = (uint32_t)((int)(short)(best >> sh) + 32768);
                const uint32_t j = (uint32_t)jl + ((bcol >> sh) & 0xffffu);
                return (unsigned long long)vh << 32 | ((brow >> sh) & 0xffffu) << 16 | j;
            };
            unsigned long long ka = half_key(0), kb = half_key(16);
#pragma unroll
            for (int off = G / 2; off > 0; off >>= 1) {
                ka = max(ka, __shfl_xor_sync(FULLM, ka, off));
                kb = max(kb, __shfl_xor_sync(FULLM, kb, off));
            }
            if (lg == 0) {
                const int va = max((int)(ka >> 32) - 32768 - beta, 0), vb = max((int)(kb >> 32) - 32768 - beta, 0);
                if (ha) {
                    P.scores[qa] = (ma == 0 || na == 0) ? 0 : va;
                    P.cells[qa] = reads_cell(va, (uint32_t)ka >> 16, (uint32_t)ka & 0xffffu, ma, na);
                }
                if (hb) {
                    P.scores[qb] = (mb == 0 || nb == 0) ? 0 : vb;
                    P.cells[qb] = reads_cell(vb, (uint32_t)kb >> 16, (uint32_t)kb & 0xffffu, mb, nb);
                }
            }
        } else {
#pragma unroll
            for (int off = G / 2; off > 0; off >>= 1) best = __vmaxs2(best, __shfl_xor_sync(FULLM, best, off));
            if (lg == 0) {
                const int sa = max((int)(short)(best & 0xffffu) - beta, 0);
                const int sb = max((int)(short)(best >> 16) - beta, 0);
                if (ha) P.scores[qa] = (ma == 0 || na == 0) ? 0 : sa;
                if (hb) P.scores[qb] = (mb == 0 || nb == 0) ? 0 : sb;
            }
        }
    }
}

template <int G, int K>
static int launch_reads16_gk(const ReadsParams &rp, int sm_count, cudaStream_t st) {
    const int threads = 256;
    const uint64_t duals_per_cta = (uint64_t)(threads / 32) * (32 / G);
    const uint64_t n_dual = ((uint64_t)rp.n_pairs + 1) / 2;
    uint64_t want = (n_dual + duals_per_cta - 1) / duals_per_cta;
    uint64_t cap = (uint64_t)sm_count * 8;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (rp.cells) gx_reads16_kernel<G, K, true><<<grid, threads, 0, st>>>(rp);
    else gx_reads16_kernel<G, K, false><<<grid, threads, 0, st>>>(rp);
    return 0;
}

// packed path usable?  (local only; every intermediate must fit a signed 16-bit half)
static bool reads16_ok(const ReadsParams &rp, int max_len) {
    if (!rp.is_local) return false;
    const int beta = -(rp.h + rp.g);
    if (rp.b >= 0 || rp.b + beta < 0 || rp.a < rp.b) return false;
    const long long vmax = (long long)max_len * (rp.a > 0 ? rp.a : 0) + beta + (rp.a > 0 ? rp.a : 0);
    if (vmax >= 16000 || -rp.g >= 8000 || beta >= 8000) return false;
    return true;
}

template <int G, int K>
static int launch_reads_gk(const ReadsParams &rp, int sm_count, cudaStream_t st) {
    const int threads = 256;
    const uint64_t groups_per_cta = (uint64_t)(threads / 32) * (32 / G);
    uint64_t want = (rp.n_pairs + groups_per_cta - 1) / groups_per_cta;
    uint64_t cap = (uint64_t)sm_count * 8;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (rp.is_local && rp.cells) gx_reads_kernel<G, K, true, true><<<grid, threads, 0, st>>>(rp);
    else if (rp.is_local) gx_reads_kernel<G, K, true, false><<<grid, threads, 0, st>>>(rp);
    else gx_reads_kernel<G, K, false, false><<<grid, threads, 0, st>>>(rp);
    return 0;
}

// returns -1 if max_len is not supported by this kernel family; *bits (if given) = lane width of the kernel launched.
// rp.cells != null (local only): the start-cell variants, which also write each pair's start cell there.
static int launch_reads(const ReadsParams &rp, int max_len, int sm_count, cudaStream_t st, bool force32 = false, int *bits = nullptr) {
    const bool s16 = reads16_ok(rp, max_len) && !force32 && max_len <= 32 * 20;
    if (bits) *bits = s16 ? 16 : 32;
    if (s16) {
        if (max_len <= 8 * 19) return launch_reads16_gk<8, 19>(rp, sm_count, st);
        if (max_len <= 16 * 20) return launch_reads16_gk<16, 20>(rp, sm_count, st);
        return launch_reads16_gk<32, 20>(rp, sm_count, st);
    }
    if (max_len <= 8 * 19) return launch_reads_gk<8, 19>(rp, sm_count, st);
    if (max_len <= 16 * 20) return launch_reads_gk<16, 20>(rp, sm_count, st);
    if (max_len <= 32 * 20) return launch_reads_gk<32, 20>(rp, sm_count, st);
    return -1;
}

}  // namespace gx
