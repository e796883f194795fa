// gx_fill.cuh -- K1/K2: anti-diagonal wavefront fill of the affine-gap S/D/I tables.
//
// Replaces the CPU fill of /root/reference/src/alignment/algo.rs:191-268 (alignment_table).
// Per cell the reference keeps six 8-byte lanes (algo.rs:25-35); here the state is E = V + (h+g)
// and D per column in registers (SURVEY.md 3.4), I runs along the row inside the thread, and the
// only thing written per cell is a 2-bit direction code (0 S, 1 I, 2 D -- the order retrace()
// tests them in, algo.rs:351-400).
//
// Decomposition
//   tile  = (panel p, strip s) of one pair: PANEL_H rows x (32*K) columns, owned by ONE WARP.
//   lane  = K consecutive columns, register-blocked; the 32 lanes run a systolic skew:
//           at step t lane l updates row t-l, so lane l needs from lane l-1 exactly the
//           (E,I) that lane l-1 produced one step earlier -> two __shfl_up per step.
//   strip -> strip hand-off (right boundary column, 8 B per row) goes through an L2-resident
//           buffer with an LL-style protocol: one 64-bit store carries E, I and a parity bit of
//           the current execute, the consumer polls the data itself, no flag, no fence.  Rows are
//           published and consumed in batches of 8 so that a strip trails its left neighbour by
//           ~50 steps only (pipeline ramp of a pair = strips x lag).
//   panel -> panel hand-off (bottom row of a tile, (E,D) per column) goes through `top` with a
//           release/acquire counter per strip (once per 4096 rows).
//   tiles are taken from a global ticket counter in an order in which every dependency has a
//   smaller ticket, so a waiting warp only ever waits for a warp that is already resident.
//   s1 (the row sequence) is staged per tile into shared memory by a 1-D TMA bulk copy
//   (cp.async.bulk + mbarrier); s2 enters either as K characters in registers (compare path) or,
//   when the batch uses at most 4 distinct symbols, as a per-warp match/mismatch profile in shared
//   memory (PROF): two conflict-free LDS.128 per row replace 2 ALU instructions per cell.
//
// Pipe budget per cell (PROF, what the SASS shows):
//   score only   ALU: VIADDMNMX (I), VIADDMNMX (D), VIMNMX3 (V)      FMA pipe: IMAD.IADD (S), IMAD.IADD (E)
//   with codes   + ALU: 2x ISETP                                      + FMA pipe: 2x predicated IMAD (code bits)
// The contractual roofline of bench.py counts 7 / 8 / 13 INT32 ops per cell (SURVEY.md 8d).
#pragma once
#include <type_traits>

#include "gx_common.cuh"

namespace gx {

constexpr unsigned FULL = 0xffffffffu;
// A dependency wait that lasts longer than this many polls (>= ~1 s) is a bug or a lost device: raise the
// abort word instead of hanging the GPU; every waiter also leaves as soon as it sees the word set.
constexpr uint32_t SPIN_LIMIT = 1u << 22;

__device__ __forceinline__ bool spin_check(uint32_t &spins, uint32_t *abort_word) {
    if (++spins > SPIN_LIMIT) atomicExch(abort_word, 1u);
    if ((spins & 63u) == 0u || spins > SPIN_LIMIT) {
        if (*reinterpret_cast<volatile uint32_t *>(abort_word) != 0u) return true;
    }
    return false;
}

template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

// code bits of one cell added to a 32-bit code word: += UNIT if S != V, += UNIT again if also I != V.
// Two ISETP on the ALU pipe, two predicated IMAD on the FMA pipe (`one` is an opaque register holding 1,
// so ptxas cannot turn the IMADs back into ALU-pipe adds).
template <uint32_t UNIT>
__device__ __forceinline__ void code_acc(uint32_t &cw, int S, int I, int V, uint32_t one) {
    asm("{\n\t.reg .pred p1, p2;\n\t"
        "setp.ne.s32 p1, %1, %3;\n\t"
        "setp.ne.and.s32 p2, %2, %3, p1;\n\t"
        "@p1 mad.lo.u32 %0, %4, %5, %0;\n\t"
        "@p2 mad.lo.u32 %0, %4, %5, %0;\n\t}"
        : "+r"(cw)
        : "r"(S), "r"(I), "r"(V), "r"(one), "n"(UNIT));
}

// geometry shared by fill, walk and host.  A lane owns K consecutive columns and works on one row per step; the 32 lanes
// of a warp run a systolic skew: at step t lane l updates row t-l.  Steps are unrolled one 16-byte code chunk at a time
// (SPC steps = 64 cells per lane).  The boundary hand-off between strips works in batches of `cpb` chunks = cpb*SPC steps,
// a RUN-TIME parameter of the plan (FillParams::cpb, 1..CPB_MAX): the per-batch glue (publish the right boundary, settle
// the left one, two warp syncs) costs ~170 instructions, which 8 steps of K = 8 columns cannot amortise (2.7 instructions
// per cell), while a strip trails its left neighbour by 31 + batch steps (profiles/r2e_sweep_batch_*.jsonl: 1 Mbp x 1 Mbp
// 322 -> 282 ms, 45 coronavirus pairs 17.9 -> 16.7 ms at 32 steps; one BRCA2 pair 1.0 -> 1.4 ms).  At most 32 rows per
// batch: one boundary row per lane.
template <int K>
struct Geo {
    static_assert(K >= 2 && K <= 64 && (K & (K - 1)) == 0, "K cells must fit one 16-byte code chunk");
    static constexpr int W = 32 * K;                       // columns per strip
    static constexpr int SPC = 64 / K;                     // steps per 16-byte code chunk
    static constexpr int CPB_MAX = K / 2;                  // chunks per batch: at most 32 rows per batch
    static constexpr int KB = Log2<K>::value;
};
// batches of one tile: its rows + 31 steps of skew, in batches of `batch` steps
__host__ __device__ __forceinline__ uint32_t tile_batches(uint32_t rows, uint32_t batch) {
    return (rows + 31 + batch - 1) / batch;
}

// lane 0's left boundary comes from the in-ring, every other lane's from its left neighbour's registers: a predicated
// shared-memory load over the shuffle results instead of LDS + 2 SEL (the selects would sit on the ALU pipe, 2/K per
// cell; ptxas turns this into a predicated LDS.64 + two predicated moves on the FMA pipe -- two scalar loads were tried
// and still get the moves, because SHFL writes its destination late).
__device__ __forceinline__ void lds_over_if(int &x, int &y, const uint2 *p, bool pred) {
    // (no memory clobber: the load depends on this step's shuffle results, which pins it behind the __syncwarp that
    // published the in-ring; a clobber would serialise it against every other shared-memory access of the step)
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q ld.shared.v2.u32 {%0,%1}, [%2];\n\t}"
                 : "+r"(x), "+r"(y)
                 : "r"(smem_u32(p)), "r"((uint32_t)pred));
}

// One batch of BATCH systolic steps of one warp.
// THRU (last strip of a column band whose width is not a multiple of the strip): padding columns pass (E,I) of
// the band's last real column through unchanged, so that lane 31 still publishes the band's right boundary.
//
// CHAIN1 selects the latency-optimised form of the recurrence.  The classic form has a 3-instruction dependency
// per cell along the row (I -> V -> E -> next I, 14 clk); CHAIN1 keeps everything in E-space (x + h + g) and takes
// max(D,S) out of the chain:
//     Sh = Ediag + sub                (S + h + g: the profile holds the raw match/mismatch scores)
//     D' = max(D + g, Eup)            Mh = max(D' + (h+g), Sh)
//     I' = max(I + g, Mh_left)        the only op on the row chain: 1 VIADDMNMX = 4 clk per cell
//     E  = max(I' + (h+g), Mh)
// (I' = max(I+g, E_left) = max(I+g, I+h+g, Mh_left) and h <= 0.)  One more ALU-pipe op per cell than the classic
// form, a much shorter chain: chosen when there are too few strips to hide latency with warps.
//
// Match / mismatch score of a cell.  PROF (the batch uses at most 4 distinct symbols and the scores fit a byte): sequences
// are staged as SHIFT AMOUNTS 8*symbol, a row's character becomes the one-hot word 1 << c1 (one SHF per row), a column's
// four possible scores sit in the bytes of one register (prof4[k], built once per tile), and
//     S = E_diag + score  =  IDP.4A(onehot, prof4[k], E_diag)
// is ONE instruction on the FMA pipe -- the add it replaces -- with no profile in shared memory (round 1 fetched a
// profile row with K/4 LDS.128 + an address IMAD per step).  Otherwise: compare path (ISETP + SEL per cell).
// The s1 character of the NEXT step is fetched while this one runs (`c1a` carries it from step to step, batch to batch).
template <int K, bool LOCAL, bool CODES, int TRACK, bool PROF, bool MASKED, bool PAD, bool CHAIN1, bool THRU = false>
__device__ __forceinline__ void run_batch(int (&eu)[K], int (&du)[K], const int (&c2)[K], int &eo, int &io, int &vd,
                                          int &best, int &best_r, const int g, const int hg, const int ap, const int bp,
                                          const uint32_t one, const uint8_t *s1base /* s1 row 0 of this tile */,
                                          const int (&prof4)[K] /* PROF: byte s = score of symbol s against column k */,
                                          const uint2 *inr /* left-boundary (E,I) of this batch's rows */, uint2 *outring, uint4 *code_dst,
                                          const int t0, const int rows, const int lane, const int kvalid,
                                          int &c1a /* s1 character of the step about to run */, const int cpb /* chunks in this batch */,
                                          uint32_t *chk /* checked build: violation word */, const int s1lo, const int s1hi /* valid s1base indices */) {
    using G = Geo<K>;
    constexpr int KB = G::KB;
    const bool lane0 = lane == 0;
    // s1 character of tile row r; rows outside the tile are clamped only where they can occur (masked batches) --
    // an unmasked batch looks at most one byte past the tile's rows, which the staging buffer's slack covers
    auto s1char = [&](int r) __attribute__((always_inline)) -> int {
        if (MASKED) return (int)s1base[min(max(r, 0), rows - 1)];
        GX_CHECK(chk, r >= s1lo && r < s1hi, 11);
        return (int)s1base[r];
    };
#pragma unroll 1
    for (int ch = 0; ch < cpb; ++ch) {
        uint32_t cw[4] = {0u, 0u, 0u, 0u};
        // TRACK 2/3 (start cell / first maximum): the row maxima of this chunk's steps are kept in registers and folded into
        // (best, best_r) AFTER the chunk.  Updating per step put a compare + two selects on predicates between the cells of
        // consecutive steps and cost a lone strip 50 % (BRCA2 local fill 1.93 -> 1.30 ms, tools/mode_probe.py).
        int rbk[(TRACK == 2 || TRACK == 3) ? G::SPC : 1];
        static_for<G::SPC>([&](auto uc) {
            constexpr int uu = decltype(uc)::value;
            const int step = ch * G::SPC + uu;          // step inside the batch
            const int r0 = t0 + step - lane;            // row of this lane at this step
            // ---- left boundary of the row: neighbour lane's registers, lane 0: the in-ring
            int el = __shfl_up_sync(FULL, eo, 1);
            int il = __shfl_up_sync(FULL, io, 1);
            GX_CHECK(chk, step >= 0 && step < 32, 12);
            lds_over_if(el, il, inr + step, lane0);
            const bool act = MASKED ? ((r0 >= 0) && (r0 < rows)) : true;
            // ---- this step's s1 character (fetched one step ago); fetch the next step's
            const int c1 = PROF ? (int)(1u << c1a) : c1a;      // PROF: one-hot word of the symbol (shift amounts 0, 8, 16, 24)
            c1a = s1char(r0 + 1);
            // ---- the K cells of the row
            int e_ = el, i_ = il, ed_ = vd;
            int mh_ = el;   // CHAIN1: "max(D,S) of the cell to the left" -- for the lane's first column that is E_left itself
            int rowbest = (CHAIN1 || TRACK == 3) ? INT32_MIN : -1;
            static_for<K>([&](auto kc) {
                constexpr int k = decltype(kc)::value;
                int In, Dn, En, Skey, Ikey, Vkey;   // S/I/V keys: equal keys decide the direction code; Vkey orders the local maximum
                if (CHAIN1) {
                    In = LOCAL ? __viaddmax_s32_relu(i_, g, mh_) : __viaddmax_s32(i_, g, mh_);
                    Dn = LOCAL ? __viaddmax_s32_relu(du[k], g, eu[k]) : __viaddmax_s32(du[k], g, eu[k]);
                    const int Sh = PROF ? __dp4a(c1, prof4[k], ed_) : ed_ + ((c1 == c2[k]) ? ap : bp);
                    const int Mh = __viaddmax_s32(Dn, hg, Sh);
                    En = __viaddmax_s32(In, hg, Mh);   // local: I' >= 0 keeps E >= h+g, i.e. V >= 0
                    if (THRU) mh_ = (k < kvalid) ? Mh : mh_;
                    else mh_ = Mh;
                    Skey = Sh;
                    Ikey = CODES ? In + hg : 0;
                    Vkey = En;     // E-space: same order, same equalities
                } else {
                    In = LOCAL ? __viaddmax_s32_relu(i_, g, e_) : __viaddmax_s32(i_, g, e_);
                    Dn = LOCAL ? __viaddmax_s32_relu(du[k], g, eu[k]) : __viaddmax_s32(du[k], g, eu[k]);
                    const int Sn = PROF ? __dp4a(c1, prof4[k], ed_) : ed_ + ((c1 == c2[k]) ? ap : bp);
                    const int Vn = LOCAL ? __vimax3_s32_relu(In, Dn, Sn) : __vimax3_s32(In, Dn, Sn);
                    En = Vn + hg;
                    Skey = Sn;
                    Ikey = In;
                    Vkey = Vn;
                }
                if (CODES) {
                    constexpr int bitpos = (uu * K + k) * 2;
                    code_acc<(1u << (bitpos & 31))>(cw[bitpos >> 5], Skey, Ikey, Vkey, one);
                }
                ed_ = eu[k];
                if (MASKED) {
                    eu[k] = act ? En : eu[k];
                    du[k] = act ? Dn : du[k];
                } else {
                    eu[k] = En;
                    du[k] = Dn;
                }
                if (THRU) {
                    e_ = (k < kvalid) ? En : e_;
                    i_ = (k < kvalid) ? In : i_;
                } else {
                    e_ = En;
                    i_ = In;
                }
                if (TRACK == 2) {
                    int key = (Vkey << KB) | k;
                    if (PAD) key = (k < kvalid) ? key : (CHAIN1 ? INT32_MIN : -1);
                    rowbest = max(rowbest, key);
                } else if (TRACK == 1) {
                    int key = Vkey;
                    if (PAD) key = (k < kvalid) ? key : (CHAIN1 ? INT32_MIN : -1);
                    rowbest = max(rowbest, key);
                } else if (TRACK == 3) {
                    // first maximum in row-major order (alignment_table's max_cell, algo.rs:258-262, strict `<`):
                    // inside the row the key's low bits prefer the SMALLER column
                    int key = (Vkey << KB) | (K - 1 - k);
                    if (PAD) key = (k < kvalid) ? key : INT32_MIN;
                    rowbest = max(rowbest, key);
                }
            });
            if (MASKED) vd = act ? el : vd;
            else vd = el;
            eo = e_;
            io = i_;
            if (TRACK == 2 || TRACK == 3) {
                rbk[uu] = act ? rowbest : INT32_MIN;     // INT32_MIN: no row here
            } else if (TRACK == 1) {
                best = act ? max(best, rowbest) : best;
            }
            GX_CHECK(chk, step < 32, 13);
            if (lane == 31 && act) outring[step] = make_uint2((uint32_t)e_, (uint32_t)i_);   // row t0+step-31
        });
        if (TRACK == 2 || TRACK == 3) {
            // TRACK 2: the LAST maximum in row-major order wins (Iterator::max_by, algo.rs:311-322): a later row replaces an
            // equal value; inside the row the key's low bits prefer the larger column.  TRACK 3: the FIRST maximum
            // (alignment_table's max_cell, algo.rs:258-262): only a strictly larger value replaces (rows arrive in
            // increasing order).  A slot without a row (INT32_MIN) never replaces anything.
            const int rbase = t0 + ch * G::SPC - lane;
#pragma unroll
            for (int x = 0; x < G::SPC; ++x) {
                const bool upd = (TRACK == 2) ? ((rbk[x] | (K - 1)) >= best && rbk[x] != INT32_MIN) : ((rbk[x] | (K - 1)) > (best | (K - 1)));
                best = upd ? rbk[x] : best;
                best_r = upd ? rbase + x : best_r;
            }
        }
        if (CODES) st_cs_uint4(code_dst + ch * 32, make_uint4(cw[0], cw[1], cw[2], cw[3]));
    }
}

// BAND (global traceback plans with a code band): the kernel carries BOTH the traceback and the score-only variant of the
// tile's batch loops and picks one per tile (FillParams::tile_codes).  The choice is made once per tile, around two complete
// copies of the loops: dispatching per batch inside shared loops slowed a resident strip's traceback variant by 8-40 %
// (BRCA2 fill 0.99 -> 1.41 ms) even when the other variant never ran.  BAND_COMPACT also takes the tile's code address
// from its slot (FillParams::tile_slot, gx_common.cuh) instead of from its position in the table; its LOCAL instance runs
// with TRACK 0, after a score-only start-cell pass (TRACK 2) whose tile_best it leaves to the walk.
constexpr int BAND_NONE = 0, BAND_DENSE = 1, BAND_COMPACT = 2;
template <int K, bool LOCAL, bool CODES, int TRACK, bool PROF, bool CHAIN1, int BAND = BAND_NONE>
__global__ void __launch_bounds__(CTA_THREADS, CTAS_PER_SM) gx_fill_kernel(const FillParams P) {
    using G = Geo<K>;
    constexpr int W = G::W;
    const int cpb = (int)P.cpb;          // code chunks per hand-off batch (run-time: see Geo)
    const int B = cpb * G::SPC;          // steps (= rows) per batch, <= 32
    constexpr int KB = G::KB;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    uint8_t *wsm = smem + wib * WARP_SMEM_BYTES;
    uint8_t *s1buf = wsm;
    uint2 *inring = reinterpret_cast<uint2 *>(wsm + WARP_SMEM_S1);   // 2 x B entries (double-buffered by batch)
    uint2 *outring = inring + 64;
    uint64_t *mbar = reinterpret_cast<uint64_t *>(outring + 64);
    static_assert(WARP_SMEM_S1 + 2 * 64 * 8 + 16 == WARP_SMEM_BYTES, "per-warp shared-memory layout");

    // the s1 staging buffer starts out as valid symbols: unmasked batches prefetch up to 2 bytes past the rows the
    // TMA copy delivered (stale bytes of an earlier tile, or these zeros -- any symbol 0..3 indexes a real profile row)
    for (int x = lane; x < WARP_SMEM_S1 / 16; x += 32) reinterpret_cast<uint4 *>(s1buf)[x] = make_uint4(0u, 0u, 0u, 0u);
    if (lane == 0) {
        mbar_init(mbar, 1);
        fence_mbar_init();
    }
    __syncwarp();
    uint32_t phase = 0;
    const int g = P.g, hg = P.hg, h = P.h;
    // classic form: S = Ediag + (score - (h+g)) in V-space; CHAIN1: Sh = Ediag + score in E-space
    const int ap = CHAIN1 ? P.ap + P.hg : P.ap, bp = CHAIN1 ? P.bp + P.hg : P.bp;
    const uint32_t one = P.one;
    const uint32_t parity = P.parity;
    uint32_t *abort_word = P.ticket + 1;
    uint32_t *chk = P.ticket + 2;        // checked build: site number of a failed bounds check
    (void)chk;
    bool dead = false;
    const uint8_t *seq = PROF ? P.blob_sym : P.blob;   // PROF: sequences re-encoded to symbols 0..3 (gx_encode_kernel)

    // Two ways to hand tiles to warps:
    //   tickets          (more strips than resident warps) every free warp draws the next tile of the dependency-ordered list;
    //   resident strips  (P.pmax != 0: every strip of the plan has a warp of its own) warp g owns strip g for all
    //                    of its panels.  The strips of a pair form a chain that runs at the pace of its slowest member, so
    //                    what matters is that no scheduler holds more busy warps than the others: consecutive strips go to
    //                    consecutive CTAs, which the block scheduler deals round-robin over the SMs -- with tickets the
    //                    strip-to-scheduler assignment is re-drawn at every panel and some scheduler always ends up with 4.
    // (resident mode: the tile list is laid out [strip][panel], padded to P.pmax panels per strip)
    const uint32_t wg = blockIdx.x * (blockDim.x >> 5) + (uint32_t)wib;   // global warp index
    uint32_t own = 0;
    for (;;) {
        uint32_t tk = 0;
        if (P.pmax != 0u) {
            if (own >= P.pmax) break;
            tk = wg * P.pmax + own++;
        } else {
            if (lane == 0) tk = atomicAdd(P.ticket, 1u);
            tk = __shfl_sync(FULL, tk, 0);
        }
        if (tk >= P.n_tiles) break;
        const TileDesc td = P.tiles[tk];
        if (td.pair == 0xffffffffu) break;      // padding: this strip has fewer panels
        GX_CHECK(chk, td.pair < P.n_pairs, 1);
        const PairDesc *pd = P.pairs + td.pair;
        const int m = (int)pd->m, n = (int)pd->n, S = (int)pd->S;
        const int p = (int)td.p, s = (int)td.s;
        const int i0 = p << PANEL_H_LOG2;
        const int rows = min(PANEL_H, m - i0);
        const int jl = s * W + lane * K;  // columns jl+1 .. jl+K (1-based) belong to this lane
        const int kvalid = min(max(n - jl, 0), K);
        const bool has_pad = (s + 1) * W > n;
        const int col0 = (int)pd->col0;
        GX_CHECK(chk, p >= 0 && p < (int)pd->P && s >= 0 && s < S && rows > 0 && rows <= PANEL_H, 2);
        GX_CHECK(chk, B >= 1 && B <= 32 && cpb >= 1 && cpb <= G::CPB_MAX, 3);

        // ---- stage s1[i0 .. i0+rows) with a TMA bulk copy (16-byte aligned window around it)
        const uint8_t *s1g = seq + pd->s1_off + i0;
        const uint32_t delta = (uint32_t)(reinterpret_cast<uintptr_t>(s1g) & 15u);
        __syncwarp();
        if (lane == 0) {
            fence_proxy_async_smem();  // earlier generic-proxy reads of s1buf are done (syncwarp above)
            const uint32_t bytes = (delta + (uint32_t)rows + 15u) & ~15u;
            mbar_expect_tx(mbar, bytes);
            tma_bulk_g2s(s1buf, s1g - delta, bytes, mbar);
        }

        // ---- s2 of this lane's columns: characters in registers, or the match/mismatch profile in smem
        int c2[K];
        {
            const uint8_t *s2g = seq + pd->s2_off + jl;
#pragma unroll
            for (int k = 0; k < K; ++k) c2[k] = (k < kvalid) ? (int)__ldg(s2g + k) : 256;
        }
        // PROF: the four possible scores of each column, one per byte (symbols are staged as shift amounts 0, 8, 16, 24;
        // padding columns hold 256 and score `mismatch` against everything)
        int prof4[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            uint32_t w = 0u;
#pragma unroll
            for (int sym = 0; sym < 4; ++sym) w |= ((uint32_t)((c2[k] == 8 * sym) ? ap : bp) & 0xffu) << (8 * sym);
            prof4[k] = PROF ? (int)w : 0;
        }

        // ---- top boundary of the tile: (E,D) of row i0 for this lane's columns
        int eu[K], du[K];
        if (p == 0) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                eu[k] = (LOCAL ? 0 : h + (col0 + jl + k + 1) * g) + hg;  // algo.rs:213-220 (row 0), V = insert_score
                du[k] = NEG32;
            }
        } else {
            // the previous panel of this strip must be complete (its `top` rows written)
            const uint32_t *pr = P.progress + pd->progress_off + s;
            uint32_t spins = 0;
            // poll with relaxed loads and a growing sleep (an acquire load is LDG + CCTL.IVALL: hundreds of waiting
            // warps invalidating their SM's L1 every microsecond slow the warps that do the work), acquire once at the end
            uint32_t nap = 100;
            while (ld_relaxed_u32(pr) < (uint32_t)p) {
                if (spin_check(spins, abort_word)) {
                    dead = true;
                    break;
                }
                __nanosleep(nap);
                nap = min(nap * 2u, 1000u);
            }
            (void)ld_acquire_u32(pr);
            if (dead) break;
            const int2 *tp = P.top + pd->top_off + jl;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                int2 v = make_int2(NEG32, NEG32);
                if (k < kvalid) v = ld_cg_int2(tp + k);
                eu[k] = v.x;
                du[k] = v.y;
            }
        }
        // left boundary: previous strip's column buffer, or the band inbox (written by the neighbouring band / GPU)
        const bool left_band = (s == 0) && (pd->inbox != nullptr);
        const bool right_band = (s == S - 1) && (pd->outbox != nullptr);
        const unsigned long long *cb_in =
            (s > 0) ? P.colbuf + pd->colbuf_off + (uint64_t)(s - 1) * m + i0 : (left_band ? pd->inbox + i0 : nullptr);
        unsigned long long *cb_out =
            (s < S - 1) ? P.colbuf + pd->colbuf_off + (uint64_t)s * m + i0 : (right_band ? pd->outbox + i0 : nullptr);
        const bool has_left = cb_in != nullptr;
        auto ld_bnd = [&](const unsigned long long *q) __attribute__((always_inline)) { return left_band ? ld_relaxed_sys_u64(q) : ld_relaxed_u64(q); };

        // ---- diagonal seed: E of (row i0, column jl)
        int vd = __shfl_up_sync(FULL, eu[K - 1], 1);
        if (lane == 0) {
            if (!has_left) {
                vd = ((p == 0) ? 0 : (LOCAL ? 0 : h + i0 * g)) + hg;      // algo.rs:195-211 (column 0)
            } else if (p == 0) {
                vd = (LOCAL ? 0 : h + (col0 + jl) * g) + hg;              // row 0
            } else {
                unsigned long long v;
                uint32_t spins = 0;
                while ((((uint32_t)((v = ld_bnd(cb_in - 1)) >> 32)) & 1u) != parity) {
                    if (spin_check(spins, abort_word)) {
                        dead = true;
                        break;
                    }
                    __nanosleep(100);
                }
                vd = (int)(uint32_t)v;
            }
        }
        // remote outbox: the neighbouring GPU must have finished consuming the previous execute before row 1 of
        // this one overwrites its inbox (the consumer's stream stores its finished-execute count into pd->ack)
        if (right_band && p == 0 && pd->ack != nullptr && lane == 0) {
            uint32_t spins = 0;
            while (ld_acquire_sys_u32(pd->ack) + 1u < P.epoch) {
                if (spin_check(spins, abort_word)) {
                    dead = true;
                    break;
                }
                __nanosleep(2000);
            }
        }
        dead = __any_sync(FULL, dead);
        if (dead) break;

        int eo = 0, io = 0;   // this lane's right edge (E, I) of the row of its last step: what the next lane shuffles in
        int best = (CHAIN1 || TRACK == 3) ? INT32_MIN : -1, best_r = 0;
        const uint32_t nbat = tile_batches((uint32_t)rows, B);
        uint4 *code_base = nullptr;
        int code_tile = p * S + s;       // where this tile's codes are, in tiles from the pair's codes_off
        if constexpr (BAND == BAND_COMPACT) code_tile = (int)P.tile_slot[pd->tile_base + p * S + s];
        if (CODES)
            code_base = reinterpret_cast<uint4 *>(P.codes + pd->codes_off + (uint64_t)code_tile * pd->tile_code_bytes) + lane;
        // code band (global plans): tiles away from the table's diagonal run the score-only cell and write no codes
        bool tcodes = CODES;
        if constexpr (BAND != BAND_NONE) tcodes = P.tile_codes[pd->tile_base + p * S + s] != 0;

        // ---- left boundary prefetch (LL protocol): lanes 0..B-1 fetch the entries of local rows B*bt + lane
        unsigned long long nxt = 0;
        auto issue = [&](uint32_t bt) __attribute__((always_inline)) {
            const int r = (int)(B * bt) + lane;
            GX_CHECK(chk, !(has_left && lane < B && r < rows) || (i0 + r >= 0 && i0 + r < m), 4);
            if (has_left && lane < B && r < rows) nxt = ld_bnd(cb_in + r);
        };
        issue(0);

        // wait for the s1 segment
        {
            uint32_t tries = 0;
            while (!mbar_try_wait(mbar, phase)) {
                if (++tries > (1u << 24)) {
                    atomicExch(abort_word, 1u);
                    dead = true;
                    break;
                }
            }
            dead = __any_sync(FULL, dead);
            if (dead) break;
        }
        phase ^= 1u;
        const uint8_t *s1base = s1buf + delta;
        __syncwarp();
        // the s1 character of step 0 (run_batch fetches one step ahead)
        int c1a = s1base[min(max(-lane, 0), rows - 1)];

        // ---- batch loop.  The hand-off rings are double-buffered (the global load of batch bt+2's left boundary is in
        //      flight while batch bt computes), and every batch ends with: publish its finished right-boundary rows,
        //      then settle the in-ring of the next batch (post() below).
        // settle(b): lanes 0..B-1 turn the prefetched word of local row B*b+lane into an in-ring entry.
        // The common case (data already there) is branch-free apart from one vote.
        const bool lane_b = lane < B;
        auto settle = [&](uint32_t b) __attribute__((always_inline)) -> bool {
            const int rb = (int)(B * b) + lane;
            const bool need = has_left && lane_b && (rb < rows);
            bool ok = !need || ((((uint32_t)(nxt >> 32)) & 1u) == parity);
            if (!__all_sync(FULL, ok)) {
                uint32_t spins = 0;
                bool lost = false;
                do {
                    if (__any_sync(FULL, spin_check(spins, abort_word))) {
                        lost = true;
                        break;
                    }
                    // not there yet: poll again at once.  The L2 round trip (~500 clk) paces the loop, a polling warp
                    // issues ~3 % of its scheduler's slots, and every nap here would be added to the lag of this strip
                    // behind its left neighbour -- strips x lag is the pipeline ramp of a pair.
                    if (!ok) nxt = ld_bnd(cb_in + rb);
                    ok = !need || ((((uint32_t)(nxt >> 32)) & 1u) == parity);
                } while (!__all_sync(FULL, ok));
                if (lost) return false;
            }
            uint2 cur;
            cur.x = has_left ? (uint32_t)nxt : (uint32_t)((LOCAL ? 0 : h + (i0 + rb + 1) * g) + hg);  // algo.rs:204-211: V = delete_score
            cur.y = has_left ? (uint32_t)(((int)(uint32_t)(nxt >> 32)) >> 1) : (uint32_t)NEG32;
            GX_CHECK(chk, !lane_b || (b & 1u) * B + lane < 64, 5);
            if (lane_b) inring[(b & 1u) * B + lane] = cur;
            return true;
        };
        if (!settle(0)) dead = true;
        if (nbat > 1) issue(1);
        __syncwarp();
        uint2 pub = make_uint2(0u, 0u);   // out-ring entry read back after the previous batch
        int pub_row = -1;
        auto flush_pub = [&]() __attribute__((always_inline)) {
            if (pub_row >= 0) {
                GX_CHECK(chk, i0 + pub_row < m, 6);
                const unsigned long long packed =
                    (unsigned long long)pub.x | ((unsigned long long)((pub.y << 1) | parity) << 32);
                if (right_band) st_relaxed_sys_u64(cb_out + pub_row, packed);
                else st_relaxed_u64(cb_out + pub_row, packed);
            }
        };
        // glue after the DP steps of batch bt.  Order matters for the lag of a strip behind its left neighbour
        // (strips x lag is the pipeline ramp of a pair): the in-ring of batch bt+1 is settled only now, just in time,
        // and the rows finished in batch bt are published before anything else can block.
        const bool has_out = cb_out != nullptr;
        auto post = [&](uint32_t bt, uint2 *outr) __attribute__((always_inline)) -> bool {
            // rows lane 31 finished in this batch: rows t0-31 .. t0+B-32
            const int ro = (int)(B * bt) - 31 + lane;
            const bool take = has_out && lane_b && ro >= 0 && ro < rows;
            __syncwarp();                                    // out-ring stores of this batch -> visible
            if (take) pub = lds_volatile_uint2(outr + lane);
            pub_row = take ? ro : -1;
            flush_pub();
            pub_row = -1;
            if (bt + 1 < nbat) {
                if (!settle(bt + 1)) return false;           // may wait for the left neighbour
                if (bt + 2 < nbat) issue(bt + 2);
                __syncwarp();                                // in-ring stores of batch bt+1 -> visible
            }
            return true;
        };
        // batches [0, nb_head) and [nb_body, nbat) touch rows outside the tile (skew) and run the masked steps;
        // the body runs unmasked steps with straight-line glue.
        const uint32_t nb_head = (30 + B) / B;                              // first batch with t0 >= 31
        const uint32_t nb_body = max(nb_head, (uint32_t)rows / B);          // first batch that reaches past the last row
        bool thru = false;
        if constexpr (!LOCAL && !CODES && TRACK == 0) thru = right_band && has_pad;
        // phase 0: masked head batches (all batches of a THRU tile), then the unmasked body; phase 1: masked tail.
        // (One copy of each batch variant in the code; nothing here may end up as an out-of-line call -- the DP
        // state lives in registers.)
        // The batch loops of one tile, in the variant this tile needs: with direction codes, or -- a tile outside the code
        // band of a global traceback plan -- the score-only cell.  BAND kernels carry TWO complete copies of the loops and pick
        // one per tile at this level (dispatching per batch inside shared loops cost a resident strip 8-40 %).
        auto run_tile = [&](auto codes_c) __attribute__((always_inline)) {
            constexpr bool WC = decltype(codes_c)::value;
            uint32_t bt = 0;
            for (int ph = 0; ph < 2 && !dead; ++ph) {
                const uint32_t m_end = (ph == 0 && !thru) ? min(nb_head, nbat) : nbat;
                for (; bt < m_end && !dead; ++bt) {
                    uint2 *outr = outring + (bt & 1u) * B;
                    uint4 *cdst = WC ? code_base + (size_t)bt * cpb * 32 : nullptr;
                    GX_CHECK(chk, !WC || ((size_t)(bt + 1) * cpb * 512 <= pd->tile_code_bytes &&
                                          pd->codes_off + (uint64_t)(code_tile + 1) * pd->tile_code_bytes <= P.code_bytes), 7);
                    if constexpr (!LOCAL && !CODES && TRACK == 0) {
                        if (thru)
                            run_batch<K, LOCAL, WC, TRACK, PROF, true, false, CHAIN1, true>(eu, du, c2, eo, io, vd, best, best_r, g, hg, ap, bp,
                                                                                            one, s1base, prof4, inring + (bt & 1u) * B, outr, cdst,
                                                                                            (int)(B * bt), rows, lane, kvalid, c1a, cpb, chk, -(int)delta, WARP_SMEM_S1 - (int)delta);
                    }
                    if (!thru)
                        run_batch<K, LOCAL, WC, TRACK, PROF, true, (TRACK != 0), CHAIN1>(eu, du, c2, eo, io, vd, best, best_r, g, hg, ap, bp,
                                                                                         one, s1base, prof4, inring + (bt & 1u) * B, outr, cdst,
                                                                                         (int)(B * bt), rows, lane, kvalid, c1a, cpb, chk, -(int)delta, WARP_SMEM_S1 - (int)delta);
                    if (!post(bt, outr)) dead = true;
                }
                if (ph != 0 || thru || dead) continue;
                // Columns right of the table (last strip of a pair) need their keys masked only when a padded cell could
                // reach the maximum; with s_mismatch < 0 (and g, h+g < 0) every padded cell is strictly smaller than the real
                // cell it derives from, so the plain body is exact -- the tile reductions ignore winners with j > n.
                if ((TRACK != 0) && has_pad && P.pad_keys != 0u) {
                    for (; bt < nb_body && !dead; ++bt) {
                        uint2 *outr = outring + (bt & 1u) * B;
                        uint4 *cdst = WC ? code_base + (size_t)bt * cpb * 32 : nullptr;
                        GX_CHECK(chk, !WC || ((size_t)(bt + 1) * cpb * 512 <= pd->tile_code_bytes &&
                                              pd->codes_off + (uint64_t)(code_tile + 1) * pd->tile_code_bytes <= P.code_bytes), 7);
                        run_batch<K, LOCAL, WC, TRACK, PROF, false, true, CHAIN1>(eu, du, c2, eo, io, vd, best, best_r, g, hg, ap, bp,
                                                                                  one, s1base, prof4, inring + (bt & 1u) * B, outr, cdst,
                                                                                  (int)(B * bt), rows, lane, kvalid, c1a, cpb, chk, -(int)delta, WARP_SMEM_S1 - (int)delta);
                        if (!post(bt, outr)) dead = true;
                    }
                } else {
                    for (; bt < nb_body && !dead; ++bt) {
                        uint2 *outr = outring + (bt & 1u) * B;
                        uint4 *cdst = WC ? code_base + (size_t)bt * cpb * 32 : nullptr;
                        GX_CHECK(chk, !WC || ((size_t)(bt + 1) * cpb * 512 <= pd->tile_code_bytes &&
                                              pd->codes_off + (uint64_t)(code_tile + 1) * pd->tile_code_bytes <= P.code_bytes), 7);
                        run_batch<K, LOCAL, WC, TRACK, PROF, false, false, CHAIN1>(eu, du, c2, eo, io, vd, best, best_r, g, hg, ap, bp,
                                                                                   one, s1base, prof4, inring + (bt & 1u) * B, outr, cdst,
                                                                                   (int)(B * bt), rows, lane, kvalid, c1a, cpb, chk, -(int)delta, WARP_SMEM_S1 - (int)delta);
                        if (!post(bt, outr)) dead = true;
                    }
                }
            }
        };
        if constexpr (BAND != BAND_NONE) {
            if (tcodes) run_tile(std::true_type{});
            else run_tile(std::false_type{});
        } else {
            run_tile(std::integral_constant<bool, CODES>{});
        }
        flush_pub();
        if (dead) break;

        // ---- bottom row -> top buffer (next panel of this strip, and the global score)
        {
            int2 *tp = P.top + pd->top_off + jl;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                GX_CHECK(chk, !(k < kvalid) || jl + k < n, 8);
                if (k < kvalid) st_cg_int2(tp + k, make_int2(eu[k], du[k]));
            }
            __syncwarp();
            if (lane == 0) st_release_u32(P.progress + pd->progress_off + s, (uint32_t)(p + 1));
        }

        // ---- tile-level local maximum (value, i, j): larger value, then larger i, then larger j
        if (TRACK != 0) {
            int bv, bi, bj;
            if (TRACK == 2) {
                if (CHAIN1) bv = (kvalid == 0) ? -1 : (best >> KB) - hg;   // keys were taken in E-space
                else bv = (best < 0) ? -1 : (best >> KB);
                bi = i0 + best_r + 1;
                bj = jl + (best & (K - 1)) + 1;
            } else if (TRACK == 3) {
                bv = (kvalid == 0) ? INT32_MIN : (best >> KB) - (CHAIN1 ? hg : 0);
                bi = i0 + best_r + 1;
                bj = jl + (K - 1 - (best & (K - 1))) + 1;
            } else {
                if (CHAIN1) bv = (kvalid == 0) ? -1 : best - hg;
                else bv = best;
                bi = 0;
                bj = 0;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const int ov = __shfl_xor_sync(FULL, bv, off);
                const int oi = __shfl_xor_sync(FULL, bi, off);
                const int oj = __shfl_xor_sync(FULL, bj, off);
                const bool take = (TRACK == 3) ? ((ov > bv) || (ov == bv && (oi < bi || (oi == bi && oj < bj))))
                                               : ((ov > bv) || (ov == bv && (oi > bi || (oi == bi && oj > bj))));
                bv = take ? ov : bv;
                bi = take ? oi : bi;
                bj = take ? oj : bj;
            }
            if (lane == 0) P.tile_best[pd->tile_base + p * S + s] = make_int4(bv, bi, bj, 0);
        }
    }
}

// Re-encodes sequence bytes to dense symbols through a 256-entry table (PROF path): sym 0..3, 255 = not in alphabet.
static __global__ void __launch_bounds__(256) gx_encode_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, size_t n,
                                                        const uint8_t *__restrict__ lut256) {
    __shared__ uint8_t lut[256];
    lut[threadIdx.x] = lut256[threadIdx.x];
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = lut[in[i]];
}

// Band flow control: tells the left neighbour (its memory, possibly over NVLink) that execute `epoch` of this
// band has consumed its inbox completely.  Stream-ordered after the fill kernel.
static __global__ void gx_band_ack_kernel(uint32_t *peer_ack, uint32_t epoch) { st_release_sys_u32(peer_ack, epoch); }

}  // namespace gx
