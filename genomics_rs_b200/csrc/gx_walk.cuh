// gx_walk.cuh -- K3: start-cell selection and traceback walk on the GPU.
//
// Replaces /root/reference/src/alignment/algo.rs:287-441 (retrace):
//   start cell  algo.rs:306-323  global (m,n); local = last maximum in row-major order
//   score       algo.rs:331
//   walk        algo.rs:339-422  state-less choice S > I > D (here: the stored 2-bit code),
//               off-by-one match label is_match(i,j) (algo.rs:354, sequence.rs:102-115),
//               open/extend labels from last_choice (algo.rs:373-379,388-394),
//               checked_sub index update (algo.rs:412-417), stop at (0,0) (algo.rs:419-421).
// One CTA of four warps per pair.  The walk is m+n dependent steps; what it costs is the length of the dependent
// chain ONE warp has to issue per run of equal codes, so everything that is not path finding lives in other warps:
//   path warp   (warp 0)    follows the stored direction codes inside a window of code chunks held in shared memory:
//                           lane x inspects the cell x moves ahead in the current direction, a ballot gives the run
//                           length, the look-ahead lane that already read the turn cell supplies the next direction.
//                           One self-contained 16-byte descriptor per run goes into a shared-memory ring.
//   loader warp (warp 2)    owns the code windows: on request it copies the chunks of (tile, row range) into one of three
//                           window buffers (cp.async, 16 B each) and checks the tile's code-band flag (a tile outside
//                           the band is not copied: with compact code storage it has no codes of its own).  The path warp asks
//                           for the windows it will probably need next (left neighbour strip at the rows where a
//                           diagonal path leaves this one; the rows above) when it enters a window, so a window change
//                           normally costs a few shared-memory reads.
//   emit warps  (warps 1,3) pop descriptors (even / odd sequence numbers) and do the rest: the off-by-one match labels
//                           is_match(i, j) (characters from global memory / L1), open/extend labels, the four counters,
//                           the coalesced op stores, the end cell.
#pragma once
#include "gx_common.cuh"
#include "gx_fill.cuh"

namespace gx {

// dynamic shared memory of one walk CTA: a 2 KB control block (descriptor ring, request ring, tails, ready words, partial
// results) and three code-window buffers.
// A window is `rows` rows of one strip = rows (+1) steps + 31 steps of lane skew, 64/K steps per code chunk.
__host__ __device__ constexpr uint32_t walk_chunks(int K, uint32_t rows) {
    return (uint32_t)((rows + 1 + 31 + 64 / K - 1) / (64 / K) + 1);
}
__host__ __device__ constexpr uint32_t walk_buf_bytes(int K, uint32_t rows) { return walk_chunks(K, rows) * 32 * 16; }
constexpr uint32_t WALK_CTRL_BYTES = 2048;
constexpr uint32_t WALK_RING = 64;          // run descriptors in flight between the path warp and the emit warps
constexpr uint32_t WALK_REQ = 8;            // window requests in flight between the path warp and the loader warp (<= 3 used)
constexpr uint32_t WALK_NBUF = 3;           // window buffers: the current one and two prefetch targets
constexpr uint32_t WALK_EMIT = 2;            // emit warps (<= 4: their tails are read with one 16-byte load)
constexpr uint32_t WALK_THREADS = 64 + 32 * WALK_EMIT;   // path warp, emit warp 0, loader warp, emit warps 1..
__host__ __device__ constexpr uint32_t walk_smem_bytes(int K, uint32_t rows) {
    return WALK_CTRL_BYTES + WALK_NBUF * walk_buf_bytes(K, rows);
}
static_assert(PANEL_H_LOG2 <= 12, "window requests carry panel rows in 12 bits");

__device__ __forceinline__ uint32_t lds_volatile_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void sts_volatile_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_volatile_uint4(uint4 *p, uint4 v) {
    asm volatile("st.volatile.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(smem_u32(p)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds_volatile_uint4(const uint4 *p) {
    uint4 v;
    asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)) : "memory");
    return v;
}
// a code word of the current window (written by the loader warp's cp.async: never cached in a register across a window change)
__device__ __forceinline__ uint32_t lds_code_word(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

template <int K>
__global__ void __launch_bounds__(WALK_THREADS) gx_walk_kernel(const WalkParams P) {
    const uint32_t q = blockIdx.x;
    if (q >= P.n_pairs) return;
    const int lane = threadIdx.x & 31;
    const int wid = threadIdx.x >> 5;
    const PairDesc *pd = P.pairs + q;
    const uint32_t m = pd->m, n = pd->n;
    const uint8_t *s1 = P.blob + pd->s1_off;
    const uint8_t *s2 = P.blob + pd->s2_off;
    const bool local = P.is_local != 0;

    // ---- start cell and score
    long long score;
    uint32_t i = m, j = n;
    if (local) {
        int bv = 0, bi = (int)m, bj = (int)n;  // boundary cells have V = 0; the last cell of the table wins a tie at 0
        if (m > 0 && n > 0) {
            bv = -1;
            bi = 0;
            bj = 0;
            const uint32_t ntile = pd->S * pd->P;
            for (uint32_t x = lane; x < ntile; x += 32) {
                const int4 tb = P.tile_best[pd->tile_base + x];
                // a winner right of the table can only come from a tile whose maximum is 0 (see gx_fill.cuh): the boundary
                // cell (m, n) this reduction starts from covers it
                const bool take = (tb.z <= (int)n) && ((tb.x > bv) || (tb.x == bv && (tb.y > bi || (tb.y == bi && tb.z > bj))));
                if (take) {
                    bv = tb.x;
                    bi = tb.y;
                    bj = tb.z;
                }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const int ov = __shfl_xor_sync(0xffffffffu, bv, off);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
                const bool take = (ov > bv) || (ov == bv && (oi > bi || (oi == bi && oj > bj)));
                bv = take ? ov : bv;
                bi = take ? oi : bi;
                bj = take ? oj : bj;
            }
            // Table maximum 0: every cell ties, and the last one in row-major order is (m, n) (Iterator::max_by,
            // algo.rs:311-322).  The tiles cannot be trusted to say so: a padded column right of the table also holds 0
            // and may have won its tile, which the filter above then dropped together with the tile's real zeros.
            if (bv <= 0) {
                bv = 0;
                bi = (int)m;
                bj = (int)n;
            }
        }
        score = bv;
        if (P.have_best) {
            i = (uint32_t)bi;
            j = (uint32_t)bj;
        }
    } else {
        if (m == 0 && n == 0) score = 0;
        else if (m == 0) score = (long long)P.h + (long long)n * P.g;   // algo.rs:213-220
        else if (n == 0) score = (long long)P.h + (long long)m * P.g;   // algo.rs:204-211
        else score = (long long)P.top[pd->top_off + (n - 1)].x - P.hg;
    }

    DevResult res;
    res.score = score;
    res.start_i = i;
    res.start_j = j;
    res.end_i = i;
    res.end_j = j;
    res.n_ops = 0;
    res.matches = res.mismatches = res.gap_extensions = res.opening_gaps = 0;
    res.lcs_at_first_max = 0;
    res.fill_ms = res.walk_ms = 0.0;

    if (!P.traceback) {
        if (threadIdx.x == 0) P.results[q] = res;
        return;
    }
    if (i == 0 && j == 0) {
        // only possible for m == n == 0: one Match at (0,0) (None == None), then both checked_sub fail
        if (threadIdx.x == 0) {
            P.ops[pd->ops_off] = 0;
            res.n_ops = 1;
            res.matches = 1;
            P.results[q] = res;
        }
        return;
    }

    using G = Geo<K>;
    constexpr uint32_t SPC = G::SPC;
    const uint32_t WR = P.win_rows;                          // rows per window (64..512, chosen per launch); a window spans the strip's width
    const uint32_t BUF_BYTES = walk_buf_bytes(K, WR);
    extern __shared__ __align__(16) uint8_t walk_smem[];
    // descriptor ring, LL style: {i | tag, j, direction | previous direction << 2 | run << 4 | tag, ops emitted before}.  The path warp
    // writes a descriptor with ONE 16-byte shared-memory store and the emit warp it belongs to (sequence number mod WALK_EMIT) polls
    // the slot until it carries the lap tag it expects: no head word, no fence on the path warp's dependent chain.
    // tail[e] (descriptors emit warp e is done with) is only read when the ring looks full.
    uint4 *ring = reinterpret_cast<uint4 *>(walk_smem);
    uint4 *req = reinterpret_cast<uint4 *>(walk_smem + WALK_RING * 16);              // {panel, strip, r0 | r1 << 12 | buffer << 24 | quit << 31, seq}
    uint32_t *tail = reinterpret_cast<uint32_t *>(walk_smem + WALK_RING * 16 + WALK_REQ * 16);
    uint32_t *ready = tail + 4;                                                        // per buffer: last request finished | no-codes << 31
    uint32_t *part = tail + 8;                                                         // per emit warp: 8 words of partial results
    uint32_t *scratch = tail + 16 + 8 * WALK_EMIT;                                     // 64 words
    uint8_t *bufs = walk_smem + WALK_CTRL_BYTES;
    if (threadIdx.x < WALK_RING) ring[threadIdx.x] = make_uint4(0u, 0u, 0u, 0u);       // lap tags start at 1
    if (threadIdx.x < WALK_REQ) req[threadIdx.x] = make_uint4(0u, 0u, 0u, 0u);         // request numbers start at 1
    if (threadIdx.x < 8 + 8 * WALK_EMIT) tail[threadIdx.x] = 0u;                        // tails, ready words, partial results
    __syncthreads();

    if (wid == 0) {
        // ================================================================ path warp
        // lane `lane` looks y = 31 - lane moves ahead: the run length is then a count of leading ones of the ballot.
        // y and the ring's shared-memory address make a round trip through shared memory: values ptxas cannot re-derive
        // from %tid / the CTA's shared window inside the loop (it otherwise does, with 20-clock S2R / S2UR reads per run).
        uint32_t y, ring_s;
        {
            sts_volatile_u32(scratch + lane, 31u - (uint32_t)lane);
            sts_volatile_u32(scratch + 32 + lane, smem_u32(ring));
            y = lds_volatile_u32(scratch + lane);
            ring_s = lds_volatile_u32(scratch + 32 + lane);
        }
        uint32_t pushed = 0, safe = WALK_RING;               // descriptors pushed; pushes below `safe` find their slot free
        uint32_t nops = 0, prevc = 0;                        // ops pushed so far; direction of the previous run (Match, algo.rs:338)
        auto push = [&](uint32_t pi, uint32_t pj, uint32_t meta, uint32_t before) __attribute__((always_inline)) {
            if (pushed >= safe) {           // slot reuse: its previous descriptor (RING back) must have been consumed
                do {                        // tail[e] = 1 + the last descriptor emit warp e is done with: everything below all of them is consumed
                    const uint4 tl = lds_volatile_uint4(reinterpret_cast<const uint4 *>(tail));
                    uint32_t lo = tl.x;
                    if (WALK_EMIT > 1) lo = min(lo, tl.y);
                    if (WALK_EMIT > 2) lo = min(lo, tl.z);
                    if (WALK_EMIT > 3) lo = min(lo, tl.w);
                    safe = lo + WALK_RING;
                } while (pushed >= safe);
            }
            // the lap tag rides in both 8-byte halves: a reader that caught the halves from different laps -- should
            // 16-byte shared accesses ever be split -- does not accept the slot.  Every lane stores the same value (no branch).
            const uint32_t tag = ((pushed / WALK_RING + 1u) & 7u) << 29;
            asm volatile("st.volatile.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(ring_s + (pushed % WALK_RING) * 16u), "r"(pi | tag), "r"(pj),
                         "r"(meta | tag), "r"(before)
                         : "memory");
            pushed++;
        };

        // ---- window state
        uint32_t cbase = 0;                 // shared-memory address of the current window buffer
        int rrel = 0, jw = 0;               // row inside the window (= inside the buffer), column in the strip
        uint32_t cb = 0;                    // current buffer
        // what each buffer holds / will hold: tile (bp, bs), panel rows [br0, br1], the request that fills it
        uint32_t bp[WALK_NBUF], bs[WALK_NBUF], br0[WALK_NBUF], br1[WALK_NBUF], bq[WALK_NBUF];
#pragma unroll
        for (uint32_t b = 0; b < WALK_NBUF; ++b) {
            bp[b] = 0xffffffffu;
            bs[b] = br0[b] = br1[b] = bq[b] = 0u;
        }
        uint32_t nreq = 0;
        auto post = [&](uint32_t b, uint32_t p, uint32_t s_, uint32_t r0, uint32_t r1) __attribute__((always_inline)) -> uint32_t {
            nreq++;
            sts_volatile_uint4(req + nreq % WALK_REQ, make_uint4(p, s_, r0 | (r1 << 12) | (b << 24), nreq));
            return nreq;
        };
        // code of the window cell (row rr relative to the buffer's first chunk, column jc of the strip): 0 S / 1 I / 2 D / 3 stop
        auto code_at = [&](uint32_t rr, uint32_t jc) __attribute__((always_inline)) -> uint32_t {
            // 64 cells (SPC steps x K columns) per 16-byte unit [chunk][fill-lane]; with u = t * K the cell is entry
            // (u & 63) | k of unit (u >> 6, l).  Written out so that the chain from (rr, jc) to the address is five
            // instructions deep (t, v, two masks, multiply-add, add)
            constexpr uint32_t LK = (K == 4) ? 2u : (K == 8) ? 3u : 4u;
            static_assert(K == 4 || K == 8 || K == 16, "code_at: K");
            const uint32_t l = jc >> LK, t = rr + l;              // the step at which fill-lane l worked on this row
            const uint32_t v = t << (LK - 2u);                    // u >> 2
            const uint32_t off = (v & ~15u) * 32u + (v & 12u) + (l << 4);   // (u >> 6) * 512 + l * 16 + (entry >> 4) * 4
            const uint32_t sh = ((((t << LK) | (jc & (K - 1u))) & 15u)) * 2u;
            GX_CHECK(P.check, off < BUF_BYTES, 21);
            const uint32_t word = lds_code_word(cbase + off);
            return (word >> sh) & 3u;
        };

        // first row of the window that ends at panel row r1: WR rows, rounded down to a code chunk's first row, so that the
        // row inside the buffer is the row inside the window (no offset on the chain)
        auto win_r0 = [&](uint32_t r1) __attribute__((always_inline)) -> uint32_t {
            return ((r1 >= WR - 1u) ? r1 - (WR - 1u) : 0u) / SPC * SPC;
        };
        bool left_band = false;
        bool walking = (i != 0 && j != 0);
        while (walking) {
            // ---------------- (i, j) is an interior cell outside the current window: change windows
            const uint32_t jj = j - 1u, ii = i - 1u;
            const uint32_t tp = ii >> PANEL_H_LOG2, ts = jj / G::W, tr = ii & (PANEL_H - 1);
            uint32_t hit = WALK_NBUF;
#pragma unroll
            for (uint32_t b = 0; b < WALK_NBUF; ++b)
                if (b != cb && bp[b] == tp && bs[b] == ts && tr >= br0[b] && tr <= br1[b]) hit = b;
            if (hit == WALK_NBUF) {
                // neither prediction holds this cell: load the window that ends at this row into the buffer just left
                hit = cb;
                const uint32_t r0 = win_r0(tr);
                const uint32_t sq = post(hit, tp, ts, r0, tr);
#pragma unroll
                for (uint32_t b = 0; b < WALK_NBUF; ++b)
                    if (b == hit) {
                        bp[b] = tp;
                        bs[b] = ts;
                        br0[b] = r0;
                        br1[b] = tr;
                        bq[b] = sq;
                    }
            }
            cb = hit;
            uint32_t wr0 = 0, wq = 0;
#pragma unroll
            for (uint32_t b = 0; b < WALK_NBUF; ++b)
                if (b == cb) {
                    wr0 = br0[b];
                    wq = bq[b];
                }
            uint32_t st;
            do {
                st = lds_volatile_u32(ready + cb);
            } while ((st & 0x7fffffffu) != wq);
            __threadfence_block();                                // the loader's copies are visible before the first code read
            // code band: a tile away from the table's diagonal holds no codes.  The path has left the band: give
            // up -- the host repeats the execute with codes everywhere (exactness never depends on the band).
            if (st >> 31) {
                left_band = true;
                break;
            }
            cbase = smem_u32(bufs + cb * BUF_BYTES);
            rrel = (int)(tr - wr0);                               // wr0 is the first row of the buffer's first chunk
            jw = (int)(jj % G::W);
            uint32_t c0 = code_at((uint32_t)rrel, (uint32_t)jw);
            // ask for the windows the walk will probably need next, into the two other buffers.  A diagonal path leaves this
            // window on the left after jw + 1 rows: the left neighbour strip around that row, with WR/4 rows of slack below it
            // (insertions) and the rest above (deletions, and the way across that strip); and the rows above this window.
            {
                uint32_t o1 = (cb + 1u) % WALK_NBUF, o2 = (cb + 2u) % WALK_NBUF;
                const int pred = (int)tr - (int)(jw + 1);
                const bool want_left = ts > 0 && pred + (int)(WR / 4u) >= 0;
                // (the rows above only when the path can get there before it leaves on the left: not for a full-height window)
                const bool want_top = (wr0 > 0 || tp > 0) && (!want_left || pred < (int)(wr0 + WR / 4u));
                uint32_t lp = 0xffffffffu, ls = 0, lr0 = 0, lr1 = 0, lq = 0;
                uint32_t up = 0xffffffffu, us = 0, ur0 = 0, ur1 = 0, uq = 0;
                if (want_left) {
                    lp = tp;
                    ls = ts - 1u;
                    lr1 = (uint32_t)min((int)tr, pred + (int)(WR / 4u));
                    lr0 = win_r0(lr1);
                    lq = post(o1, lp, ls, lr0, lr1);
                }
                if (want_top) {
                    us = ts;
                    if (wr0 > 0) {
                        up = tp;
                        ur1 = wr0 - 1u;
                        ur0 = win_r0(ur1);
                    } else {
                        up = tp - 1u;
                        ur1 = PANEL_H - 1;
                        ur0 = PANEL_H - WR;
                    }
                    uq = post(o2, up, us, ur0, ur1);
                }
#pragma unroll
                for (uint32_t b = 0; b < WALK_NBUF; ++b) {
                    if (b == o1) {
                        bp[b] = lp;
                        bs[b] = ls;
                        br0[b] = lr0;
                        br1[b] = lr1;
                        bq[b] = lq;
                    }
                    if (b == o2) {
                        bp[b] = up;
                        bs[b] = us;
                        br0[b] = ur0;
                        br1[b] = ur1;
                        bq[b] = uq;
                    }
                }
            }
            if (c0 == 3u) break;                          // local alignment ends here; the cell is not emitted (algo.rs:401-405)

            // ---------------- run following inside the window
            for (;;) {
                // lane y looks y moves ahead in the direction of c0, as far as the window reaches; the run ends at the
                // first different code.  Window cells are interior cells (i, j >= 1): no boundary cases on this chain.
                const bool mi = (c0 != 1u), mj = (c0 != 2u);
                const uint32_t a = mi ? (uint32_t)rrel : 31u, bcol = mj ? (uint32_t)jw : 31u;
                const uint32_t lim = min(a, bcol);
                const uint32_t ys = __vimin3_u32(y, a, bcol);
                const uint32_t cx = code_at((uint32_t)rrel - (mi ? ys : 0u), (uint32_t)jw - (mj ? ys : 0u));
                const uint32_t same = __ballot_sync(0xffffffffu, (cx == c0) & (ys == y));
                // >= 1: lane 31 looks at the current cell; <= 31: when every look-ahead agrees the last one still supplies c_next
                const uint32_t run = (uint32_t)__clz((int)(~same | 1u));
                // the cell the walk reaches next is the one the lane with y == run just looked at, if the window reached that far
                const uint32_t c_next = __shfl_sync(0xffffffffu, cx, (int)((31u - run) & 31u));
                push(i, j, c0 | (prevc << 2) | (run << 4), nops);     // labels, counters and op stores happen in the emit warps
                prevc = c0;
                nops += run;
                // the checked_sub move (algo.rs:412-417): run cells are interior, so neither index underflows
                i -= mi ? run : 0u;
                j -= mj ? run : 0u;
                rrel -= mi ? (int)run : 0;
                jw -= mj ? (int)run : 0;
                if (__builtin_expect(run <= lim, 1)) {
                    c0 = c_next;
                } else {
                    // the run ran into the window's edge: the next cell is a boundary cell (row or
                    // column 0), still inside the window (look it up), or in another window
                    if (i == 0u || j == 0u) {
                        walking = false;
                        break;
                    }
                    if (rrel < 0 || jw < 0) break;
                    c0 = code_at((uint32_t)rrel, (uint32_t)jw);
                }
                if (c0 == 3u) {
                    walking = false;
                    break;
                }
            }
            if (!walking) break;
        }
        // ---------------- boundary cells (algo.rs:195-220): row 0 holds only finite insert scores (code I), column 0 only
        // delete scores (code D); a local alignment stops on them (algo.rs:401-405); (0,0) is never emitted after a move
        // (algo.rs:419-421).  One long run each, cut into pieces the descriptor's run field holds.
        if (!left_band && !local && (i == 0u) != (j == 0u)) {
            const uint32_t c0 = (i == 0u) ? 1u : 2u;
            uint32_t left = (i == 0u) ? j : i;
            while (left) {
                const uint32_t run = min(left, 1u << 16);
                push(i, j, c0 | (prevc << 2) | (run << 4), nops);
                prevc = c0;
                nops += run;
                if (c0 == 1u) j -= run;
                else i -= run;
                left -= run;
            }
        }
        if (left_band && lane == 0) {
            atomicAdd(P.left_band, 1u);
            if (P.left_cell) P.left_cell[q] = make_uint2(i, j);   // compact storage: the host widens this pair's band to hold it
        }
        for (uint32_t e = 0; e < WALK_EMIT; ++e) push(0u, 0u, 3u, nops);   // end of path, one marker per emit warp
        nreq++;
        sts_volatile_uint4(req + nreq % WALK_REQ, make_uint4(0u, 0u, 0x80000000u, nreq));   // the loader warp may leave
    } else if (wid == 2) {
        // ================================================================ loader warp
        for (uint32_t seq = 1;; ++seq) {
            uint4 d;
            do {
                d = lds_volatile_uint4(req + seq % WALK_REQ);
            } while (d.w != seq);
            __syncwarp();
            if (d.z >> 31) break;
            const uint32_t p = d.x, s_ = d.y, r0 = d.z & 0xfffu, r1 = (d.z >> 12) & 0xfffu, b = (d.z >> 24) & 3u;
            uint32_t flag = 1u;
            if (P.tile_codes) flag = P.tile_codes[pd->tile_base + p * pd->S + s_];
            // the tile's codes: at its position in the table, or (compact storage) at its slot
            uint32_t ct = p * pd->S + s_;
            if (P.tile_slot) ct = P.tile_slot[pd->tile_base + ct];
            const uint32_t c0w = r0 / SPC;
            const uint32_t nch = (r1 + 31u) / SPC - c0w + 1u;
            GX_CHECK(P.check, b < WALK_NBUF && nch * 512u <= BUF_BYTES && (uint64_t)(c0w + nch) * 512 <= pd->tile_code_bytes &&
                                  pd->codes_off + (uint64_t)(ct + 1u) * pd->tile_code_bytes <= P.code_bytes, 23);
            const uint4 *tile = reinterpret_cast<const uint4 *>(P.codes + pd->codes_off + (uint64_t)ct * pd->tile_code_bytes) +
                                (size_t)c0w * 32 + lane;
            uint32_t dst = smem_u32(bufs + b * BUF_BYTES) + (uint32_t)lane * 16u;
            // a tile outside the code band holds no codes: post its flag only (the path warp gives up if it enters it)
            for (uint32_t q2 = 0; flag && q2 < nch; ++q2) {
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(tile + (size_t)q2 * 32) : "memory");
                dst += 32 * 16;
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncwarp();
            __threadfence_block();                            // every lane's copies before the ready word
            if (lane == 0) sts_volatile_u32(ready + b, seq | (flag ? 0u : 0x80000000u));
        }
    } else {
        // ================================================================ emit warps: descriptors e, e + 2, e + 4, ...
        const uint32_t e = (wid == 1) ? 0u : (uint32_t)wid - 2u;
        uint8_t *ops = P.ops + pd->ops_off;
        uint32_t nops_end = 0, n_match = 0, n_mis = 0, n_ext = 0, n_open = 0;
        uint32_t last_seq = 0, end_i = i, end_j = j;
        for (uint32_t seq = e;; seq += WALK_EMIT) {
            const uint32_t tag = (seq / WALK_RING + 1u) & 7u;
            uint4 d;
            do {
                d = lds_volatile_uint4(ring + seq % WALK_RING);
            } while ((d.x >> 29) != tag || (d.z >> 29) != tag);
            __syncwarp();                                 // every lane has its copy: the slot may be reused
            if (lane == 0) sts_volatile_u32(tail + e, seq + 1u);
            const uint32_t c0 = d.z & 3u;
            if (c0 == 3u) break;
            const uint32_t ri = d.x & 0x1fffffffu, rj = d.y;              // row indices stay below 2^29 (gx_check_scores)
            const uint32_t run = (d.z >> 4) & 0x1ffffffu, before = d.w;
            const bool diag = (c0 == 0u);
            const bool opens = !diag && c0 != ((d.z >> 2) & 3u);      // last_choice differs (algo.rs:373-379, 388-394)
            const uint32_t di = (c0 != 1u) ? 1u : 0u, dj = (c0 != 2u) ? 1u : 0u;
            const uint32_t ext = (c0 == 1u) ? 2u : 3u;          // Insert / Delete
            for (uint32_t base = 0; base < run; base += 32u) {
                const uint32_t x = base + (uint32_t)lane;
                const bool mine = x < run;
                const uint32_t ci = ri - (mine ? x * di : 0u), cj = rj - (mine ? x * dj : 0u);
                // labels.  Diagonal: is_match(i, j), Option<u8> equality with None == None (sequence.rs:113-114): the characters
                // AFTER the cell's own (0-based s1[i], s2[j]; algo.rs:354).  Gaps: open/extend from last_choice (algo.rs:373-379, 388-394).
                const bool lab = diag & mine;
                const int a = (lab && ci < m) ? (int)__ldg(s1 + ci) : -1;
                const int b = (lab && cj < n) ? (int)__ldg(s2 + cj) : -1;
                const uint32_t nm = (uint32_t)__popc(__ballot_sync(0xffffffffu, lab && a == b));
                const uint32_t gop = (x == 0u && opens) ? ext + 2u : ext;   // OpenInsert = 4, OpenDelete = 5
                const uint32_t op = diag ? ((a == b) ? 0u : 1u) : gop;
                GX_CHECK(P.check, !mine || ((uint64_t)before + x <= (uint64_t)m + n && pd->ops_off + before + x < P.ops_bytes), 22);
                if (mine) ops[before + x] = (uint8_t)op;
                n_match += nm;
                n_mis += diag ? min(32u, run - base) - nm : 0u;
            }
            n_open += opens ? 1u : 0u;
            n_ext += diag ? 0u : (opens ? run - 1u : run);
            last_seq = seq + 1u;
            nops_end = before + run;
            end_i = ri - (run - 1u) * di;                 // last emitted cell
            end_j = rj - (run - 1u) * dj;
        }
        if (lane == 0) {
            uint32_t *pp = part + e * 8u;
            pp[0] = n_match;
            pp[1] = n_mis;
            pp[2] = n_ext;
            pp[3] = n_open;
            pp[4] = last_seq;
            pp[5] = end_i;
            pp[6] = end_j;
            pp[7] = nops_end;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t *pl = part;                            // the emit warp that handled the last run
        uint32_t nm = 0, nx = 0, ne = 0, no = 0;
        for (uint32_t e = 0; e < WALK_EMIT; ++e) {
            const uint32_t *pe = part + e * 8u;
            if (pe[4] > pl[4]) pl = pe;
            nm += pe[0];
            nx += pe[1];
            ne += pe[2];
            no += pe[3];
        }
        if (pl[4] != 0u) {
            res.end_i = pl[5];
            res.end_j = pl[6];
            res.n_ops = pl[7];
        }
        res.matches = nm;
        res.mismatches = nx;
        res.gap_extensions = ne;
        res.opening_gaps = no;
        P.results[q] = res;
    }
}

}  // namespace gx
