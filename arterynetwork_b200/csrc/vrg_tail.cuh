// k_tail: everything of an iteration that follows the sweep, in ONE cooperative launch (vrg_run's production path).
//
// The serial tail of an iteration -- cancel rule + flips (VRG:165-230), statistics exchange + exit tests (VRG:91-117), halo
// exchange, the next decision table (VRG:79-87) -- used to be five to seven short launches (k_cancel, k_p2p_push_halo,
// k_p2p_wait_unpack_halo, k_quirks, k_p2p_stats / k_advance, k_table), each a few microseconds of work behind a launch
// boundary.  On an 8-GPU slab of config C3 that tail was 40 % of the iteration.  Here it is one grid of one block per SM, with
// two device-wide barriers between its three phases:
//
//   phase 1  cancel rule over the front rows, executed flips applied to S in place, integer histogram deltas      (all blocks)
//   ---- barrier ----
//   phase 2  block 0: statistics all-reduce over the peers' mailboxes (slabs) + exit tests + bookkeeping of the next sweep
//            blocks 1..: halo exchange of the executed-flip planes, cut into one chunk per block: store the chunk into the
//            neighbour's receive buffer, raise that chunk's flag, wait for the matching incoming chunk, apply it          (slabs)
//   ---- barrier ----
//   phase 3  decision table from the global histograms (one level per warp), order-dependence counters over the front rows
//
// Runs without label 4 in the input (the absorb step needs two more halo exchanges: that path keeps the separate kernels).
#pragma once
#include "vrg_p2p.cuh"

namespace vrg {

constexpr int TAIL_BLOCK = 1024;
constexpr int TAIL_WARPS = TAIL_BLOCK / 32;
constexpr int TAIL_STAGE_LEVELS = 4096;                // histograms up to this many levels are staged in shared memory (64 KB)
constexpr int MAX_CHUNKS = 256;                         // halo chunks per side (one per block of the tail grid)
constexpr int CHUNK_FLAGS = DONE_BASE + 8;              // flag words [side][MAX_CHUNKS] behind the ones of vrg_p2p.cuh
constexpr int FLAG_WORDS_ALL = CHUNK_FLAGS + 2 * MAX_CHUNKS;

// Device-wide barrier of a cooperative launch (all blocks resident).  bar[0] = arrival count, bar[1] = generation.
__device__ __forceinline__ void grid_barrier(unsigned int *bar, unsigned int nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile unsigned int *vgen = bar + 1;
        const unsigned int gen = *vgen;  // cannot move on before this block has arrived
        __threadfence();                 // release: this block's writes before its arrival
        if (atomicAdd(bar, 1u) == nblocks - 1) {
            atomicExch(bar, 0u);
            __threadfence();
            atomicAdd(bar + 1, 1u);
        } else {
            while (*vgen == gen) {}
        }
        __threadfence();                 // acquire: the other blocks' writes
    }
    __syncthreads();
}

// advance_state + prepare_sweep by one warp: a single thread walking the control block pays one L2 round trip per word (the
// separate k_advance took 3.6 us); here lane i < 16 fetches control word i and lane 16 + j the j-th counter of the global
// statistics, all at once, and lane 0 then applies the exit tests of VRG:91-104,118 and the bookkeeping of VRG:113-117.
__device__ __forceinline__ void advance_and_prepare_warp(const Params &p, int lane) {
    const long long *g = p.gstats + 2 * p.L;
    const long long v = lane < 16 ? __ldcg(p.ctrl + lane) : __ldcg(g + (lane - 16));
    const long long status = __shfl_sync(FULL, v, C_STATUS), apply = __shfl_sync(FULL, v, C_APPLY), tn = __shfl_sync(FULL, v, C_TRACE_N);
    const long long iter = __shfl_sync(FULL, v, C_ITER), itmax = __shfl_sync(FULL, v, C_ITER_MAX), sweeps = __shfl_sync(FULL, v, C_SWEEPS);
    const long long applied = __shfl_sync(FULL, v, C_APPLIED), maxseg = __shfl_sync(FULL, v, C_MAX_SEG);
    const long long nfl = __shfl_sync(FULL, v, 16 + ST_N_FLIPS), nin = __shfl_sync(FULL, v, 16 + ST_N_IN);
    const long long nout = __shfl_sync(FULL, v, 16 + ST_N_OUT), tup = __shfl_sync(FULL, v, 16 + ST_TIME_UP);
    if (lane != 0 || status != RUNNING) return;
    long long *c = p.ctrl;
    c[C_SWEEPS] = sweeps + 1;
    if (nfl == 0) { c[C_STATUS] = 0; return; }     // converged, VRG:91
    if (!apply) { c[C_STATUS] = 2; return; }       // max segment size, VRG:101
    p.trace[3 * tn] = nfl; p.trace[3 * tn + 1] = nin; p.trace[3 * tn + 2] = nout;
    c[C_TRACE_N] = tn + 1; c[C_APPLIED] = applied + 1; c[C_ITER] = iter + 1;
    if (iter + 1 > itmax) { c[C_STATUS] = 3; return; }  // VRG:58,118
    if (tup != 0) { c[C_STATUS] = 1; return; }          // VRG:97 on slabs (see advance_state)
    // prepare_sweep: the cap test of VRG:101 and the resets of what the next sweep accumulates
    c[C_APPLY] = nin < maxseg;
    p.lstats[2 * p.L + ST_N_FLIPS] = 0;
    front_list(p, (int)((sweeps + 1) & 1))[0] = 0;
    dirty_list(p, (int)((sweeps + 2) & 1))[0] = 0;
    c[C_NEXT_UNIT] = 0;
}

__device__ __forceinline__ unsigned long long tail_clock() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// The decision words of one table block: word w = 32 levels = the block's 32 warps.  Bit-identical to k_table (same terms in the
// same order: table_level_from), but with every load of the first word's sums in flight at once -- kernel-matrix row, the old
// decision word and the region sizes are requested before the histograms are staged, so the block pays about two L2 round trips
// instead of six.  t = index of this block among the T table blocks.
constexpr int TABLE_PRE = 8;   // kernel-matrix values per lane fetched ahead of the histogram staging (256 levels); the rest
                               // follows in batches of eight
__device__ __forceinline__ void table_words(const Params &p, int t, int T, long long next_sweep, int lane, int warp, double *s_hist,
                                            uint32_t *s_bits, int stage_hist) {
    const long long *g = p.gstats;
    int w = t;
    const int b0 = w * 32 + warp;
    double kv0[TABLE_PRE];
    const bool pre = p.kmat != nullptr && b0 < p.L;
#pragma unroll
    for (int k = 0; k < TABLE_PRE; ++k) {
        const int c = lane + 32 * k;
        kv0[k] = (pre && c < p.L) ? p.kmat[(size_t)b0 * p.L + c] : 0.0;
    }
    const double n_in = (double)__ldcg(g + 2 * p.L + ST_N_IN), n_out = (double)__ldcg(g + 2 * p.L + ST_N_OUT);
    uint32_t *bits = table_bits(p);
    uint32_t oldw = threadIdx.x == 0 ? __ldcg(bits + w) : 0u;
    if (stage_hist) {  // the two histograms once per block, as doubles, in shared memory: one coalesced round trip
        for (int i = threadIdx.x; i < 2 * p.L; i += TAIL_BLOCK) s_hist[i] = (double)__ldcg(g + i);
        __syncthreads();
    }
    auto hist = [&](int c, double &hi, double &ho) {
        if (stage_hist) { hi = s_hist[c]; ho = s_hist[p.L + c]; }
        else { hi = (double)__ldcg(g + c); ho = (double)__ldcg(g + p.L + c); }
    };
    for (bool first = true; w < p.LW; w += T, first = false) {
        const int b = w * 32 + warp;
        uint32_t bit = 0u;
        if (b < p.L) {
            if (first && pre) {  // table_level_from with the first TABLE_PRE terms per lane already in registers
                double hb, ob;
                hist(b, hb, ob);
                if (hb + ob != 0.0) {
                    double si = 0.0, so = 0.0;
#pragma unroll
                    for (int k = 0; k < TABLE_PRE; ++k) {
                        const int c = lane + 32 * k;
                        double hi = 0.0, ho = 0.0;
                        if (c < p.L) hist(c, hi, ho);
                        si += hi * kv0[k];
                        so += ho * kv0[k];
                    }
                    for (int c0 = lane + 32 * TABLE_PRE; c0 < p.L; c0 += 32 * TABLE_PRE) {
                        double kv[TABLE_PRE];
#pragma unroll
                        for (int k = 0; k < TABLE_PRE; ++k) {
                            const int c = c0 + 32 * k;
                            kv[k] = c < p.L ? p.kmat[(size_t)b * p.L + c] : 0.0;
                        }
#pragma unroll
                        for (int k = 0; k < TABLE_PRE; ++k) {
                            const int c = c0 + 32 * k;
                            double hi = 0.0, ho = 0.0;
                            if (c < p.L) hist(c, hi, ho);
                            si += hi * kv[k];
                            so += ho * kv[k];
                        }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        si += __shfl_xor_sync(FULL, si, o);
                        so += __shfl_xor_sync(FULL, so, o);
                    }
                    const double pi = si / n_in, po = so / n_out;  // VRG:81-82
                    if (lane == 0) { p.pin[b] = pi; p.pout[b] = po; }
                    bit = pi >= po ? 1u : 0u;  // ties go inside, VRG:87
                }
            } else bit = table_level_from(p, b, lane, n_in, n_out, hist);
        }
        if (!first && threadIdx.x == 0) oldw = __ldcg(bits + w);
        if (lane == 0) s_bits[warp] = bit << warp;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t word = 0;
#pragma unroll
            for (int i = 0; i < 32; ++i) word |= s_bits[i];
            if (word != oldw) { bits[w] = word; p.ctrl[C_FULL_SWEEP] = next_sweep + 1; }  // that sweep looks at every band voxel
        }
        __syncthreads();
    }
}

// dbg (profiling runs only, else nullptr): [0] launches, [1..5] nanoseconds block 0 spent in phase 1 / barrier / phase 2 /
// barrier / phase 3 ([6], [7]: k_tail_pipe's halo push and counters, the first two parts of its phase 2; [3] is then the wait +
// unpack), [9..15] the same for the last block; [16 + b], [16 + grid + b]: block b's phase 1 / phase 3.
template <int MODE, bool LATTICE, bool TIMED>
__global__ void __launch_bounds__(TAIL_BLOCK, 1) k_tail(Params p, P2P q, long long *gstats, unsigned int *gbar, int p2p,
                                                        int stage_hist, unsigned long long *dbg) {
    extern __shared__ double s_hist[];  // [2L] when stage_hist
    __shared__ long long s_ctl[4];
    __shared__ uint32_t s_bits[32];
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        s_ctl[0] = p.ctrl[C_STATUS]; s_ctl[1] = p.ctrl[C_APPLY]; s_ctl[2] = p.ctrl[C_SWEEPS]; s_ctl[3] = p.ctrl[C_EPOCH];
    }
    __syncthreads();
    // the control block only moves in phase 2, behind the first barrier: every block reads the same values here
    if (s_ctl[0] != RUNNING) return;
    const bool go = s_ctl[1] != 0;  // the cap of VRG:101 is tested before the flips are applied
    const int sweep = (int)s_ctl[2];
    const unsigned long long seq = ((unsigned long long)s_ctl[3] << 32) | (unsigned long long)(sweep + 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = (int)gridDim.x;
    const int gw = blockIdx.x * TAIL_WARPS + warp, nw = G * TAIL_WARPS;
    const int *fl = front_list(p, sweep & 1);
    const int nfront = go ? fl[0] : 0;
    // table blocks: the last T blocks of the grid, one decision word (32 levels) per block and pass
    const int T = min(p.LW, G - 1), t_idx = (int)blockIdx.x - (G - T);
    // blocks that count the order-dependence patterns in phase 2: all but block 0 and, on one GPU where the table is built in
    // phase 2 as well, the table blocks (unless that would leave fewer than half the grid)
    const int qblocks = (!p2p && G - 1 - T >= G / 2) ? G - 1 - T : G - 1;
    QuirkCounts qc;
    auto quirk_rows = [&](int first, int stride, bool boundary) {
        // rows whose neighbour planes are all own planes are counted in phase 2 (beside the statistics exchange), rows next to
        // a halo plane in phase 3 (after the halo exchange)
        for (int k = first; k < nfront; k += stride) {
            const int rr = fl[1 + k];
            const int sg = rr % p.nseg, t = rr / p.nseg, zl = t / p.Y;
            const bool at_halo = (zl - 1 < p.own_lo && zl - 1 >= p.valid_lo) || (zl + 1 >= p.own_hi && zl + 1 < p.valid_hi);
            if (at_halo == boundary) quirks_row(p, zl, t % p.Y, sg, lane, qc);
        }
    };
    const bool timing = TIMED && threadIdx.x == 0 && (blockIdx.x == 0 || (int)blockIdx.x == G - 1);
    unsigned long long *tdst = dbg + (blockIdx.x == 0 ? 0 : 8);
    unsigned long long t_prev = timing ? tail_clock() : 0ull;
    auto stamp = [&](int slot) {
        if (TIMED && timing) { const unsigned long long tc = tail_clock(); tdst[slot] += tc - t_prev; t_prev = tc; }
    };
    const unsigned long long tb0 = (TIMED && threadIdx.x == 0) ? tail_clock() : 0ull;
    if (TIMED && timing && blockIdx.x == 0) dbg[0] += 1;

    // ---- phase 1: cancel rule, flips, histogram deltas ------------------------------------------------------------
    if (go) {
        const bool dirty = p.dirty_lists && p.valid_lo == p.own_lo && p.valid_hi == p.own_hi;
        long long d_in = 0;
        // A warp with more than one row (the front holds more rows than the grid has warps) has the next row's list entry and
        // its own two words under way while it works on the current row.
        auto fetch = [&](int rr, uint32_t &s, uint32_t &f) {
            s = 0u; f = 0u;
            if (rr < 0) return;
            const int sg = rr % p.nseg, t = rr / p.nseg;
            const int c = sg * p.segw - 1 + lane;
            if (c >= 0 && c < p.XW) {
                const long long widx = (long long)(t / p.Y) * p.plane_words + (long long)(t % p.Y) * p.WP + c;
                s = p.S[widx]; f = p.F[widx];
            }
        };
        int k = gw;
        int rrA = k < nfront ? fl[1 + k] : -1, rrB = k + nw < nfront ? fl[1 + k + nw] : -1;
        uint32_t sA, fA, sB, fB;
        fetch(rrA, sA, fA);
        fetch(rrB, sB, fB);
        while (rrA >= 0) {
            const int kC = k + 2 * nw;
            const int rrC = kC < nfront ? fl[1 + kC] : -1;
            const int sg = rrA % p.nseg, t = rrA / p.nseg;
            cancel_row_loaded<MODE, LATTICE>(p, t / p.Y, t % p.Y, sg, lane, dirty, d_in, sA, fA);
            rrA = rrB; sA = sB; fA = fB;
            rrB = rrC;
            fetch(rrB, sB, fB);
            k += nw;
        }
        cancel_finish(p, d_in, lane);
    }
    stamp(1);
    if (TIMED) { __syncthreads(); if (threadIdx.x == 0) dbg[16 + blockIdx.x] += tail_clock() - tb0; }
    grid_barrier(gbar, gridDim.x);
    stamp(2);

    // ---- phase 2: statistics + exit tests (block 0); halo exchange, counters, on one GPU the table (the other blocks) ------
    if (blockIdx.x == 0) {
        bool ok = true;
        if (p2p) {
            const int par = (int)(seq & 1ull), n = 2 * p.L + ST_EXTRA;
            for (int r = 0; r < q.world; ++r) {
                long long *dst = q.peer_slots[r] + ((long long)par * q.world + q.rank) * q.slot_words;
                for (int i = threadIdx.x; i < n; i += TAIL_BLOCK) dst[i] = p.lstats[i];
            }
            __syncthreads();
            if (threadIdx.x == 0) s_ok = 1;
            if (threadIdx.x < q.world) __threadfence_system();  // the block's stores precede it through the barrier
            if (threadIdx.x < q.world) st_release_sys(q.peer_flags[threadIdx.x] + STATS_FLAGS + par * P2P_MAX_WORLD + q.rank, seq);
            __syncthreads();
            if (threadIdx.x < q.world && !p2p_wait(q.flags + STATS_FLAGS + par * P2P_MAX_WORLD + threadIdx.x, seq)) s_ok = 0;
            __threadfence_system();
            __syncthreads();
            ok = s_ok != 0;
            if (ok) {
                const long long *base = q.slots + (long long)par * q.world * q.slot_words;
                for (int i = threadIdx.x; i < n; i += TAIL_BLOCK) {
                    long long sum = 0;
                    for (int r = 0; r < q.world; ++r) sum += __ldcg(base + (long long)r * q.slot_words + i);
                    gstats[i] = sum;
                }
                __threadfence();
                __syncthreads();
            }
        }
        if (!ok) {
            if (threadIdx.x == 0) { p.ctrl[C_PEER_TIMEOUT] = 1; p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
        } else if (warp == 0) advance_and_prepare_warp(p, lane);  // exit tests, trace row, bookkeeping of the next sweep
    } else {
        // one GPU: the statistics are final behind the first barrier, so the next table is built here, beside the exit tests
        // (a table computed in the iteration that turns out to be the last one is the table of the final state)
        if (!p2p && t_idx >= 0) table_words(p, t_idx, T, (long long)sweep + 1, lane, warp, s_hist, s_bits, stage_hist);
        const int bq = (int)blockIdx.x - 1;
        const int first = bq * TAIL_WARPS + warp, stride = qblocks * TAIL_WARPS;
        if (go && !p2p) {
            if (bq < qblocks) quirk_rows(first, stride, false);
        } else if (go) {
            const long long n = (long long)HALO * p.plane_words;
            const int nch = min(G - 1, MAX_CHUNKS);
            const long long par_off = (long long)(seq & 1ull) * P2P_KINDS * 2 * n;
            const int j = bq;  // this block's chunk of the halo planes (blocks beyond MAX_CHUNKS have none)
            const long long lo = j < nch ? n * j / nch : 0, hi = j < nch ? n * (j + 1) / nch : 0;
            if (j < nch) {
#pragma unroll
                for (int side = 0; side < 2; ++side) {  // side 0: to the lower neighbour (lands in its "from above" region)
                    uint32_t *dst = q.peer_recv[side];
                    if (dst == nullptr) continue;
                    dst += par_off + ((long long)PK_F * 2 + (side ^ 1)) * n;
                    const uint32_t *src = p.F + (long long)(side == 0 ? p.own_lo : p.own_hi - HALO) * p.plane_words;
                    for (long long i = lo + threadIdx.x; i < hi; i += TAIL_BLOCK) dst[i] = __ldcg(src + i);
                }
                __syncthreads();  // the block's stores are ordered before thread 0's fence by the barrier (cumulativity)
                if (threadIdx.x == 0) {
                    __threadfence_system();
                    if (q.peer_recv[0]) st_release_sys(q.peer_flags[q.rank - 1] + CHUNK_FLAGS + 1 * MAX_CHUNKS + j, seq);
                    if (q.peer_recv[1]) st_release_sys(q.peer_flags[q.rank + 1] + CHUNK_FLAGS + 0 * MAX_CHUNKS + j, seq);
                }
            }
            quirk_rows(first, stride, false);  // while the neighbours' chunks travel
            if (j < nch) {
                if (threadIdx.x == 0) {
                    int ok = 1;
                    if (q.peer_recv[0] && !p2p_wait(q.flags + CHUNK_FLAGS + 0 * MAX_CHUNKS + j, seq)) ok = 0;
                    if (ok && q.peer_recv[1] && !p2p_wait(q.flags + CHUNK_FLAGS + 1 * MAX_CHUNKS + j, seq)) ok = 0;
                    if (!ok) { p.ctrl[C_PEER_TIMEOUT] = 1; p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
                    s_ok = ok;
                    __threadfence_system();
                }
                __syncthreads();
                if (s_ok) {
#pragma unroll
                    for (int side = 0; side < 2; ++side) {  // side 0: data from the lower neighbour -> my lower halo planes
                        if (q.peer_recv[side] == nullptr) continue;
                        const uint32_t *src = q.recv + par_off + ((long long)PK_F * 2 + side) * n;
                        const int z0 = side == 0 ? p.own_lo - HALO : p.own_hi;
                        uint32_t *fdst = p.F + (long long)z0 * p.plane_words, *sdst = p.S + (long long)z0 * p.plane_words;
                        for (long long i = lo + threadIdx.x; i < hi; i += TAIL_BLOCK) {
                            const uint32_t f = __ldcg(src + i);
                            fdst[i] = f;
                            if (f) {  // the halo copy of the segmented plane follows the neighbour slab
                                sdst[i] = __ldcg(sdst + i) ^ f;
                                const int zl = z0 + (int)(i / p.plane_words), y = (int)((i % p.plane_words) / p.WP), c = (int)(i % p.WP);
                                p.unitmap[unit_index(p, zl, y, c)] = 1;
                            }
                        }
                    }
                }
            }
        }
    }
    stamp(3);
    if (!p2p) {  // one GPU: nothing is left to wait for
        if (go) quirks_finish(p, qc, lane);
        return;
    }
    grid_barrier(gbar, gridDim.x);
    stamp(4);
    const unsigned long long tb3 = (TIMED && threadIdx.x == 0) ? tail_clock() : 0ull;

    // ---- phase 3 (slabs): next decision table from the global statistics; counters of the rows next to a halo plane ---------
    const long long status = *(volatile long long *)&p.ctrl[C_STATUS];
    if (status == RUNNING && t_idx >= 0) table_words(p, t_idx, T, (long long)sweep + 1, lane, warp, s_hist, s_bits, stage_hist);
    if (go && status != EXIT_PEER_TIMEOUT) quirk_rows(gw, nw, true);
    if (go) quirks_finish(p, qc, lane);
    __syncthreads();
    stamp(5);
    if (TIMED && threadIdx.x == 0) dbg[16 + gridDim.x + blockIdx.x] += tail_clock() - tb3;
}

// =====================================================================================================================
// The pipelined run: statistics, exit tests and the next decision table travel BESIDE the next sweep.
//
// The decision table depends on the regions only through their normalised Parzen sums, and those barely move from one
// update to the next: on the bench phantom not one decision bit changes in 118 updates.  So sweep k+1 does not wait for the
// table of update k: it starts right behind the tail kernel of update k and reads the table it already has, while on a
// second stream two small kernels (they fit on the SMs beside the sweep's blocks) exchange update k's statistics, run the
// exit tests and build the table of update k+1 into the OTHER table buffer.  The tail kernel of update k+1 waits for them
// (stream event) and looks at the result before it touches any state:
//   * run over (converged, cap reached, ...)            -> it returns; the sweep was one too many and is not counted
//   * a decision bit changed                            -> it switches the table buffers, marks the next sweep `full` and
//                                                          returns; the stream's next sweep / tail pair redoes update k+1
//   * otherwise (the rule)                              -> update k+1 is applied exactly as the in-order run would
// The sweep only writes flip flags, row flags and the front list, all of which the redone sweep rewrites; nothing it writes
// is read by the statistics kernels (the flip count of update k is set aside in ST_N_FLIPS_SNAP by the tail kernel).
// Results are identical to the in-order run by construction: every applied update used the table of the statistics before it.
// What the iteration waits for is down to: sweep -> cancel rule -> halo exchange with the two neighbours.  The all-to-all
// statistics exchange has a whole sweep of slack, which also absorbs the ranks' skew.
//
// k_tail_pipe: phase 1 cancel rule + flips; barrier; phase 2 halo exchange (slabs) + order-dependence counters; on slabs a
// second barrier and the counters of the rows next to a halo plane; bookkeeping of the next sweep.
template <int MODE, bool LATTICE, bool TIMED>
__global__ void __launch_bounds__(TAIL_BLOCK, 1) k_tail_pipe(Params p, P2P q, unsigned int *gbar, int p2p, unsigned long long *dbg) {
    __shared__ long long s_ctl[6];
    if (threadIdx.x == 0) {
        s_ctl[0] = p.ctrl[C_STATUS]; s_ctl[1] = p.ctrl[C_APPLY]; s_ctl[2] = p.ctrl[C_SWEEPS]; s_ctl[3] = p.ctrl[C_EPOCH];
        s_ctl[4] = p.ctrl[C_TABLE_NEW]; s_ctl[5] = p.ctrl[C_TABLE_BUF];
    }
    __syncthreads();
    // nothing else runs on this device's handle while the tail kernel does: the control words are stable
    if (s_ctl[0] != RUNNING) return;  // the run ended with the previous update; the sweep in front of this kernel is not counted
    const int sweep = (int)s_ctl[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = (int)gridDim.x;
    if (s_ctl[4] != 0) {
        // the sweep read a table that update `sweep - 1` has changed: switch to the new one, redo the sweep (a full one)
        grid_barrier(gbar, gridDim.x);  // every block has read the control words
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            p.ctrl[C_TABLE_BUF] = 1 - s_ctl[5];
            p.ctrl[C_TABLE_NEW] = 0;
            p.ctrl[C_FULL_SWEEP] = sweep + 1;
            p.ctrl[C_TAIL_APPLIED] = 0;
            p.ctrl[C_REDOS] += 1;
            p.lstats[2 * p.L + ST_N_FLIPS] = 0;
            front_list(p, sweep & 1)[0] = 0;
            p.ctrl[C_NEXT_UNIT] = 0;
        }
        return;
    }
    const bool go = s_ctl[1] != 0;  // the cap of VRG:101 is tested before the flips are applied
    const int gw = blockIdx.x * TAIL_WARPS + warp, nw = G * TAIL_WARPS;
    const int *fl = front_list(p, sweep & 1);
    const int nfront = go ? fl[0] : 0;
    QuirkCounts qc;
    auto quirk_rows = [&](bool boundary) {
        for (int k = gw; k < nfront; k += nw) {
            const int rr = fl[1 + k];
            const int sg = rr % p.nseg, t = rr / p.nseg, zl = t / p.Y;
            const bool at_halo = (zl - 1 < p.own_lo && zl - 1 >= p.valid_lo) || (zl + 1 >= p.own_hi && zl + 1 < p.valid_hi);
            if (at_halo == boundary) quirks_row(p, zl, t % p.Y, sg, lane, qc);
        }
    };
    const bool timing = TIMED && threadIdx.x == 0 && (blockIdx.x == 0 || (int)blockIdx.x == G - 1);
    unsigned long long *tdst = dbg + (blockIdx.x == 0 ? 0 : 8);
    unsigned long long t_prev = timing ? tail_clock() : 0ull;
    auto stamp = [&](int slot) {
        if (TIMED && timing) { const unsigned long long tc = tail_clock(); tdst[slot] += tc - t_prev; t_prev = tc; }
    };
    const unsigned long long tb0 = (TIMED && threadIdx.x == 0) ? tail_clock() : 0ull;
    if (TIMED && timing && blockIdx.x == 0) dbg[0] += 1;

    // ---- phase 1: cancel rule, flips, histogram deltas ------------------------------------------------------------
    if (go) {
        const bool dirty = p.dirty_lists && p.valid_lo == p.own_lo && p.valid_hi == p.own_hi;
        long long d_in = 0;
        auto fetch = [&](int rr, uint32_t &s, uint32_t &f) {
            s = 0u; f = 0u;
            if (rr < 0) return;
            const int sg = rr % p.nseg, t = rr / p.nseg;
            const int c = sg * p.segw - 1 + lane;
            if (c >= 0 && c < p.XW) {
                const long long widx = (long long)(t / p.Y) * p.plane_words + (long long)(t % p.Y) * p.WP + c;
                s = p.S[widx]; f = p.F[widx];
            }
        };
        int k = gw;
        int rrA = k < nfront ? fl[1 + k] : -1, rrB = k + nw < nfront ? fl[1 + k + nw] : -1;
        uint32_t sA, fA, sB, fB;
        fetch(rrA, sA, fA);
        fetch(rrB, sB, fB);
        while (rrA >= 0) {
            const int kC = k + 2 * nw;
            const int rrC = kC < nfront ? fl[1 + kC] : -1;
            const int sg = rrA % p.nseg, t = rrA / p.nseg;
            cancel_row_loaded<MODE, LATTICE>(p, t / p.Y, t % p.Y, sg, lane, dirty, d_in, sA, fA);
            rrA = rrB; sA = sB; fA = fB;
            rrB = rrC;
            fetch(rrB, sB, fB);
            k += nw;
        }
        cancel_finish(p, d_in, lane);
    }
    stamp(1);
    if (TIMED) { __syncthreads(); if (threadIdx.x == 0) dbg[16 + blockIdx.x] += tail_clock() - tb0; }
    grid_barrier(gbar, gridDim.x);
    stamp(2);

    // ---- phase 2: halo exchange with the two neighbour slabs; order-dependence counters ---------------------------------
    if (go && !p2p) quirk_rows(false);
    else if (go) {
        // Halo exchange, self-validating: every 32-bit word of the two boundary planes travels as one 8-byte store that
        // carries the update's tag in its upper half (what NCCL calls the LL protocol).  No fence and no flag: a system-scope
        // fence behind stores to a peer costs a full NVLink round trip per block (8 us measured here), an 8-byte store is
        // visible as a whole.  The receiver polls each slot until the tag matches.  Slots are double-buffered by update parity
        // (a neighbour may be one update ahead); a tag never repeats within 2048 runs x 2^20 updates.
        const long long n = (long long)HALO * p.plane_words;
        const unsigned long long tag = (unsigned long long)((((uint32_t)s_ctl[3] & 0x7FFu) << 20) | ((uint32_t)(sweep + 1) & 0xFFFFFu) | 0x80000000u);
        const long long par_off = (long long)((sweep + 1) & 1) * 2 * n;
        const long long lo = n * blockIdx.x / G, hi = n * (blockIdx.x + 1) / G;  // this block's chunk of the halo planes
#pragma unroll
        for (int side = 0; side < 2; ++side) {  // side 0: to the lower neighbour (lands in its "from above" region)
            if (q.peer_recv[side] == nullptr) continue;
            unsigned long long *dst = p2p_ll_region(q.peer_recv[side], n) + par_off + (long long)(side ^ 1) * n;
            const uint32_t *src = p.F + (long long)(side == 0 ? p.own_lo : p.own_hi - HALO) * p.plane_words;
            for (long long i = lo + threadIdx.x; i < hi; i += TAIL_BLOCK)
                st_relaxed_sys(dst + i, (tag << 32) | (unsigned long long)__ldcg(src + i));
        }
        stamp(6);
        quirk_rows(false);  // while the neighbours' words travel
        stamp(7);
        bool ok = true;
#pragma unroll
        for (int side = 0; side < 2; ++side) {  // side 0: data from the lower neighbour -> my lower halo planes
            if (q.peer_recv[side] == nullptr) continue;
            const unsigned long long *src = p2p_ll_region(q.recv, n) + par_off + (long long)side * n;
            const int z0 = side == 0 ? p.own_lo - HALO : p.own_hi;
            uint32_t *fdst = p.F + (long long)z0 * p.plane_words, *sdst = p.S + (long long)z0 * p.plane_words;
            for (long long i = lo + threadIdx.x; i < hi; i += TAIL_BLOCK) {
                unsigned long long v = ld_relaxed_sys(src + i);
                if ((v >> 32) != tag) {
                    const long long t0 = clock64();
                    while (((v = ld_relaxed_sys(src + i)) >> 32) != tag) {
                        if (clock64() - t0 > P2P_SPIN_LIMIT) { ok = false; break; }
                        __nanosleep(32);
                    }
                    if (!ok) break;
                }
                const uint32_t f = (uint32_t)v;
                fdst[i] = f;
                if (f) {  // the halo copy of the segmented plane follows the neighbour slab
                    sdst[i] = __ldcg(sdst + i) ^ f;
                    const int zl = z0 + (int)(i / p.plane_words), y = (int)((i % p.plane_words) / p.WP), c = (int)(i % p.WP);
                    p.unitmap[unit_index(p, zl, y, c)] = 1;
                }
            }
        }
        if (!ok) { p.ctrl[C_PEER_TIMEOUT] = 1; p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
    }
    stamp(3);
    if (p2p) {
        grid_barrier(gbar, gridDim.x);
        stamp(4);
        if (go) quirk_rows(true);  // rows next to a halo plane: their neighbours' flips have arrived
    }
    if (go) quirks_finish(p, qc, lane);
    // bookkeeping of the next sweep (the other blocks read the control words at their start and are past them)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        p.lstats[2 * p.L + ST_N_FLIPS_SNAP] = p.lstats[2 * p.L + ST_N_FLIPS];  // the sweep's atomics are complete
        p.lstats[2 * p.L + ST_N_FLIPS] = 0;
        p.ctrl[C_SWEEPS] = sweep + 1;
        front_list(p, (sweep + 1) & 1)[0] = 0;
        dirty_list(p, (sweep + 2) & 1)[0] = 0;
        p.ctrl[C_NEXT_UNIT] = 0;
        p.ctrl[C_TAIL_APPLIED] = 1;
    }
    __syncthreads();
    stamp(5);
}

// k_async_stats (second stream, one small block beside the running sweep): the statistics all-reduce of the update the tail
// kernel just applied (slabs), then the exit tests of VRG:91-104,118 and the loop bookkeeping of VRG:113-117.
constexpr int ASYNC_BLOCK = 256;  // these blocks have to find room on SMs the sweep's blocks occupy: see k_sweep_dense_slim
__global__ void __launch_bounds__(ASYNC_BLOCK) k_async_stats(Params p, P2P q, long long *gstats, int p2p) {
    __shared__ int s_ok;
    if (p.ctrl[C_STATUS] != RUNNING || !p.ctrl[C_TAIL_APPLIED]) return;
    const long long k = p.ctrl[C_SWEEPS] - 1;  // the update just applied (the tail kernel moved C_SWEEPS on)
    const unsigned long long seq = ((unsigned long long)p.ctrl[C_EPOCH] << 32) | (unsigned long long)(k + 1);
    bool ok = true;
    if (p2p) {
        const int par = (int)(seq & 1ull), n = 2 * p.L + ST_EXTRA;
        for (int r = 0; r < q.world; ++r) {
            long long *dst = q.peer_slots[r] + ((long long)par * q.world + q.rank) * q.slot_words;
            for (int i = threadIdx.x; i < n; i += ASYNC_BLOCK) dst[i] = __ldcg(p.lstats + i);
        }
        __syncthreads();
        if (threadIdx.x == 0) s_ok = 1;
        if (threadIdx.x < q.world) __threadfence_system();  // the block's stores precede it through the barrier
        if (threadIdx.x < q.world) st_release_sys(q.peer_flags[threadIdx.x] + STATS_FLAGS + par * P2P_MAX_WORLD + q.rank, seq);
        __syncthreads();
        if (threadIdx.x < q.world && !p2p_wait(q.flags + STATS_FLAGS + par * P2P_MAX_WORLD + threadIdx.x, seq)) s_ok = 0;
        __threadfence_system();
        __syncthreads();
        ok = s_ok != 0;
        if (ok) {
            const long long *base = q.slots + (long long)par * q.world * q.slot_words;
            for (int i = threadIdx.x; i < n; i += ASYNC_BLOCK) {
                long long sum = 0;
                for (int r = 0; r < q.world; ++r) sum += __ldcg(base + (long long)r * q.slot_words + i);
                gstats[i] = sum;
            }
            __threadfence();
            __syncthreads();
        }
    }
    if (!ok) {
        if (threadIdx.x == 0) { p.ctrl[C_PEER_TIMEOUT] = 1; p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
        return;
    }
    if (threadIdx.x < 32) {  // advance_state by one warp; C_SWEEPS and the sweep's accumulators belong to the tail kernel
        const int lane = threadIdx.x;
        const long long *g = p.gstats + 2 * p.L;
        const long long v = lane < 16 ? __ldcg(p.ctrl + lane) : __ldcg(g + (lane - 16));
        const long long apply = __shfl_sync(FULL, v, C_APPLY), tn = __shfl_sync(FULL, v, C_TRACE_N);
        const long long iter = __shfl_sync(FULL, v, C_ITER), itmax = __shfl_sync(FULL, v, C_ITER_MAX);
        const long long applied = __shfl_sync(FULL, v, C_APPLIED), maxseg = __shfl_sync(FULL, v, C_MAX_SEG);
        const long long nfl = __shfl_sync(FULL, v, 16 + ST_N_FLIPS_SNAP), nin = __shfl_sync(FULL, v, 16 + ST_N_IN);
        const long long nout = __shfl_sync(FULL, v, 16 + ST_N_OUT), tup = __shfl_sync(FULL, v, 16 + ST_TIME_UP);
        if (lane != 0) return;
        long long *c = p.ctrl;
        if (nfl == 0) { c[C_STATUS] = 0; return; }     // converged, VRG:91
        if (!apply) { c[C_STATUS] = 2; return; }       // max segment size, VRG:101
        p.trace[3 * tn] = nfl; p.trace[3 * tn + 1] = nin; p.trace[3 * tn + 2] = nout;
        c[C_TRACE_N] = tn + 1; c[C_APPLIED] = applied + 1; c[C_ITER] = iter + 1;
        if (iter + 1 > itmax) { c[C_STATUS] = 3; return; }  // VRG:58,118
        if (tup != 0) { c[C_STATUS] = 1; return; }          // VRG:97 on slabs (see advance_state)
        c[C_APPLY] = nin < maxseg;                          // the cap of VRG:101 for the next update
    }
}

// k_async_table (second stream, behind k_async_stats): the decision table of the new statistics into the table buffer the
// sweeps do NOT read; raises C_TABLE_NEW if a bit differs from the current one.  One decision word (32 levels) per block of
// eight warps -- its latency hides behind the sweep, its footprint has to fit beside the sweep's blocks.
__global__ void __launch_bounds__(ASYNC_BLOCK) k_async_table(Params p) {
    __shared__ uint32_t s_bits[ASYNC_BLOCK / 32];
    if (p.ctrl[C_STATUS] != RUNNING || !p.ctrl[C_TAIL_APPLIED]) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, w = blockIdx.x;
    uint32_t mine = 0u;
    for (int i = 0; i < 32 / (ASYNC_BLOCK / 32); ++i) {
        const int j = warp * (32 / (ASYNC_BLOCK / 32)) + i, b = w * 32 + j;
        if (b < p.L) mine |= table_level(p, b, lane) << j;
    }
    if (lane == 0) s_bits[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t word = 0;
#pragma unroll
        for (int i = 0; i < ASYNC_BLOCK / 32; ++i) word |= s_bits[i];
        const long long cur = p.ctrl[C_TABLE_BUF];
        p.dbits[(size_t)(1 - cur) * p.LW + w] = word;
        if (word != p.dbits[(size_t)cur * p.LW + w]) p.ctrl[C_TABLE_NEW] = 1;
    }
}

}  // namespace vrg
