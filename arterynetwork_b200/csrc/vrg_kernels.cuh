// Device code of the B200-native variational region growing path (sm_100a).
//
// State is bit-packed along x: one uint32 word = 32 voxels of one row.  Planes:
//   S  segmented (updated in place)          E  excluded, label 4 (only if the input has any)
//   F  flip flags of the current iteration   C  cancelled additions (only with E)
// plus one byte per (row, 30-word segment) saying whether its F words are non-zero, so that the
// kernels after the sweep touch only rows at the moving front.  The reference's label alphabet
// (VRG:21) is a function of (S, E) and the 26-neighbourhood; it is materialised on download.
//
// Per iteration (reference: Code/variationalRegionGrowing.py, VRG:line):
//   k_table   region histograms -> normalised Parzen sums per level -> decision bit      VRG:79-87,151-155
//   k_sweep*  the stencil sweep: bands from S (26-neighbourhood), decision per voxel, F   VRG:87-88,139-145
//   k_cancel  front rows: cancel rule, executed flips applied to S in place, histogram deltas   VRG:173,183-190,198,201,232-247
//   k_absorb  label 4 -> 3 around flips (only when the input holds label 4)               VRG:167-168,177-179
//   k_flip_halo  (slab runs) S ^= F on the halo planes after the flip exchange
//   k_advance exit tests and trace row                                                    VRG:91-117
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace vrg {

constexpr int HALO = 2;
constexpr int WORDS_PER_WARP = 30;  // a warp covers up to 30 output words + 1 halo word on each side (rows are cut into
                                    // nseg segments of equal width segw <= 30: 64 words are 22+22+20, not 30+30+4)
constexpr int ROWS_PER_UNIT = 16;   // rows a warp slides over per work unit of the sweep
constexpr int BLOCK = 256;
constexpr int WARPS = BLOCK / 32;
constexpr unsigned FULL = 0xFFFFFFFFu;
// dense sweep: per-warp ring of TMA bulk-copy stages, one stage = the fp64 intensities of one row segment
constexpr int DENSE_WARPS = 14;
constexpr int DENSE_STAGES = 2;
constexpr int STAGE_BYTES = WORDS_PER_WARP * 32 * 8;

enum { ST_N_IN = 0, ST_N_OUT = 1, ST_N_EXCL = 2, ST_N_FLIPS = 3, ST_N_BAND = 4, ST_BAD_LABEL = 5, ST_NONFINITE = 6, ST_TIME_UP = 7,
       // cumulative counts of the flip patterns on which the reference's result depends on its list order (k_quirks)
       ST_Q_CANCELLED = 8, ST_Q_ADD_INSIDE = 9, ST_Q_REM_OUTSIDE = 10, ST_Q_REPROMOTED = 11,
       ST_N_FLIPS_SNAP = 12,  // pipelined run (vrg_tail.cuh): the flip count of the update just applied, set aside by the tail kernel
                              // while the next sweep already counts into ST_N_FLIPS
       ST_EXP_EVALS = 13,     // continuous mode: Parzen kernel evaluations (fp64 exp) so far -- its roofline is the exp rate
       ST_EXTRA = 16 };
enum { C_STATUS = 0, C_ITER = 1, C_ITER_MAX = 2, C_MAX_SEG = 3, C_APPLY = 4, C_APPLIED = 5, C_TRACE_N = 6, C_SWEEPS = 7, C_FULL_SWEEP = 8,
       C_EPOCH = 9, C_PEER_TIMEOUT = 10, C_HALO_SEQ = 11, C_HALO_GO = 12,  // 9..12: slab runs (vrg_p2p.cuh)
       // C_FULL_SWEEP: 1 + index of the latest sweep that must look at every band voxel (first sweep of a run, a sweep behind a
       // changed decision table, a sweep behind caller-chosen flips); every other band / index sweep is incremental.  A stamp,
       // not a flag: whoever builds a table writes it, nobody has to clear it.
       C_NEXT_UNIT = 13,  // dense sweep: work-unit counter (units beyond the statically assigned ones are handed out dynamically)
       // pipelined run (vrg_tail.cuh): which of the two decision-table buffers the sweeps read; `the table built beside the last
       // sweep differs from the one it read`; `the last tail kernel applied its update` (statistics kernels have work)
       C_TABLE_BUF = 14, C_TABLE_NEW = 15, C_TAIL_APPLIED = 16,
       C_REDOS = 17,  // sweeps of the pipelined run that were repeated because the table changed beside them
       C_REFRESHES = 18,  // dense sweeps that evaluated every decision bit from the intensities (the others read them from Dc)
       C_WORDS = 24 };
constexpr long long RUNNING = -1;

enum { MODE_F64_DENSE = 0, MODE_F64_BAND = 1, MODE_INDEX = 2, MODE_CONT = 3 };  // MODE_CONT: no level table (vrg_parzen.cuh)

struct Params {
    // geometry
    int Y, X, XW, WP, nseg, segw;    // rows, voxels/row, words/row, word pitch, warp segments per row, words per segment (<= 30)
    int nzl;                          // local planes incl. halos
    int dense_rows;                   // rows per work unit of the dense sweep (8 on large volumes, 4 on thin slabs)
    int dirty_lists;                  // 1: k_sweep_band's incremental pass wants the dirty-row lists (k_cancel builds them)
    int own_lo, own_hi;               // local plane range owned
    int valid_lo, valid_hi;           // local planes that lie inside the global volume
    uint32_t tail_mask;               // valid bits of word XW-1
    long long plane_words;            // Y * WP
    long long plane_vox;              // Y * X
    // state
    uint32_t *S, *E, *F, *C;          // E, C: nullptr when the run never had label 4
    uint32_t *Cq;                     // cancelled additions of the front rows (always valid; == C when C != nullptr)
    uint8_t *rowflag;                 // [nzl * Y * nseg]
    uint8_t *unitmap;                 // [nzl * nyb * nseg]: 1 if the sweep unit ever held a segmented voxel (never cleared)
    int *dirty;                       // 2 x [front_cap]: rows the next incremental sweep must re-evaluate (built by k_flip)
    int *front;                       // 2 x [front_cap]: [0] = count, then the own-plane rows that flip in this sweep;
    int front_cap;                    //   sweep k writes list k & 1, the next sweep reads it as its dirty seed
    int *stamp;                       // [nzl * Y * nseg]: sweep number that last claimed the row (incremental pass)
    const double *data;               // fp64 intensities, local planes
    const uint16_t *index;            // level index volume (MODE_INDEX)
    // levels / table
    int L;                            // table size
    int LW;                           // ceil(L / 32)
    int lattice;                      // 1: index = rint((v - lev0) * inv_step)
    double lev0, inv_step;
    const double *levels;             // [L]
    const double *kmat;               // [L][L] Parzen kernel values A*exp(-0.5*H*(lev_b-lev_c)^2), or nullptr (L too large)
    uint32_t *dbits;                  // 2 x [LW]: decision bits; ctrl[C_TABLE_BUF] says which buffer is current (always 0 outside
                                      // the pipelined run, which builds the next table in the other one beside the running sweep)
    double *pin, *pout;               // [L] normalised Parzen sums of the last table
    double mhH;                       // -0.5 * H
    long long *lstats;                // local  [2L + ST_EXTRA]
    const long long *gstats;          // global [2L + ST_EXTRA] (aliases lstats on one GPU)
    long long *ctrl;                  // [C_WORDS]
    long long *trace;                 // [3 * (iter_max + 2)]
    uint32_t *Dc;                     // F64_DENSE: decision bit-plane (layout of S) written by the last refresh sweep, or nullptr
                                      // (switch VRG_NO_DCACHE: every dense sweep is a refresh).  Last: in front of `index` it
                                      // moved the later fields and k_sweep_dense<true> lost 14 registers and 20 % of its speed
};

__device__ __forceinline__ uint32_t *table_bits(const Params &p) { return p.dbits + (size_t)p.ctrl[C_TABLE_BUF] * p.LW; }
__device__ __forceinline__ int *front_list(const Params &p, int which) { return p.front + (size_t)which * p.front_cap; }
__device__ __forceinline__ int *dirty_list(const Params &p, int which) { return p.dirty + (size_t)which * p.front_cap; }

__device__ __forceinline__ uint32_t valid_mask(const Params &p, int c) {
    return c < p.XW - 1 ? 0xFFFFFFFFu : (c == p.XW - 1 ? p.tail_mask : 0u);
}

// x-dilation of a row of words held one-per-lane (lane l = column c0 + l)
__device__ __forceinline__ uint32_t dilate_x1(uint32_t v) {
    const uint32_t l = __shfl_up_sync(FULL, v, 1), r = __shfl_down_sync(FULL, v, 1);
    return v | __funnelshift_l(l, v, 1) | __funnelshift_r(v, r, 1);
}
// same for a warp whose 32 lanes ARE the row (no halo lanes): nothing lies beyond lane 0 and lane 31
__device__ __forceinline__ uint32_t dilate_x1_row(uint32_t v, int lane) {
    uint32_t l = __shfl_up_sync(FULL, v, 1), r = __shfl_down_sync(FULL, v, 1);
    if (lane == 0) l = 0u;
    if (lane == 31) r = 0u;
    return v | __funnelshift_l(l, v, 1) | __funnelshift_r(v, r, 1);
}
__device__ __forceinline__ uint32_t dilate_x2(uint32_t v) {
    const uint32_t l = __shfl_up_sync(FULL, v, 1), r = __shfl_down_sync(FULL, v, 1);
    return v | __funnelshift_l(l, v, 1) | __funnelshift_r(v, r, 1) | __funnelshift_l(l, v, 2) | __funnelshift_r(v, r, 2);
}

// 32x32 bit-matrix transpose across a warp: in = row `lane`, out = column `lane` (5 butterfly steps)
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) {
        const uint32_t m = k == 16 ? 0x0000FFFFu : k == 8 ? 0x00FF00FFu : k == 4 ? 0x0F0F0F0Fu : k == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(FULL, x, k);
        // lanes with bit k clear keep their low half-blocks and take the partner's low half-blocks as high ones
        x = (lane & k) ? ((x & ~m) | ((y >> k) & m)) : ((x & m) | ((y << k) & ~m));
    }
    return x;
}

// intensity -> table slot.  LATTICE: levels sit on lev0 + k*step, one DADD + one DFMA (round-to-nearest via the
// 2^52+2^51 trick: the integer lands in the low word).  Otherwise a binary search over the sorted levels.
template <bool LATTICE>
__device__ __forceinline__ int level_of(const Params &p, double v) {
    if (LATTICE) return __double2loint(__fma_rn(v - p.lev0, p.inv_step, 6755399441055744.0));
    int lo = 0, hi = p.L - 1;
    v += 0.0;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (p.levels[m] < v) lo = m + 1; else hi = m;
    }
    return lo;
}

template <int MODE, bool LATTICE>
__device__ __forceinline__ int level_at(const Params &p, long long vox) {
    if (MODE == MODE_INDEX) return p.index[vox];
    return level_of<LATTICE>(p, p.data[vox]);
}

__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

__device__ __forceinline__ long long unit_index(const Params &p, int zl, int y, int c) {
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    return ((long long)zl * nyb + y / ROWS_PER_UNIT) * p.nseg + c / p.segw;
}
// A sweep unit (one plane, ROWS_PER_UNIT rows, 30 words) can hold a band voxel only if it or one of its 26 neighbour
// units (z, y-block, x-segment) holds a segmented voxel: far from every vessel the full band sweep skips the unit
// after 27 byte loads (one per lane).
__device__ __forceinline__ bool unit_near_segmented(const Params &p, int zl, int y0, int sg, int lane) {
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    bool hit = false;
    if (lane < 27) {
        const int zz = zl + lane / 9 - 1, yb = y0 / ROWS_PER_UNIT + (lane / 3) % 3 - 1, ss = sg + lane % 3 - 1;
        if (zz >= p.valid_lo && zz < p.valid_hi && yb >= 0 && yb < nyb && ss >= 0 && ss < p.nseg)
            hit = p.unitmap[((long long)zz * nyb + yb) * p.nseg + ss] != 0;
    }
    return __ballot_sync(FULL, hit) != 0u;
}

// Parzen kernel matrix of a level set (symmetric: (lev_c - lev_b)^2 is exact either way round)
__global__ void __launch_bounds__(BLOCK) k_kmat(Params p, double *kmat) {
    const long long n = (long long)p.L * p.L;
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) {
        const double diff = p.levels[i % p.L] - p.levels[i / p.L];
        kmat[i] = 0.3989422804014327 * exp(p.mhH * (diff * diff));
    }
}

// ---------------------------------------------------------------------------------------------
// k_table: one block per 32 levels; a warp sums one level's two Parzen sums over all levels.
// Fixed order: lane-strided partial sums, then an xor-shuffle tree -> deterministic.
constexpr int TABLE_BLOCK = 1024;  // 32 warps: one level per warp, one decision word per block

// loop bookkeeping in front of a sweep (one thread): the cap test of VRG:101 and the resets of what the sweep accumulates
__device__ __forceinline__ void prepare_sweep(const Params &p) {
    p.ctrl[C_APPLY] = p.gstats[2 * p.L + ST_N_IN] < p.ctrl[C_MAX_SEG];  // cap is tested before the flips are applied, VRG:101
    p.lstats[2 * p.L + ST_N_FLIPS] = 0;
    front_list(p, (int)(p.ctrl[C_SWEEPS] & 1))[0] = 0;
    dirty_list(p, (int)((p.ctrl[C_SWEEPS] + 1) & 1))[0] = 0;  // this iteration's flips fill it for the next sweep
    p.ctrl[C_NEXT_UNIT] = 0;
}

// the two normalised Parzen sums of level b (one warp; fixed order: lane-strided partial sums in increasing level order, then
// an xor tree) and its decision bit.  A level absent from both regions is never looked up: bit 0, sums untouched.
// hist(c, hi, ho) hands out the two region counts of level c as doubles (global statistics, or a copy staged in shared
// memory).  Loads come in batches with nothing conditional between them: a `skip the empty level` branch in front of
// the kernel-matrix load made every step two dependent L2 round trips, 15 us for 468 levels.  Batches of eight.  (Adding the +0.0 of an empty
// level changes no bit of the sums.)
template <typename Hist>
__device__ __forceinline__ uint32_t table_level_from(const Params &p, int b, int lane, double n_in, double n_out, Hist hist) {
    {
        double hb, ob;
        hist(b, hb, ob);
        if (hb + ob == 0.0) return 0u;
    }
    const double lb = p.levels[b];
    const double *krow = p.kmat != nullptr ? p.kmat + (size_t)b * p.L : nullptr;
    double si = 0.0, so = 0.0;
    constexpr int TB = 8;  // kernel-matrix loads in flight per lane
    for (int c0 = lane; c0 < p.L; c0 += 32 * TB) {
        double kv[TB];
#pragma unroll
        for (int k = 0; k < TB; ++k) {
            const int c = c0 + 32 * k;
            kv[k] = 0.0;
            if (c < p.L) {
                if (krow != nullptr) kv[k] = krow[c];  // same expression, evaluated once per level set
                else {
                    const double diff = p.levels[c] - lb;
                    kv[k] = 0.3989422804014327 * exp(p.mhH * (diff * diff));  // A * exp(-0.5*H*d^2), VRG:7,154
                }
            }
        }
#pragma unroll
        for (int k = 0; k < TB; ++k) {
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
    return pi >= po ? 1u : 0u;  // ties go inside, VRG:87
}
__device__ __forceinline__ uint32_t table_level(const Params &p, int b, int lane) {
    const long long *g = p.gstats;  // read through L2
    const double n_in = (double)__ldcg(g + 2 * p.L + ST_N_IN), n_out = (double)__ldcg(g + 2 * p.L + ST_N_OUT);
    return table_level_from(p, b, lane, n_in, n_out, [&](int c, double &hi, double &ho) {
        hi = (double)__ldcg(g + c);
        ho = (double)__ldcg(g + p.L + c);
    });
}

// final: the table of the state a finished run leaves behind (no bookkeeping, whatever the status) -- vrg_get_table then
// describes the final state on every path
__global__ void __launch_bounds__(TABLE_BLOCK) k_table(Params p, int final) {
    if (!final && p.ctrl[C_STATUS] != RUNNING) return;
    if (!final && blockIdx.x == 0 && threadIdx.x == 0) prepare_sweep(p);
    __shared__ uint32_t s_bits[32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 32 + warp;
    const uint32_t mybit = b < p.L ? table_level(p, b, lane) << warp : 0u;
    if (lane == 0) s_bits[warp] = mybit;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t w = 0;
        for (int i = 0; i < 32; ++i) w |= s_bits[i];
        uint32_t *bits = table_bits(p);
        if (bits[blockIdx.x] != w) p.ctrl[C_FULL_SWEEP] = p.ctrl[C_SWEEPS] + 1;  // the sweep behind this table looks at every band voxel
        bits[blockIdx.x] = w;
    }
}

// ---------------------------------------------------------------------------------------------
// The sweep's per-lane state: a sliding 3x3 (z,y) window over the segmented plane for one word column.
// For a row, o = OR of the three planes' words and a = AND (outside the volume: o = 0, a = ~0), so
//   dil26(S)            = x-dilate(o[y-1] | o[y] | o[y+1])
//   dil26(~S in volume) = x-dilate(~(a[y-1] & a[y] & a[y+1]) & valid)
// Rows are loaded two ahead of their use, so the L2 latency of the three 128-byte loads per row is hidden.
struct Strip {
    long long base;  // word index of this lane's column in plane zl, row 0
    uint32_t vm;
    int flags;       // bit 0: column inside the row, bit 1: plane zl-1 exists, bit 2: plane zl+1 exists, bit 3: active lane
    bool active;
    uint32_t op, ap, oc, ac, sc, on, an, sn, o2, a2, s2;  // rows y-1, y, y+1, y+2

    __device__ __forceinline__ void row(const Params &p, int yy, uint32_t &o, uint32_t &a, uint32_t &s) const {
        o = 0u; a = 0xFFFFFFFFu; s = 0u;
        if ((flags & 1) && yy >= 0 && yy < p.Y) {
            const uint32_t *q = p.S + base + (long long)yy * p.WP;
            s = q[0];
            const uint32_t w0 = (flags & 2) ? q[-p.plane_words] : 0u, w2 = (flags & 4) ? q[p.plane_words] : 0u;
            o = w0 | s | w2;
            a = ((flags & 2) ? w0 : 0xFFFFFFFFu) & s & ((flags & 4) ? w2 : 0xFFFFFFFFu);
        }
    }
    // WIDE: the warp's 32 lanes are the whole row (lane = word column, no halo lanes); dense sweep on rows of 31 / 32 words
    template <bool WIDE = false>
    __device__ __forceinline__ void begin(const Params &p, int zl, int y0, int c, int lane) {
        const bool inr = c >= 0 && c < p.XW;
        active = WIDE ? inr : (inr && lane >= 1 && lane <= p.segw);
        vm = inr ? valid_mask(p, c) : 0u;
        base = (long long)zl * p.plane_words + c;
        flags = (inr ? 1 : 0) | ((inr && zl - 1 >= p.valid_lo) ? 2 : 0) | ((inr && zl + 1 < p.valid_hi) ? 4 : 0);
        uint32_t sp;
        row(p, y0 - 1, op, ap, sp);
        row(p, y0, oc, ac, sc);
        row(p, y0 + 1, on, an, sn);
    }
    // bands of row y (s = segmented word, returns inner | outer-without-E); then slides one row down
    template <bool WIDE = false>
    __device__ __forceinline__ void step(const Params &p, int y, uint32_t &s, uint32_t &inner, uint32_t &outer, int lane = 0) {
        row(p, y + 2, o2, a2, s2);
        const uint32_t dil_s = WIDE ? dilate_x1_row(op | oc | on, lane) : dilate_x1(op | oc | on);
        const uint32_t dil_n = WIDE ? dilate_x1_row(~(ap & ac & an) & vm, lane) : dilate_x1(~(ap & ac & an) & vm);
        s = sc;
        inner = active ? (s & dil_n) : 0u;
        outer = active ? (~s & vm & dil_s) : 0u;
        op = oc; ap = ac;
        oc = on; ac = an; sc = sn;
        on = o2; an = a2; sn = s2;
    }
};

struct Unit { int zl, y0, y1, sg; };
__device__ __forceinline__ Unit decode_unit(const Params &p, long long u, int zlo, int nyb) {
    Unit r;
    r.sg = (int)(u % p.nseg);
    const long long t = u / p.nseg;
    r.y0 = (int)(t % nyb) * ROWS_PER_UNIT;
    r.zl = zlo + (int)(t / nyb);
    r.y1 = min(p.Y, r.y0 + ROWS_PER_UNIT);
    return r;
}

// writes the flip word of a row segment; rows away from the front cost no store (warp-uniform branch)
// and appends own-plane rows that flip to the front list, which k_cancel / k_flip consume one row per warp
// (rows at the front are spatially clustered; a list spreads them evenly over the machine).
// `was` = the row's flag, loaded by the caller early in the row so that its L2 latency hides behind the row's work.
__device__ __forceinline__ void store_flips(const Params &p, long long widx, long long ridx, uint8_t was, uint32_t f, bool active,
                                            bool own, int lane) {
    const bool any = __ballot_sync(FULL, f != 0u) != 0u;
    if (any || was) {
        if (active) {
            p.F[widx] = f;
            if (p.C != nullptr) p.C[widx] = 0u;  // k_cancel refills it for rows that still flip
        }
        if (lane == 0) {
            if (any != (was != 0)) p.rowflag[ridx] = any ? 1 : 0;
            if (any && own) {
                int *fl = front_list(p, (int)(p.ctrl[C_SWEEPS] & 1));
                fl[1 + atomicAdd(&fl[0], 1)] = (int)ridx;
            }
        }
    }
}

// the same for a warp that holds a whole row of two 16-word segments (lanes 0..15 and 16..31): flags, stores and front rows
// stay per segment, as every other kernel expects them; `was` = the flag of the lane's own segment
__device__ __forceinline__ void store_flips_wide(const Params &p, long long widx, long long ridx, uint8_t was, uint32_t f, bool active,
                                                 bool own, int lane) {
    const unsigned hit = __ballot_sync(FULL, f != 0u);
    const bool any = ((lane < 16 ? hit : hit >> 16) & 0xFFFFu) != 0u;
    if (any || was) {
        if (active) {
            p.F[widx] = f;
            if (p.C != nullptr) p.C[widx] = 0u;
        }
        if ((lane & 15) == 0) {
            if (any != (was != 0)) p.rowflag[ridx] = any ? 1 : 0;
            if (any && own) {
                int *fl = front_list(p, (int)(p.ctrl[C_SWEEPS] & 1));
                fl[1 + atomicAdd(&fl[0], 1)] = (int)ridx;
            }
        }
    }
}

// The two kinds of dense sweep.  A voxel's decision bit D = dbits[level(I)] depends on the iteration only through the table, and
// every change of the table stamps C_FULL_SWEEP, as do the start of a run and caller-chosen flips.  So a REFRESH sweep (the
// stamp names it) evaluates D from the fp64 intensities and keeps the words in the bit-plane Dc (layout of S); every other sweep
// of the run is k_sweep_band<MODE_F64_DENSE>: the band sweep with D read from Dc, and only for the words that hold a band voxel,
// instead of streaming 8 B per voxel.  Both kernels are enqueued for every sweep and one of them returns at once (the choice is
// on the device: the table is known only there, and the batches are replayed graphs).  Without Dc (VRG_NO_DCACHE) every sweep
// is a refresh.
__device__ __forceinline__ bool dense_refresh(const Params &p) {
    return p.Dc == nullptr || p.ctrl[C_FULL_SWEEP] == p.ctrl[C_SWEEPS] + 1;
}

// Decision + flip word of one row segment of the band sweep: the decision bit D is looked up only for the 32-voxel words
// that hold a band voxel -- BAND / INDEX: gathered through the level and the table (four gathers in flight); F64_DENSE: the
// word of Dc, one load per lane.  A band voxel flips iff D != S (VRG:87).
template <int MODE, bool LATTICE>
__device__ __forceinline__ int band_row(const Params &p, const uint32_t *s_dbits, int zl, int y, int sg, uint32_t s,
                                        uint32_t inner, uint32_t outer, bool active, bool own, int lane) {
    const int c0 = sg * p.segw - 1;
    const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c0 + lane;
    const long long ridx = ((long long)zl * p.Y + y) * p.nseg + sg;
    const uint8_t was = p.rowflag[ridx];
    if (p.E != nullptr && outer) outer &= ~p.E[widx];
    const uint32_t band = inner | outer;
    uint32_t D = 0;
    if constexpr (MODE == MODE_F64_DENSE) {
        if (band) D = p.Dc[widx];  // F = band & (D ^ s) ignores D elsewhere (band = 0 on inactive lanes)
    } else {
        unsigned m = __ballot_sync(FULL, band != 0u);
        const long long rowvox = (long long)zl * p.plane_vox + (long long)y * p.X + lane;
        while (m) {  // warp-uniform: only words that hold a band voxel, four at a time
            int js[4], lv[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                js[k] = -1; lv[k] = -1;
                if (m) {
                    js[k] = __ffs(m) - 1;
                    m &= m - 1;
                    const int x = (c0 + js[k]) * 32 + lane;
                    if (x < p.X) lv[k] = level_at<MODE, LATTICE>(p, rowvox + (long long)(c0 + js[k]) * 32);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (js[k] < 0) break;
                const int l = lv[k];
                const uint32_t bit = l >= 0 ? (s_dbits[l >> 5] >> (l & 31)) & 1u : 0u;
                const unsigned word = __ballot_sync(FULL, bit);
                if (lane == js[k]) D = word;
            }
        }
    }
    const uint32_t f = band & (D ^ s);  // inner band leaves iff in < out, outer band enters iff in >= out
    store_flips(p, widx, ridx, was, f, active, own, lane);
    return own ? __popc(f) : 0;
}

// k_sweep_band: the stencil sweep of the BAND / INDEX modes, and every sweep but the refreshes of the F64_DENSE mode.  Bands:
//   inner = S & dil26(~S in volume)      (segmented with an unsegmented in-bounds neighbour, VRG:139-142)
//   outer = ~S & ~E & dil26(S)           (unsegmented, not excluded, with a segmented neighbour, VRG:143-145)
// Full pass: a warp owns a strip of ROWS_PER_UNIT rows x 30 words of one plane and slides down it, over the units
// near a segmented voxel (unit occupancy map).
// Incremental pass (single slab, decision table unchanged since the last sweep): a voxel's flip flag can differ
// from last time only if a voxel of its 26-neighbourhood flipped, so only the rows within one row / plane /
// segment of last sweep's front rows are re-evaluated (each claimed once through `stamp`); every other row keeps
// its all-zero flip word.  The work is then proportional to the moving front, like the reference's narrow band.
// F64_DENSE: the sweep behind a refresh is incremental too, so the refresh kernels leave F, the row flags and the front
// list as the full pass would.  No shared memory: D comes from Dc, not from the table.
template <int MODE, bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_sweep_band(Params p) {
    if (p.ctrl[C_STATUS] != RUNNING) return;
    if (MODE == MODE_F64_DENSE && dense_refresh(p)) return;
    extern __shared__ uint32_t s_dbits[];
    if (MODE != MODE_F64_DENSE) {
        for (int i = threadIdx.x; i < p.LW; i += BLOCK) s_dbits[i] = table_bits(p)[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int zlo = max(p.valid_lo, p.own_lo - 1), zhi = min(p.valid_hi, p.own_hi + 1);
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nwarps = (long long)gridDim.x * WARPS;
    const long long warp0 = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5);
    long long flips = 0;
    Strip st;
    const bool single_slab = p.valid_lo == p.own_lo && p.valid_hi == p.own_hi;
    if (single_slab && p.ctrl[C_FULL_SWEEP] != p.ctrl[C_SWEEPS] + 1) {
        const int *dl = dirty_list(p, (int)(p.ctrl[C_SWEEPS] & 1));  // built by the previous iteration's k_flip
        const int n = dl[0];
        for (int i = (int)warp0; i < n; i += (int)nwarps) {
            const int r = dl[1 + i];
            const int sg = r % p.nseg, t = r / p.nseg, y = t % p.Y, zl = t / p.Y;
            st.begin(p, zl, y, sg * p.segw - 1 + lane, lane);
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            flips += band_row<MODE, LATTICE>(p, s_dbits, zl, y, sg, s, inner, outer, st.active, true, lane);
        }
    } else {
        const long long nunits = (long long)(zhi - zlo) * nyb * p.nseg;
        for (long long u = warp0; u < nunits; u += nwarps) {
            const Unit un = decode_unit(p, u, zlo, nyb);
            if (!unit_near_segmented(p, un.zl, un.y0, un.sg, lane)) continue;
            const bool own = un.zl >= p.own_lo && un.zl < p.own_hi;
            st.begin(p, un.zl, un.y0, un.sg * p.segw - 1 + lane, lane);
            for (int y = un.y0; y < un.y1; ++y) {
                uint32_t s, inner, outer;
                st.step(p, y, s, inner, outer);
                flips += band_row<MODE, LATTICE>(p, s_dbits, un.zl, y, un.sg, s, inner, outer, st.active, own, lane);
            }
        }
    }
    flips = warp_sum(flips);
    if (lane == 0 && flips) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_FLIPS], (unsigned long long)flips);
}

// ---------------------------------------------------------------------------------------------
// TMA helpers (1-D bulk copies, cp.async.bulk -> SASS UBLKCP) and mbarriers
__device__ __forceinline__ uint32_t smem_u32(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, 0x989680;\n\t"
        "@P1 bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// the refresh sweep's counter (vrg_result.dense_refresh_sweeps); nothing else touches the word while a sweep runs
__device__ __forceinline__ void count_refresh(const Params &p) {
    if (blockIdx.x == 0 && threadIdx.x == 0) p.ctrl[C_REFRESHES] += 1;
}

// Work distribution of the dense sweep.  A work unit = `dense_rows` consecutive rows of one (plane, segment) column; units are
// numbered so that consecutive units are consecutive in memory.  Every warp starts with two statically assigned units
// (w, w + nwarps) and then draws further units from a device-wide counter: at any moment the whole machine streams one
// compact window of the volume (kind to the TLB and the DRAM pages), and a warp on a slow SM simply takes fewer units, so
// the kernel has no tail (on an 82-plane slab the static split left the average SM idle for 12 % of the kernel).
// Lane 0 walks the unit sequence first, as the TMA prefetcher, and hands the unit numbers to the consuming warp through a
// small ring in shared memory; the counter's latency hides behind a whole unit of work.
constexpr int UNIT_RING = 8;  // the prefetcher is at most DENSE_STAGES + 1 rows, hence (one-row units) 3 units ahead

// k_sweep_dense: the stencil sweep of the F64_DENSE mode.  Every voxel's decision is evaluated from its fp64 intensity
// every iteration: the volume is streamed at 8 B/voxel by 1-D TMA bulk copies, one row segment (<= 7680 B) per stage,
// into a per-warp ring in shared memory; the warp that consumed a stage re-arms it, so no cross-warp sync exists.
// Needs X even (16-byte alignment of every row segment); otherwise the host launches k_sweep_dense_ldg.
// WIDE (rows of 31 or 32 words, e.g. X = 1024): such a row is two 16-word segments for every other kernel, which left half
// of this kernel's lanes idle; here one warp takes the whole row -- lane = word column, no halo lanes (nothing lies beyond
// the row ends), one 8 KB stage per row, flags and front rows still per segment.
constexpr int WIDE_STAGE_BYTES = 32 * 32 * 8;
template <bool LATTICE, bool WIDE>
__device__ __forceinline__ void sweep_dense_body(const Params &p) {
    constexpr int SB = WIDE ? WIDE_STAGE_BYTES : STAGE_BYTES;
    if (p.ctrl[C_STATUS] != RUNNING || !dense_refresh(p)) return;
    count_refresh(p);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t *s_dbits = (uint32_t *)smem_raw;
    const int dbits_bytes = (p.LW * 4 + 127) & ~127;
    uint64_t *bars = (uint64_t *)(smem_raw + dbits_bytes);                                     // [DENSE_WARPS][DENSE_STAGES]
    int *rings = (int *)(bars + DENSE_WARPS * DENSE_STAGES);                                   // [DENSE_WARPS][UNIT_RING]
    double *stages = (double *)(smem_raw + dbits_bytes + ((DENSE_WARPS * (DENSE_STAGES * 8 + UNIT_RING * 4) + 127) & ~127));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < p.LW; i += DENSE_WARPS * 32) s_dbits[i] = table_bits(p)[i];
    uint64_t *mybar = bars + warp * DENSE_STAGES;
    int *myring = rings + warp * UNIT_RING;
    double *mystage = stages + (size_t)warp * DENSE_STAGES * (SB / 8);
    // the part of a stage that no row segment ever overwrites (beyond the shortest segment: the row's tail, and the
    // words up to the batch width) must hold a valid intensity, since the evaluation below is branch-free
    {
        const int shortest = WIDE ? p.X : min(p.segw * 32, p.X - (p.nseg - 1) * p.segw * 32);
#pragma unroll
        for (int s = 0; s < DENSE_STAGES; ++s)
            for (int i = shortest + lane; i < SB / 8; i += 32) mystage[s * (SB / 8) + i] = p.lev0;
    }
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < DENSE_STAGES; ++s) mbar_init(mybar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy fill before the async-proxy copies
    __syncthreads();
    const int zlo = max(p.valid_lo, p.own_lo - 1), zhi = min(p.valid_hi, p.own_hi + 1);
    const int R = p.dense_rows;
    const int nyb = (p.Y + R - 1) / R;
    const int nwarps = gridDim.x * DENSE_WARPS;
    const int w = blockIdx.x * DENSE_WARPS + warp;
    const int nunits = (zhi - zlo) * nyb * (WIDE ? 1 : p.nseg);
    unsigned long long *next_unit = (unsigned long long *)&p.ctrl[C_NEXT_UNIT];
    auto decode = [&](int u, int &zl, int &sg, int &y, int &y1) {
        sg = WIDE ? 0 : u % p.nseg;
        const int t = WIDE ? u : u / p.nseg;
        y = (t % nyb) * R;
        zl = zlo + t / nyb;
        y1 = min(p.Y, y + R);
    };
    // ---- lane 0: the prefetcher's walk ----
    int pu = w, pu_next = w + nwarps, pzl = 0, psg = 0, py = 0, py1 = 0, phead = 0;
    auto pre_enter = [&]() {  // announce the unit to the consumer; ids >= nunits end its walk
        myring[phead++ & (UNIT_RING - 1)] = pu;
        if (pu < nunits) decode(pu, pzl, psg, py, py1);
    };
    auto pre_issue = [&](int s) {  // one row segment into stage s, then step to the next row
        const int x0 = WIDE ? 0 : psg * p.segw * 32;
        const uint32_t bytes = (uint32_t)(WIDE ? p.X : min(p.segw * 32, p.X - x0)) * 8u;
        const double *src = p.data + (long long)pzl * p.plane_vox + (long long)py * p.X + x0;
        mbar_expect_tx(mybar + s, bytes);
        tma_bulk_load(mystage + (size_t)s * (SB / 8), src, bytes, mybar + s);
        if (++py >= py1) {
            pu = pu_next;
            pu_next = pu_next < nunits ? 2 * nwarps + (int)atomicAdd(next_unit, 1ull) : pu_next;  // used a whole unit later
            pre_enter();
        }
    };
    if (lane == 0) {
        pre_enter();
#pragma unroll
        for (int s = 0; s < DENSE_STAGES; ++s)
            if (pu < nunits) pre_issue(s);
    }
    __syncwarp();
    // ---- the consuming warp ----
    int ctail = 0, cu = myring[ctail++ & (UNIT_RING - 1)], czl = 0, csg = 0, cy = 0, cy1 = 0;
    bool fresh = true;
    if (cu < nunits) decode(cu, czl, csg, cy, cy1);
    int stage = 0;
    uint32_t parity = 0;
    long long flips = 0;
    Strip st, nx;  // nx: the window of this warp's NEXT unit, requested while the last row of the current one is evaluated (a
                   // window restart is nine loads, one L2 round trip; behind a unit of 4 rows that was 5 % of a thin slab's sweep)
    int c0 = 0, nu = nunits, nzl = 0, nsg = 0, ny = 0, ny1 = 0;
    bool own = false;
    while (cu < nunits) {
        const int y = cy;
        if (fresh) {  // first unit: start the window
            c0 = WIDE ? 0 : csg * p.segw - 1;
            own = czl >= p.own_lo && czl < p.own_hi;
            st.template begin<WIDE>(p, czl, y, c0 + lane, lane);
            fresh = false;
        }
        if (y + 1 >= cy1) {  // last row of the unit: lane 0 announced the next one when it issued this row
            nu = myring[ctail & (UNIT_RING - 1)];
            if (nu < nunits) {
                decode(nu, nzl, nsg, ny, ny1);
                nx.template begin<WIDE>(p, nzl, ny, (WIDE ? 0 : nsg * p.segw - 1) + lane, lane);
            }
        }
        uint32_t s, inner, outer;
        st.template step<WIDE>(p, y, s, inner, outer, lane);
        const long long widx = (long long)czl * p.plane_words + (long long)y * p.WP + c0 + lane;
        const long long ridx = ((long long)czl * p.Y + y) * p.nseg + (WIDE ? (lane >> 4) : csg);
        const uint8_t was = p.rowflag[ridx];
        if (p.E != nullptr && outer) outer &= ~p.E[widx];
        const uint32_t band = inner | outer;
        // decision bit of every voxel of the row segment: word j of the segment ends up in lane j + 1.
        // Branch-free over all 30 words (the stage beyond the row end holds valid intensities, see the fill above;
        // their bits are masked by the band), so the compiler interleaves the words' dependency chains.
        const double *sv = mystage + (size_t)stage * (SB / 8) + lane;
        mbar_wait(mybar + stage, parity);
        // phase 1 (no convergence points, so the 30 dependency chains overlap): bit j+1 of `mine` = decision of this
        // lane's voxel in word j;  phase 2: 32x32 bit transpose across the warp, lane j+1 ends up with word j.
        uint32_t mine = 0;
        // batches of 10 words: loads first, then the level arithmetic, then the table look-ups, so that ten
        // dependency chains are in flight at once whatever the register allocator would prefer.  (Narrower batches
        // that overshoot segw less -- 4 x 7 for 28 words, 3 x 8 for 22 -- measured the same or slower: profiles/README.md.)
        constexpr int BW = WIDE ? 8 : 10;
        const int nbatch = ((WIDE ? p.XW : p.segw) + BW - 1) / BW;
#pragma unroll
        for (int jb = 0; jb < (WIDE ? 32 : WORDS_PER_WARP); jb += BW) {
            if (jb / BW >= nbatch) break;  // warp-uniform (words past segw hold valid stale data, masked by the band)
            double v[BW];
            int l[BW];
            uint32_t wd[BW];
#pragma unroll
            for (int k = 0; k < BW; ++k) v[k] = sv[(jb + k) * 32];
#pragma unroll
            for (int k = 0; k < BW; ++k) l[k] = level_of<LATTICE>(p, v[k]);
#pragma unroll
            for (int k = 0; k < BW; ++k) wd[k] = s_dbits[l[k] >> 5];
#pragma unroll
            for (int k = 0; k < BW; ++k) mine |= ((wd[k] >> (l[k] & 31)) & 1u) << (jb + k + (WIDE ? 0 : 1));
        }
        const uint32_t D = transpose32(mine, lane);
        if (p.Dc != nullptr && st.active) p.Dc[widx] = D;
        __syncwarp();
        if (lane == 0 && pu < nunits) pre_issue(stage);  // the stage is drained (values are in registers): re-arm it for a later row
        if (++stage == DENSE_STAGES) { stage = 0; parity ^= 1u; }
        const uint32_t f = band & (D ^ s);
        if (WIDE) store_flips_wide(p, widx, ridx, was, f, st.active, own, lane);
        else store_flips(p, widx, ridx, was, f, st.active, own, lane);
        if (own) flips += __popc(f);
        if (++cy >= cy1) {  // on to the next unit of this warp's sequence: its window is under way
            ++ctail;
            cu = nu; czl = nzl; csg = nsg; cy = ny; cy1 = ny1;
            st = nx;
            c0 = WIDE ? 0 : csg * p.segw - 1;
            own = czl >= p.own_lo && czl < p.own_hi;
        }
    }
    flips = warp_sum(flips);
    if (lane == 0 && flips) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_FLIPS], (unsigned long long)flips);
}

template <bool LATTICE, bool WIDE = false>
__global__ void __launch_bounds__(DENSE_WARPS * 32) k_sweep_dense(Params p) { sweep_dense_body<LATTICE, WIDE>(p); }
// The same sweep held to 96 registers per thread, for the pipelined run (vrg_tail.cuh): its statistics and table kernels have
// to find room on the SMs this kernel's blocks occupy.  Registers are handed out 512 per warp, so 100..112 per thread all cost
// 14 warps x 3584 = 50176 of the 65536 and leave 15360: not enough for a 256-thread block of k_async_table (63 -> 64
// registers, 16384), which then runs BEHIND the sweep instead of beside it.  8 GPUs, C3, per run: 19.7 ms with 112 registers
// and 128-thread side kernels (they fit, but take twice as long and the sweep's blocks still crowd them), 17.5 ms with 112 /
// 256 (a cap of 104 allocates the same 112: 17.6 ms), 15.8 ms with 96 / 256 although the sweep itself is 5 % slower
// (profiles/r2ak_*, r2z_scale_8.json).
template <bool LATTICE, bool WIDE = false>
__global__ void __maxnreg__(96) k_sweep_dense_slim(Params p) { sweep_dense_body<LATTICE, WIDE>(p); }

// Fallback of the dense sweep for odd X (row segments not 16-byte aligned): plain coalesced 8-byte loads.
template <bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_sweep_dense_ldg(Params p) {
    if (p.ctrl[C_STATUS] != RUNNING || !dense_refresh(p)) return;
    count_refresh(p);
    extern __shared__ uint32_t s_dbits[];
    for (int i = threadIdx.x; i < p.LW; i += BLOCK) s_dbits[i] = table_bits(p)[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int zlo = max(p.valid_lo, p.own_lo - 1), zhi = min(p.valid_hi, p.own_hi + 1);
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(zhi - zlo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    long long flips = 0;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, zlo, nyb);
        const int c0 = un.sg * p.segw - 1, c = c0 + lane;
        const bool own = un.zl >= p.own_lo && un.zl < p.own_hi;
        st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            const long long widx = (long long)un.zl * p.plane_words + (long long)y * p.WP + c;
            const long long ridx = ((long long)un.zl * p.Y + y) * p.nseg + un.sg;
            const uint8_t was = p.rowflag[ridx];
            if (p.E != nullptr && outer) outer &= ~p.E[widx];
            const uint32_t band = inner | outer;
            uint32_t D = 0;
            const int xlane = (c0 + 1) * 32 + lane;
            const double *drow = p.data + (long long)un.zl * p.plane_vox + (long long)y * p.X + xlane;
            constexpr int U = 10;
#pragma unroll
            for (int jb = 0; jb < WORDS_PER_WARP; jb += U) {
                if (jb >= p.segw || c0 + 1 + jb >= p.XW) break;  // warp-uniform
                double v[U];
#pragma unroll
                for (int k = 0; k < U; ++k) v[k] = (xlane + (jb + k) * 32 < p.X) ? drow[(jb + k) * 32] : p.lev0;
#pragma unroll
                for (int k = 0; k < U; ++k) {
                    const int l = level_of<LATTICE>(p, v[k]);
                    const unsigned word = __ballot_sync(FULL, (s_dbits[l >> 5] >> (l & 31)) & 1u);
                    if (lane == jb + k + 1) D = word;
                }
            }
            if (p.Dc != nullptr && st.active) p.Dc[widx] = D;
            const uint32_t f = band & (D ^ s);
            store_flips(p, widx, ridx, was, f, st.active, own, lane);
            if (own) flips += __popc(f);
        }
    }
    flips = warp_sum(flips);
    if (lane == 0 && flips) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_FLIPS], (unsigned long long)flips);
}

// ---------------------------------------------------------------------------------------------
// The front list: own-plane row segments whose flip word is non-zero; calls fn(zl, y, sg) warp-uniformly, one row per warp.
template <typename Fn>
__device__ __forceinline__ void for_front_rows(const Params &p, Fn fn) {
    const int *fl = front_list(p, (int)(p.ctrl[C_SWEEPS] & 1));
    const int n = fl[0];
    const int nwarps = gridDim.x * WARPS;
    for (int k = blockIdx.x * WARPS + (threadIdx.x >> 5); k < n; k += nwarps) {
        const int rr = fl[1 + k];
        const int sg = rr % p.nseg, t = rr / p.nseg;
        fn(t / p.Y, t % p.Y, sg);
    }
}

// A row that flips, and its (z, y, segment) neighbours, may change band status: each is claimed once (stamp) and
// appended to the list the next incremental sweep walks.
__device__ __forceinline__ void claim_dirty_rows(const Params &p, int zl, int y, int sg, int lane) {
    const int next = (int)p.ctrl[C_SWEEPS] + 1;  // the sweep that will read the list
    int *dl = dirty_list(p, next & 1);
    const int nds = p.nseg > 1 ? 3 : 1;
    int ridx = -1;
    if (lane < 9 * nds) {
        const int ss = sg + (nds == 3 ? lane % 3 - 1 : 0), yy = y + (lane / nds) % 3 - 1, zz = zl + lane / (3 * nds) - 1;
        if (zz >= p.own_lo && zz < p.own_hi && yy >= 0 && yy < p.Y && ss >= 0 && ss < p.nseg) {
            ridx = (zz * p.Y + yy) * p.nseg + ss;
            if (atomicExch(&p.stamp[ridx], next) == next) ridx = -1;
        }
    }
    const unsigned won = __ballot_sync(FULL, ridx >= 0);
    if (won) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&dl[0], __popc(won));
        base = __shfl_sync(FULL, base, 0);
        if (ridx >= 0) dl[1 + base + __popc(won & ((1u << lane) - 1u))] = ridx;
    }
}

// k_cancel: an outer-band voxel marked to enter is dropped when every segmented neighbour leaves in the same
// iteration (VRG:183-190 then VRG:198).  Rewrites F to the executed flips (race-free: only non-segmented bits are
// cleared, neighbours read F & S), keeps the cancelled ones in C for the absorb rule, and applies the integer
// histogram deltas that replace the reference's incremental float sums (VRG:232-247).
// cancel_row: one front row, one warp.  d_in accumulates this lane's change of the inside region's size.
// s, f: this lane's words of the segmented and flip planes (0 outside the row), loaded by the caller -- k_tail fetches them for
// a warp's next row while it works on the current one
template <int MODE, bool LATTICE>
__device__ __forceinline__ void cancel_row_loaded(const Params &p, int zl, int y, int sg, int lane, bool dirty, long long &d_in,
                                                  uint32_t s, uint32_t f) {
    unsigned long long *hin = (unsigned long long *)p.lstats, *hout = hin + p.L;
    const int c0 = sg * p.segw - 1, c = c0 + lane;
    const bool inr = c >= 0 && c < p.XW;
    const bool active = inr && lane >= 1 && lane <= p.segw;
    const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
    const uint32_t a0 = active ? (f & ~s) : 0u, r = active ? (f & s) : 0u;
    // The levels of the flipped voxels feed the histogram deltas below (the continuous mode has none: see k_cont_incr).
    // Word-cooperative: for every 32-voxel word that holds a candidate (removals + additions before the cancel rule) the
    // whole warp fetches the word's 32 levels in one coalesced load -- a thick vessel's front puts 10-16 flips into one word,
    // which one lane gathering its own word's voxels paid for with four dependent DRAM round trips.  Four words are in flight
    // at once, and they start here, beside the neighbour loads of the cancel rule instead of behind them.
    const long long rowvox0 = (long long)zl * p.plane_vox + (long long)y * p.X + (long long)c0 * 32 + lane;
    unsigned wm = MODE == MODE_CONT ? 0u : __ballot_sync(FULL, (r | a0) != 0u);
    int wj[4], wl[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        wj[k] = wm ? __ffs(wm) - 1 : -1;
        wm &= wm - 1;  // 0 stays 0
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        wl[k] = (wj[k] >= 0 && (c0 + wj[k]) * 32 + lane < p.X) ? level_at<MODE, LATTICE>(p, rowvox0 + (long long)wj[k] * 32) : 0;
    uint32_t a = 0;
    if (__ballot_sync(FULL, a0 != 0u)) {
        uint32_t keepv = s & ~f;
        if (inr) {
#pragma unroll
            for (int dz = -1; dz <= 1; ++dz) {
                const int zz = zl + dz;
                if (zz < p.valid_lo || zz >= p.valid_hi) continue;
#pragma unroll
                for (int dy = -1; dy <= 1; ++dy) {
                    const int yy = y + dy;
                    if ((dz == 0 && dy == 0) || yy < 0 || yy >= p.Y) continue;
                    const long long i = (long long)zz * p.plane_words + (long long)yy * p.WP + c;
                    keepv |= p.S[i] & ~p.F[i];
                }
            }
        }
        a = a0 & dilate_x1(keepv);
        if (active && a != a0) p.F[widx] = r | a;
    }
    if (active) p.Cq[widx] = a0 & ~a;  // == p.C with label 4 (k_absorb reads it); the quirk counters read the front rows' words
    // Flip in place right here.  Safe against the warps that are reading this row as a neighbour: they use
    // S & ~F, and that value is the same before, between and after the two stores (executed flip: F = 1 both
    // times -> 0; cancelled addition: S = 0 both times -> 0; everything else is untouched).
    const uint32_t done = r | a;  // executed flips
    if (active && done) {
        p.S[widx] = s ^ done;
        p.unitmap[unit_index(p, zl, y, c)] = 1;
    }
    if (dirty) claim_dirty_rows(p, zl, y, sg, lane);
    d_in += __popc(a) - __popc(r);
    // histogram deltas: lane b of the warp owns voxel b of each fetched word
    auto deltas = [&](int j, int level) {
        const uint32_t md = __shfl_sync(FULL, done, j), ma = __shfl_sync(FULL, a, j);
        if ((md >> lane) & 1u) {
            const unsigned long long d = (ma >> lane) & 1u ? 1ull : ~0ull;  // entered: +1 inside, -1 outside; left: the reverse
            atomicAdd(&hin[level], d);
            atomicAdd(&hout[level], 0ull - d);
        }
    };
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (wj[k] >= 0) deltas(wj[k], wl[k]);  // warp-uniform
    while (wm) {  // more than four words with flips in one row segment
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            wj[k] = wm ? __ffs(wm) - 1 : -1;
            wm &= wm - 1;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            wl[k] = (wj[k] >= 0 && (c0 + wj[k]) * 32 + lane < p.X) ? level_at<MODE, LATTICE>(p, rowvox0 + (long long)wj[k] * 32) : 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (wj[k] >= 0) deltas(wj[k], wl[k]);
    }
}
template <int MODE, bool LATTICE>
__device__ __forceinline__ void cancel_row(const Params &p, int zl, int y, int sg, int lane, bool dirty, long long &d_in) {
    const int c = sg * p.segw - 1 + lane;
    const bool inr = c >= 0 && c < p.XW;
    const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
    cancel_row_loaded<MODE, LATTICE>(p, zl, y, sg, lane, dirty, d_in, inr ? p.S[widx] : 0u, inr ? p.F[widx] : 0u);
}
__device__ __forceinline__ void cancel_finish(const Params &p, long long d_in, int lane) {
    d_in = warp_sum(d_in);
    if (lane == 0 && d_in) {
        atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_IN], (unsigned long long)d_in);
        atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_OUT], (unsigned long long)(-d_in));
    }
}

template <int MODE, bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_cancel(Params p) {
    const bool go = p.ctrl[C_STATUS] == RUNNING && p.ctrl[C_APPLY];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        // snapshot for the slab halo exchange and k_quirks that follow (vrg_p2p.cuh): they read this iteration from it, not
        // from C_SWEEPS / C_STATUS, which the statistics exchange advances.  Sequence number = (run epoch << 32) | (sweep + 1).
        p.ctrl[C_HALO_GO] = go;
        p.ctrl[C_HALO_SEQ] = (long long)(((unsigned long long)p.ctrl[C_EPOCH] << 32) | (unsigned long long)(p.ctrl[C_SWEEPS] + 1));
    }
    if (!go) return;
    const int lane = threadIdx.x & 31;
    long long d_in = 0;
    const bool dirty = p.dirty_lists && p.valid_lo == p.own_lo && p.valid_hi == p.own_hi;
    for_front_rows(p, [&](int zl, int y, int sg) { cancel_row<MODE, LATTICE>(p, zl, y, sg, lane, dirty, d_in); });
    cancel_finish(p, d_in, lane);
}

// k_quirks: counts, over the front rows of the iteration k_cancel just applied, the flip patterns on which the
// reference's sequential list processing is order-dependent (SURVEY.md section 8(a); oracle/vrg_oracle.py counts the same
// sets as `quirk_potential`).  With S' the segmented plane after the flips, Aex / R the executed additions / removals and
// Cn the cancelled additions:
//   cancelled         |Cn|                          Q1, VRG:183-190 then :198 (order-free; part of the semantics)
//   add_to_inside     |Aex & ~dil26(~S' in volume)| an added voxel with no unsegmented neighbour left: the reference labels
//                                                   it 1 unconditionally (VRG:202) and corrects it only if a later flip looks (Q2)
//   remove_to_outside |R & ~dil26(S')|              a removed voxel with no segmented neighbour left: labelled 2 (VRG:174), same (Q2);
//                                                   both kinds drop out of the reference's delta sums (VRG:232-233, Q3)
//   cancel_repromoted |Cn & dil26(Aex)|             a cancelled addition next to an executed one: the reference adds it after all
//                                                   if that neighbour precedes it in the band list ("Q4")
// A run whose last three counters are zero lies inside the domain where the reference's result is order-free, i.e. where
// bit-identity with it is defined.  Runs after k_cancel and, on slabs, after the halo planes received the neighbours' flips.
struct QuirkCounts { int c = 0, a = 0, r = 0, p = 0; };  // per warp and launch: far below 2^31
__device__ __forceinline__ void quirks_row(const Params &p, int zl, int y, int sg, int lane, QuirkCounts &q) {
    const int c = sg * p.segw - 1 + lane;
    const bool inr = c >= 0 && c < p.XW;
    const bool active = inr && lane >= 1 && lane <= p.segw;
    const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
    // read through L2: inside k_tail other blocks wrote these words earlier in the same launch
    const uint32_t s1 = inr ? __ldcg(p.S + widx) : 0u, f = inr ? __ldcg(p.F + widx) : 0u;
    const uint32_t cn = active ? __ldcg(p.Cq + widx) : 0u;
    const uint32_t aex = active ? (f & s1) : 0u, r = active ? (f & ~s1) : 0u;
    const bool need_f = __ballot_sync(FULL, cn != 0u) != 0u;
    uint32_t o = s1, a = inr ? s1 : 0xFFFFFFFFu, ax = f & s1;
    if (inr) {
#pragma unroll
        for (int dz = -1; dz <= 1; ++dz) {
            const int zz = zl + dz;
            if (zz < p.valid_lo || zz >= p.valid_hi) continue;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy) {
                const int yy = y + dy;
                if ((dz == 0 && dy == 0) || yy < 0 || yy >= p.Y) continue;
                const long long i = (long long)zz * p.plane_words + (long long)yy * p.WP + c;
                const uint32_t sn = __ldcg(p.S + i);
                o |= sn; a &= sn;
                if (need_f) ax |= __ldcg(p.F + i) & sn;
            }
        }
    }
    const uint32_t vm = inr ? valid_mask(p, c) : 0u;
    const uint32_t dil_s = dilate_x1(o), dil_n = dilate_x1(~a & vm);
    const uint32_t dil_a = need_f ? dilate_x1(ax) : 0u;
    q.c += __popc(cn);
    q.a += __popc(aex & ~dil_n);
    q.r += __popc(r & ~dil_s);
    q.p += __popc(cn & dil_a);
}
__device__ __forceinline__ void quirks_finish(const Params &p, QuirkCounts q, int lane) {
    const int qc = __reduce_add_sync(FULL, q.c), qa = __reduce_add_sync(FULL, q.a), qr = __reduce_add_sync(FULL, q.r), qp = __reduce_add_sync(FULL, q.p);
    if (lane == 0) {
        unsigned long long *ex = (unsigned long long *)p.lstats + 2 * p.L;
        if (qc) atomicAdd(&ex[ST_Q_CANCELLED], (unsigned long long)qc);
        if (qa) atomicAdd(&ex[ST_Q_ADD_INSIDE], (unsigned long long)qa);
        if (qr) atomicAdd(&ex[ST_Q_REM_OUTSIDE], (unsigned long long)qr);
        if (qp) atomicAdd(&ex[ST_Q_REPROMOTED], (unsigned long long)qp);
    }
}
__global__ void __launch_bounds__(BLOCK) k_quirks(Params p) {
    if (!p.ctrl[C_HALO_GO]) return;  // snapshot of "this iteration applied its flips", left by k_cancel
    const int sweep = (int)((unsigned long long)p.ctrl[C_HALO_SEQ] & 0xFFFFFFFFull) - 1;
    const int *fl = front_list(p, sweep & 1);
    const int n = fl[0];
    const int lane = threadIdx.x & 31, nwarps = gridDim.x * WARPS;
    QuirkCounts q;
    for (int k = blockIdx.x * WARPS + (threadIdx.x >> 5); k < n; k += nwarps) {
        const int rr = fl[1 + k];
        const int sg = rr % p.nseg, t = rr / p.nseg;
        quirks_row(p, t / p.Y, t % p.Y, sg, lane, q);
    }
    quirks_finish(p, q, lane);
}

// k_flip_halo (slab runs only, after the F exchange): S ^= F on the halo planes, so the halo copy of the segmented
// plane follows the neighbour slab without ever being exchanged itself.  Own planes are flipped inside k_cancel.
__global__ void __launch_bounds__(BLOCK) k_flip_halo(Params p) {
    if (p.ctrl[C_STATUS] != RUNNING || !p.ctrl[C_APPLY]) return;
    const long long tid = (long long)blockIdx.x * BLOCK + threadIdx.x, nth = (long long)gridDim.x * BLOCK;
    for (int side = 0; side < 2; ++side) {
        const int zlo = side ? p.own_hi : max(p.valid_lo, p.own_lo - HALO);
        const int zhi = side ? min(p.valid_hi, p.own_hi + HALO) : p.own_lo;
        if (zhi <= zlo) continue;
        const long long b = (long long)zlo * p.plane_words, n = (long long)(zhi - zlo) * p.plane_words;
        for (long long i = tid; i < n; i += nth) {
            const uint32_t f = p.F[b + i];
            if (f) {
                p.S[b + i] ^= f;
                const long long w = b + i;
                const int zl = (int)(w / p.plane_words), y = (int)((w % p.plane_words) / p.WP), c = (int)(w % p.WP);
                p.unitmap[unit_index(p, zl, y, c)] = 1;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// k_absorb: excluded voxels within 1 of any listed flip (executed or cancelled), or within 2 of an executed flip,
// become outside (VRG:167-168, 177-179, 207-208).  Runs after k_cancel (and the F/C halo exchange).
// ab_out (continuous mode only, else nullptr): bit-plane that receives the absorbed voxels of this iteration -- that mode
// has no histograms, its band voxels get the absorbed voxels' kernel terms one by one (VRG:235,247, k_cont_incr).
template <int MODE, bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_absorb(Params p, uint32_t *ab_out) {
    if (p.ctrl[C_STATUS] != RUNNING || !p.ctrl[C_APPLY]) return;
    const int lane = threadIdx.x & 31;
    const long long nrows = (long long)(p.own_hi - p.own_lo) * p.Y * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    long long n_abs = 0;
    unsigned long long *hout = (unsigned long long *)p.lstats + p.L;
    for (long long rr = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); rr < nrows; rr += nwarps) {
        const int sg = (int)(rr % p.nseg);
        const long long t = rr / p.nseg;
        const int y = (int)(t % p.Y), zl = p.own_lo + (int)(t / p.Y);
        // any flagged row within +-2 rows/planes (and the neighbouring segments)?  75 candidates, 3 per lane
        bool near = false;
        for (int q = lane; q < 75; q += 32) {
            const int dz = q / 15 - 2, dy = (q / 3) % 5 - 2, ds = q % 3 - 1;
            const int zz = zl + dz, yy = y + dy, ss = sg + ds;
            if (zz >= p.valid_lo && zz < p.valid_hi && yy >= 0 && yy < p.Y && ss >= 0 && ss < p.nseg)
                near |= p.rowflag[((long long)zz * p.Y + yy) * p.nseg + ss] != 0;
        }
        // halo planes beyond +-1 carry no row flags of their own (their F comes from the neighbour slab)
        const bool halo_near = (zl - 2 < p.own_lo - 1 && zl - 2 >= p.valid_lo) || (zl + 2 > p.own_hi && zl + 2 < p.valid_hi);
        if (!__ballot_sync(FULL, near) && !halo_near) continue;
        const int c = sg * p.segw - 1 + lane;
        const bool inr = c >= 0 && c < p.XW;
        const bool active = inr && lane >= 1 && lane <= p.segw;
        const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
        const uint32_t e = active ? p.E[widx] : 0u;
        if (!__ballot_sync(FULL, e != 0u)) continue;
        uint32_t ve = 0, vc = 0;
        if (inr) {
            for (int dz = -2; dz <= 2; ++dz) {
                const int zz = zl + dz;
                if (zz < p.valid_lo || zz >= p.valid_hi) continue;
                for (int dy = -2; dy <= 2; ++dy) {
                    const int yy = y + dy;
                    if (yy < 0 || yy >= p.Y) continue;
                    const long long i = (long long)zz * p.plane_words + (long long)yy * p.WP + c;
                    ve |= p.F[i];
                    if (dz >= -1 && dz <= 1 && dy >= -1 && dy <= 1) vc |= p.C[i];
                }
            }
        }
        const uint32_t hit = dilate_x2(ve) | dilate_x1(vc);
        uint32_t ab = e & hit;
        if (!active || ab == 0u) continue;
        p.E[widx] = e & ~ab;
        n_abs += __popc(ab);
        if (ab_out != nullptr) ab_out[widx] = ab;
        if (MODE != MODE_CONT) {
            const long long rowvox = (long long)zl * p.plane_vox + (long long)y * p.X + (long long)c * 32;
            while (ab) {
                const int b = __ffs(ab) - 1; ab &= ab - 1;
                atomicAdd(&hout[level_at<MODE, LATTICE>(p, rowvox + b)], 1ull);  // addedPoints, VRG:235,247
            }
        }
    }
    n_abs = warp_sum(n_abs);
    if (lane == 0 && n_abs) {
        atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_OUT], (unsigned long long)n_abs);
        atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_EXCL], (unsigned long long)(-n_abs));
    }
}

// ---------------------------------------------------------------------------------------------
// k_advance: the exit tests of VRG:91-104 and the loop bookkeeping of VRG:113-117.
__device__ __forceinline__ void advance_state(const Params &p) {
    long long *c = p.ctrl;
    if (c[C_STATUS] != RUNNING) return;
    const long long *g = p.gstats + 2 * p.L;
    c[C_SWEEPS] += 1;
    if (g[ST_N_FLIPS] == 0) { c[C_STATUS] = 0; return; }   // converged, VRG:91
    if (!c[C_APPLY]) { c[C_STATUS] = 2; return; }          // max segment size, VRG:101
    const long long t = c[C_TRACE_N];
    p.trace[3 * t] = g[ST_N_FLIPS];
    p.trace[3 * t + 1] = g[ST_N_IN];
    p.trace[3 * t + 2] = g[ST_N_OUT];
    c[C_TRACE_N] = t + 1;
    c[C_APPLIED] += 1;
    c[C_ITER] += 1;
    if (c[C_ITER] > c[C_ITER_MAX]) c[C_STATUS] = 3;        // VRG:58,118
    else if (g[ST_TIME_UP] != 0) c[C_STATUS] = 1;          // VRG:97 on slabs: some rank's host saw the time budget run out and
                                                           // raised the flag in its statistics; every rank reads the same sum
}
__global__ void k_advance(Params p) {
    if (threadIdx.x == 0 && blockIdx.x == 0) advance_state(p);
}

// ---------------------------------------------------------------------------------------------
// init branch of update(), VRG:129-145: bit-planes from the valueMap, read in the caller's dtype.
// Seeds are label 0 (VRG:44); a map that already holds band labels (1 inner, 2 outer: the output of an earlier run) is
// read as the state those labels describe -- segmented = {0, 1}.  (The reference re-seeds such a map from label 0 alone
// and then dies at VRG:111 once its outer band list runs empty: tests/test_oracle_golden.py keeps that probe.)
// Anything that is not an integral value in 0..4 (negative, fractional, NaN, above 4) raises ST_BAD_LABEL.
template <typename T>
__device__ __forceinline__ bool label_value(T v, int &lab) {
    if constexpr (std::is_floating_point<T>::value) {
        const bool ok = v >= T(0) && v <= T(4) && v == floor(v);  // NaN fails every comparison
        lab = ok ? (int)v : 0;
        return ok;
    } else if constexpr (std::is_signed<T>::value) {
        const bool ok = v >= T(0) && v <= T(4);
        lab = ok ? (int)v : 0;
        return ok;
    } else {
        lab = v <= T(4) ? (int)v : 0;
        return v <= T(4);
    }
}

// Wider (or signed) types: one warp per row, one lane per voxel -- a 32-voxel word is one coalesced 32-lane load and two
// ballots; lane j keeps word c0 + j, so that the 32 words of a batch go out as one coalesced warp store.  uint8 (the
// specialisation below): one word per thread, 16-byte loads and per-byte compares.
template <typename T>
__global__ void __launch_bounds__(BLOCK) k_init_planes(Params p, const T *__restrict__ vm, uint32_t *eraw) {
    const int nrows = (p.valid_hi - p.valid_lo) * p.Y, lane = threadIdx.x & 31;
    const int nwarps = gridDim.x * WARPS;
    bool bad = false;
    for (int r = blockIdx.x * WARPS + (threadIdx.x >> 5); r < nrows; r += nwarps) {
        const int y = r % p.Y, zl = p.valid_lo + r / p.Y;
        const T *src = vm + (long long)zl * p.plane_vox + (long long)y * p.X;
        for (int c0 = 0; c0 < p.XW; c0 += 32) {
            const int nw = min(32, p.XW - c0);
            uint32_t my_s = 0, my_e = 0;
#pragma unroll 4
            for (int j = 0; j < nw; ++j) {
                const int x = (c0 + j) * 32 + lane;
                int lab = 3;
                if (x < p.X) bad |= !label_value<T>(src[x], lab);
                const uint32_t s = __ballot_sync(FULL, lab <= 1), e = __ballot_sync(FULL, lab == 4);
                if (lane == j) { my_s = s; my_e = e; }
            }
            if (lane < nw) {
                const int c = c0 + lane;
                const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
                p.S[widx] = my_s;
                if (my_s) p.unitmap[unit_index(p, zl, y, c)] = 1;
                if (eraw) eraw[widx] = my_e;
            }
        }
    }
    if (bad) p.lstats[2 * p.L + ST_BAD_LABEL] = 1;
}
template <>
__global__ void __launch_bounds__(BLOCK) k_init_planes<uint8_t>(Params p, const uint8_t *__restrict__ vm, uint32_t *eraw) {
    const int nrows = (p.valid_hi - p.valid_lo) * p.Y, lane = threadIdx.x & 31;
    const int nwarps = gridDim.x * WARPS;
    bool bad = false;
    for (int r = blockIdx.x * WARPS + (threadIdx.x >> 5); r < nrows; r += nwarps)
    for (int c = lane; c < p.XW; c += 32) {
        const int y = r % p.Y, zl = p.valid_lo + r / p.Y;
        const uint8_t *src = vm + (long long)zl * p.plane_vox + (long long)y * p.X + (long long)c * 32;
        const int n = min(32, p.X - c * 32);
        uint32_t s = 0, e = 0;
        if (n == 32 && (((uintptr_t)src) & 15) == 0) {
            const uint4 *q = (const uint4 *)src;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint4 v = q[h];
                const uint32_t ws[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // per-byte compares (0xFF where equal), then the four byte flags gathered into four adjacent bits
                    // labels 0 / 1 are segmented, 2 / 3 are not, 4 is excluded (a map that a run returned can be fed back in:
                    // the bands are re-derived from the segmented set); anything above 4 is an error
                    const uint32_t z = __vcmpleu4(ws[k], 0x01010101u), f = __vcmpeq4(ws[k], 0x04040404u);
                    const int sh = h * 16 + k * 4;
                    s |= (((z & 0x01010101u) * 0x10204080u) >> 28) << sh;  // bytes 0..3 -> bits 0..3
                    e |= (((f & 0x01010101u) * 0x10204080u) >> 28) << sh;
                    bad |= __vcmpleu4(ws[k], 0x04040404u) != 0xFFFFFFFFu;
                }
            }
        } else {
            for (int b = 0; b < n; ++b) {
                const uint32_t byte = src[b];
                s |= (uint32_t)(byte <= 1u) << b;
                e |= (uint32_t)(byte == 4u) << b;
                bad |= byte > 4u;
            }
        }
        const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
        p.S[widx] = s;
        if (s) p.unitmap[unit_index(p, zl, y, c)] = 1;
        if (eraw) eraw[widx] = e;
    }
    if (bad) p.lstats[2 * p.L + ST_BAD_LABEL] = 1;
}

// E = Eraw & ~dil26(S) (VRG:137), and the initial band count.  In place on p.E (only the centre word is read).
__global__ void __launch_bounds__(BLOCK) k_init_bands(Params p) {
    const int lane = threadIdx.x & 31;
    const int zlo = max(p.valid_lo, p.own_lo - 1), zhi = min(p.valid_hi, p.own_hi + 1);
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(zhi - zlo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    long long nband = 0;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, zlo, nyb);
        const int c = un.sg * p.segw - 1 + lane;
        const bool own = un.zl >= p.own_lo && un.zl < p.own_hi;
        st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            if (!st.active) continue;
            const long long widx = (long long)un.zl * p.plane_words + (long long)y * p.WP + c;
            if (p.E) {
                const uint32_t eraw = p.E[widx];
                // ~s & vm & dil_s == outer, so the excluded voxels next to a seed are eraw & outer
                const uint32_t e = eraw & ~outer;
                if (e != eraw) p.E[widx] = e;
                outer &= ~e;
            }
            if (own) nband += __popc(inner) + __popc(outer);
        }
    }
    nband = warp_sum(nband);
    if (lane == 0 && nband) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_BAND], (unsigned long long)nband);
}

// region histograms and sizes over own planes (VRG:49-52, 149-150 as integer counts).
// Per-warp private shared histograms keep the shared-memory atomics off the few hot background levels.
template <int MODE, bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_init_hist(Params p, int copies) {
    extern __shared__ unsigned int s_h[];  // [copies][2L] when copies > 0
    for (int i = threadIdx.x; i < copies * 2 * p.L; i += BLOCK) s_h[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int *mine = copies ? s_h + (size_t)(warp % max(copies, 1)) * 2 * p.L : nullptr;
    const long long nrows = (long long)(p.own_hi - p.own_lo) * p.Y * p.XW;
    const long long nwarps = (long long)gridDim.x * WARPS;
    unsigned long long *hin = (unsigned long long *)p.lstats, *hout = hin + p.L;
    long long n_in = 0, n_out = 0, n_ex = 0;
    for (long long r = (long long)blockIdx.x * WARPS + warp; r < nrows; r += nwarps) {
        const int c = (int)(r % p.XW);
        const long long t = r / p.XW;
        const int y = (int)(t % p.Y), zl = p.own_lo + (int)(t / p.Y);
        const long long widx = (long long)zl * p.plane_words + (long long)y * p.WP + c;
        const uint32_t s = p.S[widx], e = p.E ? p.E[widx] : 0u;
        const int x = c * 32 + lane;
        if (x >= p.X) continue;
        const int l = level_at<MODE, LATTICE>(p, (long long)zl * p.plane_vox + (long long)y * p.X + x);
        const uint32_t bit = 1u << lane;
        if (s & bit) { n_in++; if (mine) atomicAdd(&mine[l], 1u); else atomicAdd(&hin[l], 1ull); }
        else if (!(e & bit)) { n_out++; if (mine) atomicAdd(&mine[p.L + l], 1u); else atomicAdd(&hout[l], 1ull); }
        else n_ex++;
    }
    n_in = warp_sum(n_in); n_out = warp_sum(n_out); n_ex = warp_sum(n_ex);
    if (lane == 0) {
        if (n_in) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_IN], (unsigned long long)n_in);
        if (n_out) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_OUT], (unsigned long long)n_out);
        if (n_ex) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_EXCL], (unsigned long long)n_ex);
    }
    if (copies) {
        __syncthreads();
        for (int i = threadIdx.x; i < 2 * p.L; i += BLOCK) {
            unsigned long long tot = 0;
            for (int k = 0; k < copies; ++k) tot += s_h[(size_t)k * 2 * p.L + i];
            if (tot) atomicAdd(&hin[i], tot);
        }
    }
}

// k_init_hist_private: same result as k_init_hist, without shared-memory atomics (2 cycles per lane on this part).
// Every lane of a warp owns a private uint16 histogram of the outside region in shared memory, laid out
// [level / 2][lane][level & 1]: a lane's counters all live in "its" bank, so a warp's 32 increments never conflict
// and each is a plain load / add / store.
// The (tiny) inside region and the excluded count go through global atomics.  hw = warps per block that fit.
template <int MODE, bool LATTICE>
__global__ void k_init_hist_private(Params p, int hw) {
    extern __shared__ uint16_t s_hp[];  // [hw][L][32]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < hw * ((p.L + 1) & ~1) * 32; i += blockDim.x) s_hp[i] = 0;
    __syncthreads();
    const int LP = (p.L + 1) & ~1;  // levels padded to an even count
    uint16_t *mine = s_hp + (size_t)warp * LP * 32 + lane * 2;
    const int nrows = (p.own_hi - p.own_lo) * p.Y;
    const int nwarps = gridDim.x * hw;
    unsigned long long *hin = (unsigned long long *)p.lstats, *hout = hin + p.L;
    long long n_in = 0, n_out = 0, n_ex = 0;
    int pending = 0;  // increments since the last flush: a uint16 bin cannot overflow before 65535
    auto flush = [&]() {
        __syncwarp();
        for (int l = 0; l < p.L; ++l) {
            unsigned int v = mine[(l >> 1) * 64 + (l & 1)];
            mine[(l >> 1) * 64 + (l & 1)] = 0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
            if (lane == 0 && v) atomicAdd(&hout[l], (unsigned long long)v);
        }
        pending = 0;
    };
    constexpr int U = 14;  // independent level loads in flight per lane: unconditional (clamped) so that they all issue first
    for (int r = blockIdx.x * hw + warp; r < nrows; r += nwarps) {
        const int y = r % p.Y, zl = p.own_lo + r / p.Y;
        const long long wbase = (long long)zl * p.plane_words + (long long)y * p.WP;
        const long long vbase = (long long)zl * p.plane_vox + (long long)y * p.X;
        for (int c32 = 0; c32 < p.XW; c32 += 32) {
            const int nw = min(32, p.XW - c32);
            const uint32_t srow = lane < nw ? p.S[wbase + c32 + lane] : 0u;
            const uint32_t erow = (p.E && lane < nw) ? p.E[wbase + c32 + lane] : 0u;
            for (int cb = 0; cb < nw; cb += U) {
                int lv[U];
#pragma unroll
                for (int k = 0; k < U; ++k) {
                    const int x = min((c32 + cb + k) * 32 + lane, p.X - 1);
                    lv[k] = level_at<MODE, LATTICE>(p, vbase + x);
                }
#pragma unroll
                for (int k = 0; k < U; ++k) {
                    const int c = c32 + cb + k;
                    const uint32_t sw = __shfl_sync(FULL, srow, (cb + k) & 31), ew = __shfl_sync(FULL, erow, (cb + k) & 31);
                    if (cb + k >= nw || c * 32 + lane >= p.X) continue;
                    const int l = lv[k];
                    const uint32_t bit = 1u << lane;
                    if (sw & bit) { n_in++; atomicAdd(&hin[l], 1ull); }
                    else if (ew & bit) n_ex++;
                    else { n_out++; mine[(l >> 1) * 64 + (l & 1)] += 1; }
                }
            }
            pending += nw;  // a lane adds at most one count per word: flushed long before a uint16 bin can wrap, whatever X
            if (pending > 60000) flush();
        }
    }
    flush();
    n_in = warp_sum(n_in); n_out = warp_sum(n_out); n_ex = warp_sum(n_ex);
    if (lane == 0) {
        if (n_in) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_IN], (unsigned long long)n_in);
        if (n_out) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_OUT], (unsigned long long)n_out);
        if (n_ex) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_EXCL], (unsigned long long)n_ex);
    }
}

// k_init_hist_shared: the result of k_init_hist, with the level source (fp64 intensities, or the uint16 index volume) streamed
// through a per-warp ring of TMA bulk-copy stages, exactly like the dense sweep: one stage = one row segment.  Needs 16-byte
// aligned row segments (host checks; k_init_hist_private and k_init_hist serve the rest).  ONE histogram per warp, updated
// by shared-memory atomics: 4 bytes per level and warp instead of the 64 of k_init_hist_private's 32 lane-private ones, so
// 12 warps fit beside their TMA rings where the lane-private layout beside the same rings left 5 (that variant ran at 22 %
// issue utilisation with 25 % of the DRAM bandwidth: too few warps to hide its own latency).
// Lanes of a warp that meet in a bin are serialised by the hardware; the outside region's levels spread over tens of bins.
constexpr int HIST_STAGES = 2;
template <int MODE, bool LATTICE>
__global__ void k_init_hist_shared(Params p, int hw, int stage_bytes) {
    using T = typename std::conditional<MODE == MODE_INDEX, uint16_t, double>::type;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int LP = (p.L + 1) & ~1;
    uint64_t *bars = (uint64_t *)smem_raw;                                                  // [hw][HIST_STAGES]
    unsigned char *stages = smem_raw + ((hw * HIST_STAGES * 8 + 127) & ~127);                // [hw][HIST_STAGES][stage_bytes]
    unsigned int *s_hp = (unsigned int *)(stages + (size_t)hw * HIST_STAGES * stage_bytes);  // [hw][LP]
    for (int i = threadIdx.x; i < hw * LP; i += blockDim.x) s_hp[i] = 0;
    uint64_t *mybar = bars + warp * HIST_STAGES;
    unsigned char *mystage = stages + (size_t)warp * HIST_STAGES * stage_bytes;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < HIST_STAGES; ++s) mbar_init(mybar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned int *mine = s_hp + (size_t)warp * LP;
    unsigned long long *hin = (unsigned long long *)p.lstats, *hout = hin + p.L;
    const long long nrows = (long long)(p.own_hi - p.own_lo) * p.Y * p.nseg;
    const long long stride = (long long)gridDim.x * hw;
    auto decode = [&](long long r, int &zl, int &y, int &sg) {
        sg = (int)(r % p.nseg);
        const long long t = r / p.nseg;
        y = (int)(t % p.Y);
        zl = p.own_lo + (int)(t / p.Y);
    };
    auto issue = [&](long long r, int s) {  // lane 0 only
        int zl, y, sg;
        decode(r, zl, y, sg);
        const int x0 = sg * p.segw * 32;
        const uint32_t bytes = (uint32_t)min(p.segw * 32, p.X - x0) * (uint32_t)sizeof(T);
        const long long vox = (long long)zl * p.plane_vox + (long long)y * p.X + x0;
        const void *src = MODE == MODE_INDEX ? (const void *)(p.index + vox) : (const void *)(p.data + vox);
        mbar_expect_tx(mybar + s, bytes);
        tma_bulk_load(mystage + (size_t)s * stage_bytes, src, bytes, mybar + s);
    };
    long long pre = (long long)blockIdx.x * hw + warp, cur = pre;
#pragma unroll
    for (int s = 0; s < HIST_STAGES; ++s) {
        if (pre < nrows) {
            if (lane == 0) issue(pre, s);
            pre += stride;
        }
    }
    long long n_in = 0, n_out = 0, n_ex = 0;
    int stage = 0;
    uint32_t parity = 0;
    for (; cur < nrows; cur += stride) {
        int zl, y, sg;
        decode(cur, zl, y, sg);
        const int cfirst = sg * p.segw, nw = min(p.segw, p.XW - cfirst);
        const long long wbase = (long long)zl * p.plane_words + (long long)y * p.WP + cfirst;
        // lane j holds word j of the segment: region sizes by popcount, per-voxel work below only for the histogram
        const uint32_t vrow = lane < nw ? valid_mask(p, cfirst + lane) : 0u;
        const uint32_t srow = lane < nw ? p.S[wbase + lane] & vrow : 0u;
        const uint32_t erow = (p.E && lane < nw) ? p.E[wbase + lane] & vrow & ~srow : 0u;
        const uint32_t orow = vrow & ~srow & ~erow;  // outside region: the histogram this kernel keeps in shared memory
        n_in += __popc(srow); n_ex += __popc(erow); n_out += __popc(orow);
        const T *sv = (const T *)(mystage + (size_t)stage * stage_bytes) + lane;
        mbar_wait(mybar + stage, parity);
        constexpr int BW = 10;
#pragma unroll
        for (int jb = 0; jb < WORDS_PER_WARP; jb += BW) {
            if (jb >= nw) break;  // warp-uniform
            int lv[BW];
#pragma unroll
            for (int k = 0; k < BW; ++k) {
                if (MODE == MODE_INDEX) lv[k] = (int)sv[(jb + k) * 32];
                else lv[k] = level_of<LATTICE>(p, (double)sv[(jb + k) * 32]);
            }
            // one shared-memory atomic per outside voxel (words past the row end hold stale bytes: their level is forced to 0
            // and they add nothing)
            uint32_t segbits = 0;
#pragma unroll
            for (int k = 0; k < BW; ++k) {
                const uint32_t ow = __shfl_sync(FULL, orow, (jb + k) & 31), sw = __shfl_sync(FULL, srow, (jb + k) & 31);
                const uint32_t inc = (ow >> lane) & 1u, seg = (sw >> lane) & 1u;
                const int l = (inc | seg) ? lv[k] : 0;
                lv[k] = l;
                segbits |= seg << k;
                if (inc) atomicAdd(mine + l, 1u);
            }
            if (__any_sync(FULL, segbits != 0u)) {  // the (tiny) inside region goes through global atomics
#pragma unroll
                for (int k = 0; k < BW; ++k)
                    if (segbits & (1u << k)) atomicAdd(&hin[lv[k]], 1ull);
            }
        }
        __syncwarp();
        if (pre < nrows) {  // the stage is drained: re-arm it for a later row
            if (lane == 0) issue(pre, stage);
            pre += stride;
        }
        if (++stage == HIST_STAGES) { stage = 0; parity ^= 1u; }
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.L; l += blockDim.x) {  // one global atomic per level and block
        unsigned long long v = 0;
        for (int w = 0; w < hw; ++w) v += s_hp[(size_t)w * LP + l];
        if (v) atomicAdd(&hout[l], v);
    }
    n_in = warp_sum(n_in); n_out = warp_sum(n_out); n_ex = warp_sum(n_ex);
    if (lane == 0) {
        if (n_in) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_IN], (unsigned long long)n_in);
        if (n_out) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_OUT], (unsigned long long)n_out);
        if (n_ex) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_EXCL], (unsigned long long)n_ex);
    }
}

// ---------------------------------------------------------------------------------------------
// distinct intensity levels: open-addressing hash set over the fp64 bit patterns
constexpr unsigned long long HEMPTY = 0xFFFFFFFFFFFFFFFFull;
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(BLOCK) k_scan_levels(const double *__restrict__ data, long long n, unsigned long long *table,
                                                       int cap_mask, int *count, int max_count, int *flags) {
    unsigned long long last = HEMPTY;
    constexpr int U = 8;  // loads in flight per thread (the hash probe below is a dependent chain)
    const long long nth = (long long)gridDim.x * BLOCK;
    for (long long i0 = (long long)blockIdx.x * BLOCK + threadIdx.x; i0 < n; i0 += nth * U) {
        double vs[U];
#pragma unroll
        for (int k = 0; k < U; ++k) vs[k] = data[min(i0 + k * nth, n - 1)];  // clamped: a repeat of the last voxel is harmless
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const double v = vs[k] + 0.0;
            if (!isfinite(v)) { flags[0] = 1; continue; }
            const unsigned long long key = (unsigned long long)__double_as_longlong(v);
            if (key == last) continue;
            last = key;
            unsigned int h = (unsigned int)mix64(key) & cap_mask;
            while (true) {
                const unsigned long long cur = table[h];
                if (cur == key) break;
                if (cur == HEMPTY) {
                    if (*(volatile int *)count >= max_count) { flags[1] = 1; break; }
                    const unsigned long long old = atomicCAS(&table[h], HEMPTY, key);
                    if (old == HEMPTY) { atomicAdd(count, 1); break; }
                    if (old == key) break;
                }
                h = (h + 1) & cap_mask;
            }
        }
    }
}

// the keys of the hash set, densely packed (unordered; the host sorts the few hundred values)
__global__ void __launch_bounds__(BLOCK) k_compact_levels(const unsigned long long *__restrict__ table, int cap,
                                                          unsigned long long *__restrict__ out, int *n_out, int max_out) {
    for (int i = blockIdx.x * BLOCK + threadIdx.x; i < cap; i += gridDim.x * BLOCK) {
        const unsigned long long k = table[i];
        if (k != HEMPTY) {
            const int j = atomicAdd(n_out, 1);
            if (j < max_out) out[j] = k;
        }
    }
}

template <bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_build_index(Params p, const double *__restrict__ data, uint16_t *index, long long n) {
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK)
        index[i] = (uint16_t)level_of<LATTICE>(p, data[i]);
}

// ---------------------------------------------------------------------------------------------
// outputs: canonical labels (VRG:21) or the 0/1 segmented map as T, own planes only, straight into a buffer of the caller's
// dtype.  One-byte types: 4 voxels (bytes) per lane and store; wider types: one voxel per lane, a warp writes the 32 voxels of
// one word per store (32 * sizeof(T) consecutive bytes).
template <typename T>
__global__ void __launch_bounds__(BLOCK) k_labels(Params p, T *__restrict__ out, int seg_only) {
    const int lane = threadIdx.x & 31;
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(p.own_hi - p.own_lo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, p.own_lo, nyb);
        const int c0 = un.sg * p.segw - 1, c = c0 + lane;
        st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            const long long widx = (long long)un.zl * p.plane_words + (long long)y * p.WP + c;
            const uint32_t e = (p.E && st.active) ? p.E[widx] : 0u;
            outer &= ~e;
            if constexpr (sizeof(T) == 1) {
                // 4 voxels (bytes) per lane and store: a warp writes 128 consecutive voxels = 4 words per step
                uint8_t *rowout = (uint8_t *)out + ((long long)(un.zl - p.own_lo) * p.Y + y) * p.X;
                for (int j0 = 1; j0 <= p.segw; j0 += 4) {
                    if (c0 + j0 >= p.XW) break;
                    const int src = j0 + (lane >> 3);  // lane that holds this lane's word
                    const uint32_t sj = __shfl_sync(FULL, s, src), ij = __shfl_sync(FULL, inner, src);
                    const uint32_t oj = __shfl_sync(FULL, outer, src), ej = __shfl_sync(FULL, e, src);
                    if (src > p.segw) continue;
                    const int x = (c0 + src) * 32 + (lane & 7) * 4;
                    uint32_t pack = 0;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const uint32_t bit = 1u << ((lane & 7) * 4 + b);
                        uint32_t lab;
                        if (seg_only) lab = (sj & bit) ? 1u : 0u;
                        else lab = (sj & bit) ? ((ij & bit) ? 1u : 0u) : ((ej & bit) ? 4u : ((oj & bit) ? 2u : 3u));
                        pack |= lab << (8 * b);
                    }
                    if (x + 3 < p.X && ((((uintptr_t)(rowout + x)) & 3) == 0)) *(uint32_t *)(rowout + x) = pack;
                    else
                        for (int b = 0; b < 4; ++b)
                            if (x + b < p.X) rowout[x + b] = (uint8_t)(pack >> (8 * b));
                }
            } else {
                T *rowout = out + ((long long)(un.zl - p.own_lo) * p.Y + y) * p.X;
                const uint32_t bit = 1u << lane;
                for (int j = 1; j <= p.segw; ++j) {
                    if (c0 + j >= p.XW) break;
                    const uint32_t sj = __shfl_sync(FULL, s, j), ij = __shfl_sync(FULL, inner, j);
                    const uint32_t oj = __shfl_sync(FULL, outer, j), ej = __shfl_sync(FULL, e, j);
                    int lab;
                    if (seg_only) lab = (sj & bit) ? 1 : 0;
                    else lab = (sj & bit) ? ((ij & bit) ? 1 : 0) : ((ej & bit) ? 4 : ((oj & bit) ? 2 : 3));
                    const int x = (c0 + j) * 32 + lane;
                    if (x < p.X) rowout[x] = (T)lab;
                }
            }
        }
    }
}

// Row compaction on the device (vrg_band_rows_device).  A warp walks a unit (ROWS_PER_UNIT rows of one row segment, the
// Strip layout: lanes 1..segw hold the segment's words) and takes from each row the word that WHICH selects:
//   0  S, the segmented voxels                  1  the inner band S & dil26(~S)  (label 1)
//   2  the outer band ~S & ~E & dil26(S)  (label 2)
// -- the bands derived as k_labels derives them.  Every lane outside 1..segw, or beyond the row, holds 0.
template <int WHICH>
__device__ __forceinline__ uint32_t row_word(const Params &p, Strip &st, int zl, int y, int c, int lane) {
    if constexpr (WHICH == 0) {
        const bool active = c >= 0 && c < p.XW && lane >= 1 && lane <= p.segw;
        return active ? p.S[(long long)zl * p.plane_words + (long long)y * p.WP + c] : 0u;
    } else {
        uint32_t s, inner, outer;
        st.step(p, y, s, inner, outer);
        if constexpr (WHICH == 1) return inner;
        const uint32_t e = (p.E && st.active) ? p.E[(long long)zl * p.plane_words + (long long)y * p.WP + c] : 0u;
        return outer & ~e;
    }
}
// slot of a row segment of the own planes: (row, segment) in C order, so that the scanned counts give C-ordered rows
__device__ __forceinline__ long long row_slot(const Params &p, int zl, int y, int sg) {
    return ((long long)(zl - p.own_lo) * p.Y + y) * p.nseg + sg;
}
// popcount of every own-plane row segment's selected words ...
template <int WHICH>
__global__ void __launch_bounds__(BLOCK) k_seg_count(Params p, long long *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(p.own_hi - p.own_lo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, p.own_lo, nyb);
        const int c = un.sg * p.segw - 1 + lane;
        if (WHICH) st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            const long long n = warp_sum(__popc(row_word<WHICH>(p, st, un.zl, y, c, lane)));
            if (lane == 0) counts[row_slot(p, un.zl, y, un.sg)] = n;
        }
    }
}
// ... and, behind an exclusive scan of those counts, the (z, y, x) triples of the set bits in C order, z_begin added: a warp
// scan of the lanes' popcounts gives each lane its first output row.  Rows from `cap` on are not written.
template <int WHICH>
__global__ void __launch_bounds__(BLOCK) k_seg_scatter(Params p, const long long *__restrict__ offs, long long *__restrict__ rows,
                                                       long long cap, long long z_begin) {
    const int lane = threadIdx.x & 31;
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(p.own_hi - p.own_lo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, p.own_lo, nyb);
        const int c = un.sg * p.segw - 1 + lane;
        if (WHICH) st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t w = row_word<WHICH>(p, st, un.zl, y, c, lane);
            if (__ballot_sync(FULL, w != 0u) == 0u) continue;
            const int n = __popc(w);
            int incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            long long k = offs[row_slot(p, un.zl, y, un.sg)] + incl - n;
            while (w) {
                const int b = __ffs(w) - 1;
                w &= w - 1;
                if (k < cap) {
                    rows[3 * k] = z_begin + (un.zl - p.own_lo);
                    rows[3 * k + 1] = y;
                    rows[3 * k + 2] = (long long)c * 32 + b;
                }
                ++k;
            }
        }
    }
}

// update()'s two Parzen sum volumes (VRG:132-133,151-155 as the host path writes them), own planes, C order: at every inner /
// outer band voxel pin * n_in and pout * n_out of its level in the current decision table (one rounding each, as NumPy's
// pin[idx] * n_in), 0.0 everywhere else.  The level comes from the sweep's lookup (level_of); intensities are read at band
// voxels only.  A warp writes the 32 voxels of one word per store into each volume (2 x 256 consecutive bytes).
template <bool LATTICE>
__global__ void __launch_bounds__(BLOCK) k_band_sums_dense(Params p, double *__restrict__ pin_out, double *__restrict__ pout_out) {
    const int lane = threadIdx.x & 31;
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(p.own_hi - p.own_lo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    const double n_in = (double)p.gstats[2 * p.L + ST_N_IN], n_out = (double)p.gstats[2 * p.L + ST_N_OUT];
    const uint32_t bit = 1u << lane;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, p.own_lo, nyb);
        const int c0 = un.sg * p.segw - 1, c = c0 + lane;
        st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            const uint32_t e = (p.E && st.active) ? p.E[(long long)un.zl * p.plane_words + (long long)y * p.WP + c] : 0u;
            const uint32_t band = inner | (outer & ~e);
            const double *rowin = p.data + ((long long)un.zl * p.Y + y) * p.X;
            const long long rowout = ((long long)(un.zl - p.own_lo) * p.Y + y) * p.X;
            for (int j = 1; j <= p.segw; ++j) {
                if (c0 + j >= p.XW) break;
                const uint32_t bj = __shfl_sync(FULL, band, j);
                const int x = (c0 + j) * 32 + lane;
                if (x >= p.X) continue;
                double a = 0.0, b = 0.0;
                if (bj & bit) {
                    const int l = level_of<LATTICE>(p, rowin[x]);
                    a = p.pin[l] * n_in;
                    b = p.pout[l] * n_out;
                }
                pin_out[rowout + x] = a;
                pout_out[rowout + x] = b;
            }
        }
    }
}

// update()'s state from the caller's two maps, each read in its own dtype, into the handle's uint8 valueMap (local planes):
// the valueMap pass writes 4 where valueMap == 4 and 3 elsewhere, the segmentedMap pass then 0 where segmentedMap == 1
// (VRG:124: what the host update() reads of its inputs).  vrg_init takes the result as any uint8 map.
template <typename T>
__global__ void __launch_bounds__(BLOCK) k_state_from_map(const T *__restrict__ map, uint8_t *__restrict__ vm, long long n,
                                                          int seg_pass) {
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) {
        const T v = map[i];
        if (!seg_pass) vm[i] = v == T(4) ? 4 : 3;
        else if (v == T(1)) vm[i] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// Position-sensitive 64-bit hash of a label volume (one byte per voxel): sum over the voxels of
// mix64((global linear index << 3) | label) modulo 2^64.  Additive, so the hashes of z-slabs add up to the hash of the whole
// volume whatever the partition -- multi-GPU runs are compared with the single-volume oracle by one number per slab.
__global__ void __launch_bounds__(BLOCK) k_hash_labels(const uint8_t *__restrict__ lab, long long n, long long base,
                                                       unsigned long long *out) {
    unsigned long long acc = 0;
    const long long nth = (long long)gridDim.x * BLOCK;
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += nth)
        acc += mix64(((unsigned long long)(base + i) << 3) | (unsigned long long)lab[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// np.count_nonzero(dataArray) of the own planes (the second printed line, VRG:95): -0.0 counts as zero, NaN as non-zero
__global__ void __launch_bounds__(BLOCK) k_count_nonzero(const double *__restrict__ data, long long n, unsigned long long *out) {
    unsigned long long acc = 0;
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) acc += data[i] != 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

__global__ void __launch_bounds__(BLOCK) k_expand_i64(const uint8_t *__restrict__ src, long long *__restrict__ dst, long long n) {
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) dst[i] = src[i];
}

// ---------------------------------------------------------------------------------------------
// device-resident flip rows (vrg_apply_flips_device): out[0] = how many lie outside the own planes, out[1] = the first of them
// (the caller sets it to ~0 beforehand)
__global__ void __launch_bounds__(BLOCK) k_check_flips(Params p, const long long *__restrict__ coords, long long n, long long z_begin,
                                                       unsigned long long *out) {
    unsigned long long bad = 0;
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) {
        const long long z = coords[3 * i] - z_begin + p.own_lo, y = coords[3 * i + 1], x = coords[3 * i + 2];
        if (z < p.own_lo || z >= p.own_hi || y < 0 || y >= p.Y || x < 0 || x >= p.X) {
            ++bad;
            atomicMin(&out[1], (unsigned long long)i);
        }
    }
    if (bad) atomicAdd(&out[0], bad);
}

// update() with caller-chosen flips (VRG:124, flipedPoints given): the listed voxels' bits go into F ...
__global__ void __launch_bounds__(BLOCK) k_set_flips(Params p, const long long *__restrict__ coords, long long n, long long z_begin) {
    for (long long i = (long long)blockIdx.x * BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * BLOCK) {
        const long long z = coords[3 * i] - z_begin + p.own_lo, y = coords[3 * i + 1], x = coords[3 * i + 2];
        if (z < p.own_lo || z >= p.own_hi || y < 0 || y >= p.Y || x < 0 || x >= p.X) continue;  // the host validated the list
        atomicOr(&p.F[z * p.plane_words + y * p.WP + (x >> 5)], 1u << (x & 31));
    }
}
// ... and are then restricted to the band voxels (a listed voxel that is in neither band does nothing in the reference
// beyond absorbing label 4 around it, VRG:167-170,198): row flags, front list and the flip count as the sweep leaves them.
__global__ void __launch_bounds__(BLOCK) k_mask_flips(Params p) {
    const int lane = threadIdx.x & 31;
    const int nyb = (p.Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
    const long long nunits = (long long)(p.own_hi - p.own_lo) * nyb * p.nseg;
    const long long nwarps = (long long)gridDim.x * WARPS;
    long long flips = 0;
    Strip st;
    for (long long u = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5); u < nunits; u += nwarps) {
        const Unit un = decode_unit(p, u, p.own_lo, nyb);
        const int c = un.sg * p.segw - 1 + lane;
        st.begin(p, un.zl, un.y0, c, lane);
        for (int y = un.y0; y < un.y1; ++y) {
            uint32_t s, inner, outer;
            st.step(p, y, s, inner, outer);
            const long long widx = (long long)un.zl * p.plane_words + (long long)y * p.WP + c;
            const long long ridx = ((long long)un.zl * p.Y + y) * p.nseg + un.sg;
            if (p.E != nullptr && outer) outer &= ~p.E[widx];
            const uint32_t raw = st.active ? p.F[widx] : 0u;
            const uint32_t f = raw & (inner | outer);
            if (__ballot_sync(FULL, raw != 0u) == 0u) continue;  // the host cleared F, C and the row flags beforehand
            if (st.active && f != raw) p.F[widx] = f;
            if (__ballot_sync(FULL, f != 0u) != 0u && lane == 0) {
                p.rowflag[ridx] = 1;
                int *fl = front_list(p, (int)(p.ctrl[C_SWEEPS] & 1));
                fl[1 + atomicAdd(&fl[0], 1)] = (int)ridx;
            }
            flips += __popc(f);
        }
    }
    flips = warp_sum(flips);
    if (lane == 0 && flips) atomicAdd((unsigned long long *)&p.lstats[2 * p.L + ST_N_FLIPS], (unsigned long long)flips);
}
// bookkeeping in front of an applied flip list: the state k_table leaves in front of a sweep, with the flips forced on
__global__ void k_prepare_apply(Params p) {
    if (threadIdx.x || blockIdx.x) return;
    p.ctrl[C_STATUS] = RUNNING;
    p.ctrl[C_APPLY] = 1;
    p.ctrl[C_FULL_SWEEP] = p.ctrl[C_SWEEPS] + 1;
    p.lstats[2 * p.L + ST_N_FLIPS] = 0;
    front_list(p, (int)(p.ctrl[C_SWEEPS] & 1))[0] = 0;
    dirty_list(p, (int)((p.ctrl[C_SWEEPS] + 1) & 1))[0] = 0;
}

// the next sweep must look at every band voxel (after caller-chosen flips)
__global__ void k_force_full_sweep(Params p) {
    if (threadIdx.x == 0 && blockIdx.x == 0) p.ctrl[C_FULL_SWEEP] = p.ctrl[C_SWEEPS] + 1;
}

}  // namespace vrg
