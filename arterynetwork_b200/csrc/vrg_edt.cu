// Exact Euclidean distance transform of a binary mask (SURVEY.md section 8(f) N3): the step after the VRG path.
// Reference call sites: Code/manualCorrectionGUI.py:248 (vessel radii from the VRG output mask) and
// Code/generateVesselVolume.py:183 (distance to the brain-mask boundary), both
// scipy.ndimage.distance_transform_edt(mask) with default arguments: every non-zero voxel gets its Euclidean distance
// to the nearest zero voxel, float64, unit spacing.
//
// Separable and exact in integers (Meijster, Roerdink, Hesselink 2000):
//   pass x   g(x)  = (distance to the nearest zero voxel of the same row)^2: a prefix-max / suffix-min scan, one warp per row
//   pass y,z out(u) = min_i (u - i)^2 + in(i) along the axis: lower envelope of parabolas, one thread per line, O(n) per
//            line whatever the distances are; neighbouring threads own neighbouring x, so every access of the scan
//            (input, envelope stacks, output) is a coalesced row of the volume
//   sqrt     fp64 square root of the integer squared distance (correctly rounded, as NumPy's)
// Squared distances are int32 (axes <= 32768 would overflow: axes are limited to 16384, 3 * 16384^2 < 2^30).
#include "../../include/vrg_b200.h"

#include "vrg_scratch.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>

void vrg_set_error_internal(const char *msg);  // vrg_b200.cu: text behind vrg_last_error()

namespace {

using vrg_scratch::Buf;

constexpr int EDT_INF = 1 << 30;  // "no zero voxel seen yet"; sums with k^2 are formed in 64 bits
constexpr unsigned FULLMASK = 0xFFFFFFFFu;

// pass x: one warp per row.  The row's foreground bits go to shared memory (and to the packed bit volume the other passes
// read); the nearest zero to the left / right of a voxel is then bit arithmetic inside its own 32-voxel word, or the running
// "last zero seen" of the words before it / the per-word "next zero" table of the words behind it.  Only FOREGROUND voxels
// get their x-distance stored (uint16; 0xFFFF = no zero in this row): the background's distance is 0 and is implied by its
// bit, so a thin mask costs the pass one byte read per voxel and next to nothing else.
__global__ void __launch_bounds__(256) k_edt_rows(const uint8_t *__restrict__ mask, uint16_t *__restrict__ d1, uint32_t *__restrict__ bits,
                                                  long long nrows, int X, int XW) {
    extern __shared__ uint32_t sm_rows[];  // per warp: XW words of bits, XW ints "last zero before the word", XW "next zero behind it"
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *rb = sm_rows + (size_t)warp * 3 * XW;
    int *lf = (int *)(rb + XW), *rf = lf + XW;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    const int NONE_L = -(1 << 20), NONE_R = 1 << 20;
    const uint32_t tail = (X & 31) ? ((1u << (X & 31)) - 1u) : 0xFFFFFFFFu;
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + warp; r < nrows; r += nwarps) {
        const uint8_t *row = mask + r * X;
        uint32_t seen = 0u;  // OR of the foreground words this lane stored
        if ((X & 3) == 0 && (((uintptr_t)row) & 3) == 0) {
            // 128 voxels per step: a 4-byte load per lane, its four "non-zero" bits, then the eight lanes of each 32-voxel word
            // OR their nibbles together (three shuffles)
            for (int w0 = 0; w0 < XW; w0 += 4) {
                const int x = 32 * w0 + 4 * lane;
                uint32_t nib = 0xFu;  // beyond the row end there is no voxel, hence no zero
                if (x < X) {
                    const uint32_t v = *(const uint32_t *)(row + x);
                    const uint32_t nz = (((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v) & 0x80808080u;
                    nib = ((nz >> 7) & 1u) | ((nz >> 14) & 2u) | ((nz >> 21) & 4u) | ((nz >> 28) & 8u);
                }
                uint32_t word = nib << (4 * (lane & 7));
                word |= __shfl_xor_sync(FULLMASK, word, 1);
                word |= __shfl_xor_sync(FULLMASK, word, 2);
                word |= __shfl_xor_sync(FULLMASK, word, 4);
                const int w = w0 + (lane >> 3);
                if ((lane & 7) == 0 && w < XW) {
                    const uint32_t real = w == XW - 1 ? (word & tail) : word;
                    rb[w] = word;
                    bits[r * XW + w] = real;
                    seen |= real;
                }
            }
        } else {
            for (int w = 0; w < XW; ++w) {
                const int x = 32 * w + lane;
                const bool fg = x < X ? row[x] != 0 : true;
                const uint32_t word = __ballot_sync(FULLMASK, fg);
                if (lane == 0) {
                    const uint32_t real = w == XW - 1 ? (word & tail) : word;
                    rb[w] = word;
                    bits[r * XW + w] = real;
                    seen |= real;
                }
            }
        }
        if (!__any_sync(FULLMASK, seen != 0u)) continue;  // a row of background: nothing to store
        __syncwarp();
        // per word: the last zero in the words before it, the next zero in the words behind it (warp scans, 32 words per step)
        int carry = NONE_L;
        for (int c = 0; c < XW; c += 32) {
            const int w = c + lane;
            const uint32_t zw = w < XW ? ~rb[w] : 0u;
            int v = zw ? 32 * w + 31 - __clz(zw) : NONE_L;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULLMASK, v, o);
                if (lane >= o) v = max(v, t);
            }
            int ex = __shfl_up_sync(FULLMASK, v, 1);
            if (lane == 0) ex = NONE_L;
            if (w < XW) lf[w] = max(ex, carry);
            carry = max(carry, __shfl_sync(FULLMASK, v, 31));
        }
        carry = NONE_R;
        for (int c = ((XW - 1) / 32) * 32; c >= 0; c -= 32) {
            const int w = c + lane;
            const uint32_t zw = w < XW ? ~rb[w] : 0u;
            int v = zw ? 32 * w + __ffs(zw) - 1 : NONE_R;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_down_sync(FULLMASK, v, o);
                if (lane + o < 32) v = min(v, t);
            }
            int ex = __shfl_down_sync(FULLMASK, v, 1);
            if (lane == 31) ex = NONE_R;
            if (w < XW) rf[w] = min(ex, carry);
            carry = min(carry, __shfl_sync(FULLMASK, v, 0));
        }
        __syncwarp();
        // the words that hold foreground, one after the other (lane = voxel of the word)
        for (int c = 0; c < XW; c += 32) {
            const int wl = c + lane;
            unsigned todo = __ballot_sync(FULLMASK, wl < XW && (wl == XW - 1 ? (rb[wl] & tail) : rb[wl]) != 0u);
            while (todo) {
                const int w = c + __ffs(todo) - 1;
                todo &= todo - 1;
                const uint32_t word = rb[w], zw = ~word;
                const int x = 32 * w + lane;
                if (x < X && ((word >> lane) & 1u)) {
                    const uint32_t below = zw & ((2u << lane) - 1u), above = zw & ~((1u << lane) - 1u);
                    const int xl = below ? 32 * w + 31 - __clz(below) : lf[w];
                    const int xr = above ? 32 * w + __ffs(above) - 1 : rf[w];
                    const int d = min(x - xl, xr - x);
                    d1[r * X + x] = d >= 32768 ? (uint16_t)0xFFFF : (uint16_t)d;
                }
            }
        }
        __syncwarp();
    }
}

// Summary of the bit volume for the line passes: one word per (line-warp, batch of 8 steps) = OR of the warp's bit words of
// the batch's rows and of the row before and the row behind it.  Zero = the batch is background and no voxel of it can
// matter to anybody's envelope: the line passes skip it after one load.
__global__ void __launch_bounds__(256) k_edt_summary(const uint32_t *__restrict__ bits, uint32_t *__restrict__ sum, long long nouter, int len,
                                                     int XW, long long bit_outer_stride, long long bit_stride) {
    const int nb = (len + 7) / 8;
    const long long total = nouter * nb * XW;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int xw = (int)(i % XW);
        const long long t = i / XW;
        const int ub = (int)(t % nb);
        const long long outer = t / nb;
        const uint32_t *bw = bits + outer * bit_outer_stride + xw;
        uint32_t acc = 0u;
#pragma unroll
        for (int k = -1; k <= 8; ++k) {
            const int u = 8 * ub + k;
            if (u >= 0 && u < len) acc |= bw[(long long)u * bit_stride];
        }
        sum[i] = acc;  // layout [outer][batch][xw]
    }
}

// pass y / z: out(u) = min_i (u - i)^2 + f(i) along one axis: lower envelope of parabolas (Meijster).  Thread = one line;
// the 32 lanes of a warp sit on 32 neighbouring x of one row (lines are enumerated over rows padded to whole words), walk
// u in lockstep, and every access is a coalesced row segment of the volume.
// Where f(u) = 0 the answer is 0, and a zero shields everything behind it ((u - i)^2 + f(i) > (u - z)^2 for i beyond a zero
// at z): only the zeros next to a positive voxel can matter to the envelope.  f(u) = 0 exactly at the background voxels, in
// every pass, so WHICH voxels are zero comes from the packed foreground bits (one 4-byte word per warp and step) and the
// input volume is read at foreground voxels only; the y pass also writes foreground voxels only (nobody reads the rest).
// For a vessel mask almost every voxel is background: the two line passes together read the bit volume four times and a few
// per cent of the distance volumes, and write the result once.  For a solid mask (the brain) the scan is O(n) per line
// whatever the distances; its envelope stack lives in global memory, one packed 8-byte entry (apex | start of its reign |
// height) per push.  A line is one dependent chain: inputs are fetched eight steps ahead in both directions, and the pops
// of the backward scan (entries below the top no longer change) fetch four stack entries at once.
// OUT: 0 = squared distance, int32, foreground voxels only (y pass); 1 = distance, float64, every voxel, raises *flag where
// no zero voxel exists (z pass of the public EDT); 2 = squared distance, int32, every voxel (z pass for the vessel-mask rule).
template <typename TIn> __device__ __forceinline__ long long edt_in(TIn v);
template <> __device__ __forceinline__ long long edt_in<uint16_t>(uint16_t v) { return v == 0xFFFF ? (long long)EDT_INF : (long long)v * v; }
template <> __device__ __forceinline__ long long edt_in<int>(int v) { return v; }
__device__ __forceinline__ unsigned long long edt_pack(int s, int t, int g) {
    return ((unsigned long long)(uint32_t)g << 32) | ((unsigned long long)(uint32_t)t << 16) | (unsigned long long)(uint32_t)s;
}

template <typename TIn, int OUT>
__global__ void __launch_bounds__(128) k_edt_lines(const TIn *__restrict__ in, void *__restrict__ outv, const uint32_t *__restrict__ bits,
                                                   unsigned long long *__restrict__ stack, long long nouter, int len, long long stride,
                                                   int X, int XW, long long outer_stride, long long bit_outer_stride,
                                                   long long bit_stride, const uint32_t *__restrict__ sum, int *flag) {
    const int lane = threadIdx.x & 31;
    const long long padded = (long long)XW * 32, nlines = nouter * padded;
    bool inf = false;
    for (long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x; line < nlines; line += (long long)gridDim.x * blockDim.x) {
        const long long outer = line / padded;
        const int x = (int)(line % padded);
        const bool active = x < X;
        const long long base = outer * outer_stride + (active ? x : 0);
        const uint32_t *bw = bits + outer * bit_outer_stride + (x >> 5);  // warp-uniform
        const int nb = (len + 7) / 8;
        const uint32_t *sw = sum + (outer * nb) * XW + (x >> 5);        // warp-uniform; batch b at sw[b * XW]
        const TIn *f = in + base;
        unsigned long long *st = stack + base;
        // forward scan.  Registers hold the top of the stack (sq, tq, fq = f(sq)); q = depth - 1, -1 = empty.
        int q = -1, sq = 0, tq = 0;
        bool prev = false;
        long long fq = 0;
        constexpr int PF = 8;
        static_assert(PF == 8, "the summary words describe batches of 8 steps");
        for (int u0 = 0; u0 < len; u0 += PF) {
            // eight rows of background under the whole warp, behind a row of background and before one (warp-uniform): no
            // voxel of them can matter to anybody's envelope
            if (sw[(long long)(u0 >> 3) * XW] == 0u) { prev = false; continue; }
            uint32_t wd[PF + 1];
#pragma unroll
            for (int k = 0; k <= PF; ++k) wd[k] = u0 + k < len ? bw[(long long)(u0 + k) * bit_stride] : 0u;
            bool bit[PF + 1];
            TIn fpre[PF];
#pragma unroll
            for (int k = 0; k <= PF; ++k) bit[k] = active && ((wd[k] >> lane) & 1u);
#pragma unroll
            for (int k = 0; k < PF; ++k) fpre[k] = bit[k] ? f[(long long)(u0 + k) * stride] : (TIn)0;
#pragma unroll
            for (int k = 0; k < PF; ++k) {
                const int u = u0 + k;
                if (u >= len) break;
                const long long fu = bit[k] ? edt_in<TIn>(fpre[k]) : 0;
                const bool wanted = bit[k] ? fu < EDT_INF : (active && (prev || bit[k + 1]));
                prev = bit[k];
                if (!wanted) continue;  // background away from any foreground, or an infinite parabola
                while (q >= 0) {
                    // F(tq, sq) > F(tq, u): the new parabola is already lower where the top one starts to reign: pop
                    const long long a = (long long)(tq - sq) * (tq - sq) + fq, b = (long long)(tq - u) * (tq - u) + fu;
                    if (a <= b) break;
                    --q;
                    if (q >= 0) {
                        const unsigned long long e = st[(long long)q * stride];
                        sq = (int)(e & 0xFFFFu); tq = (int)((e >> 16) & 0xFFFFu); fq = (long long)(e >> 32);
                    }
                }
                long long w = 0;  // first position where parabola u is the lowest
                if (q >= 0) w = 1 + ((long long)u * u - (long long)sq * sq + fu - fq) / (2LL * (u - sq));
                if (w < len) {
                    ++q; sq = u; tq = (int)w; fq = fu;
                    st[(long long)q * stride] = edt_pack(u, (int)w, (int)fu);
                }
            }
        }
        // backward scan
        constexpr int PB = 4;
        unsigned long long pe[PB];
        int have = 0;  // entries q-1 .. q-have, fetched ahead (pe[0] is the next one to pop)
        for (int ub = nb - 1; ub >= 0; --ub) {  // the same batches, last row first
            const int u0 = min(len - 1, 8 * ub + 7), ulo = 8 * ub;
            if (sw[(long long)ub * XW] == 0u) {  // background under the whole warp: zeros; the envelope is popped when a foreground voxel needs it
                if (OUT != 0 && active) {
#pragma unroll
                    for (int k = 0; k < PF; ++k) {
                        if (u0 - k < ulo) break;
                        if (OUT == 1) ((double *)outv)[base + (long long)(u0 - k) * stride] = 0.0;
                        else ((int *)outv)[base + (long long)(u0 - k) * stride] = 0;
                    }
                }
                continue;
            }
            uint32_t wd[PF];
#pragma unroll
            for (int k = 0; k < PF; ++k) wd[k] = u0 - k >= ulo ? bw[(long long)(u0 - k) * bit_stride] : 0u;
            bool bit[PF];
#pragma unroll
            for (int k = 0; k < PF; ++k) bit[k] = active && ((wd[k] >> lane) & 1u);
#pragma unroll
            for (int k = 0; k < PF; ++k) {
                const int u = u0 - k;
                if (u < ulo) break;
                while (q > 0 && u < tq) {  // the top parabola reigns from tq on: below it the previous one does
                    if (have == 0) {
#pragma unroll
                        for (int j = 0; j < PB; ++j) pe[j] = st[(long long)max(q - 1 - j, 0) * stride];
                        have = min(PB, q);
                    }
                    --q; --have;
                    sq = (int)(pe[0] & 0xFFFFu); tq = (int)((pe[0] >> 16) & 0xFFFFu); fq = (long long)(pe[0] >> 32);
#pragma unroll
                    for (int j = 0; j + 1 < PB; ++j) pe[j] = pe[j + 1];
                }
                long long d = 0;
                if (bit[k]) {
                    d = q >= 0 ? (long long)(u - sq) * (u - sq) + fq : (long long)EDT_INF;
                    if (d >= EDT_INF) { d = EDT_INF; inf = true; }
                }
                if (OUT == 0) { if (bit[k]) ((int *)outv)[base + (long long)u * stride] = (int)d; }
                else if (OUT == 1) { if (active) ((double *)outv)[base + (long long)u * stride] = sqrt((double)d); }
                else { if (active) ((int *)outv)[base + (long long)u * stride] = (int)d; }
            }
        }
    }
    if (OUT == 1 && inf) *flag = 1;
}

int edt_check(const int64_t *shape) {
    if (!shape || shape[0] <= 0 || shape[1] <= 0 || shape[2] <= 0) return VRG_ERR_ARG;
    if (shape[0] > 16384 || shape[1] > 16384 || shape[2] > 16384) return VRG_ERR_ARG;
    return VRG_OK;
}

// The three passes.  out_mode 1: Euclidean distance, float64, into `out` (*flag raised when the mask has no zero voxel);
// out_mode 2: squared distance, int32.  Scratch: uint16 x-distances, int32 y-pass result, the packed bit volume and the
// 8-byte envelope stack slots (14.1 bytes per voxel).  Asynchronous on `stream`.
int edt_passes(const uint8_t *d_mask, const int64_t *shape, void *out, int out_mode, int *flag, cudaStream_t stream) {
    const long long Z = shape[0], Y = shape[1], X = shape[2], n = Z * Y * X;
    const int XW = (int)((X + 31) / 32);
    Buf d1, a, st, bits, sum;
    const long long nby = (Y + 7) / 8, nbz = (Z + 7) / 8;
    cudaError_t e = d1.alloc(n * sizeof(uint16_t), stream);
    if (e == cudaSuccess) e = a.alloc(n * sizeof(int), stream);
    if (e == cudaSuccess) e = st.alloc(n * sizeof(unsigned long long), stream);
    if (e == cudaSuccess) e = bits.alloc((size_t)Z * Y * XW * sizeof(uint32_t), stream);
    if (e == cudaSuccess) e = sum.alloc((size_t)std::max(Z * nby, nbz * Y) * XW * sizeof(uint32_t), stream);
    if (e == cudaSuccess) {
        const int grid = 148 * 8;
        const long long per_block = 128;
        const int gy = (int)std::min<long long>((Z * XW * 32 + per_block - 1) / per_block, 148 * 16);
        const int gz = (int)std::min<long long>((Y * XW * 32 + per_block - 1) / per_block, 148 * 16);
        k_edt_rows<<<grid, 256, (size_t)8 * 3 * XW * sizeof(uint32_t), stream>>>(d_mask, d1.as<uint16_t>(), bits.as<uint32_t>(), Z * Y, (int)X, XW);
        k_edt_summary<<<grid, 256, 0, stream>>>(bits.as<uint32_t>(), sum.as<uint32_t>(), Z, (int)Y, XW, Y * XW, XW);
        k_edt_lines<uint16_t, 0><<<gy, 128, 0, stream>>>(d1.as<uint16_t>(), a.p, bits.as<uint32_t>(), st.as<unsigned long long>(), Z, (int)Y, X,
                                                          (int)X, XW, X * Y, Y * XW, XW, sum.as<uint32_t>(), nullptr);
        k_edt_summary<<<grid, 256, 0, stream>>>(bits.as<uint32_t>(), sum.as<uint32_t>(), Y, (int)Z, XW, XW, (long long)Y * XW);
        if (out_mode == 1)
            k_edt_lines<int, 1><<<gz, 128, 0, stream>>>(a.as<int>(), out, bits.as<uint32_t>(), st.as<unsigned long long>(), Y, (int)Z, X * Y,
                                                         (int)X, XW, X, XW, (long long)Y * XW, sum.as<uint32_t>(), flag);
        else
            k_edt_lines<int, 2><<<gz, 128, 0, stream>>>(a.as<int>(), out, bits.as<uint32_t>(), st.as<unsigned long long>(), Y, (int)Z, X * Y,
                                                         (int)X, XW, X, XW, (long long)Y * XW, sum.as<uint32_t>(), flag);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    return VRG_OK;
}

int edt_squared_device(const uint8_t *d_mask, const int64_t *shape, int *sq_out, cudaStream_t stream) {
    return edt_passes(d_mask, shape, sq_out, 2, nullptr, stream);
}

int edt_device(const uint8_t *d_mask, const int64_t *shape, double *d_out, cudaStream_t stream) {
    Buf flag;
    cudaError_t e = flag.alloc(sizeof(int), stream);
    int rc = VRG_OK;
    if (e == cudaSuccess) {
        cudaMemsetAsync(flag.p, 0, sizeof(int), stream);
        rc = edt_passes(d_mask, shape, d_out, 1, flag.as<int>(), stream);
        if (rc == VRG_OK) {
            int h_flag = 0;
            e = cudaMemcpyAsync(&h_flag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e == cudaSuccess && h_flag) {  // no zero voxel anywhere: the transform is undefined
                vrg_set_error_internal("distance transform: the mask has no zero voxel");
                rc = VRG_ERR_ARG;
            }
        }
    }
    if (e != cudaSuccess) {
        vrg_set_error_internal(cudaGetErrorString(e));
        rc = e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    }
    return rc;
}

int bad_args(const char *what) {
    vrg_set_error_internal(what);
    return VRG_ERR_ARG;
}

// ---- Feature transform: scipy.ndimage.distance_transform_edt(mask, sampling=..., return_indices=...) ----
// SciPy computes the feature transform (the nearest zero voxel of every voxel) with Maurer's algorithm, one line at a
// time, axis 0 (z) first, then y, then x, and the distances afterwards from the features in NumPy.  Which of two equally
// near zero voxels a voxel gets is decided by the order of the passes, by the tie rule of the query (the earlier site
// keeps a tie) and, with sampling, by the rounding of every fp64 step.  The passes below therefore restate SciPy's loop
// decision for decision: a site is a voxel that has a feature, the build pops with SciPy's test, the query walks the
// stack with SciPy's comparison, and every fp64 operation is a separately rounded __dmul_rn / __dadd_rn / __dsub_rn in
// SciPy's order of evaluation (nvcc would contract a*b - c into an FMA and change decisions).  Unit spacing is spacing
// 1.0: multiplying by 1.0 is exact, so the decisions are those of SciPy's path without sampling.
// Features travel packed: after pass z a voxel's feature differs from the voxel only in z (uint16), after pass y only in
// z and y (uint32, z | y << 16).  FT_NONE in the z field: no feature yet (a line without a zero voxel so far).
constexpr uint32_t FT_NONE = 0xFFFFu;

__device__ __forceinline__ double ft_t(int f, int c, double s) { return __dmul_rn((double)(f - c), s); }  // SciPy's t, sampled
__device__ __forceinline__ double ft_sq(double t) { return __dmul_rn(t, t); }

// SciPy's pop test for the two top sites u, v of the stack and the new site w along the pass axis (positions pu, pv, pw;
// uR, vR, wR = their squared distances over the other axes): c*vR - b*uR - a*wR - a*b*c > 0, left to right
__device__ __forceinline__ bool ft_pop(int pu, int pv, int pw, double uR, double vR, double wR, double s) {
    const double a = ft_t(pv, pu, s), b = ft_t(pw, pv, s), c = __dadd_rn(a, b);
    const double e = __dsub_rn(__dsub_rn(__dsub_rn(__dmul_rn(c, vR), __dmul_rn(b, uR)), __dmul_rn(a, wR)), __dmul_rn(__dmul_rn(a, b), c));
    return !(e <= 0.0);
}

// pass z: the sites of a line are its zero voxels.  With no other axis yet uR = vR = wR = 0, SciPy's test reads
// -a*b*c <= 0 and never pops, so the stack is every zero voxel of the line in order; the query walks it with SciPy's
// comparison (advance while strictly nearer), finding the next site by scanning the mask ahead.  One thread per (y, x)
// line, neighbouring lanes on neighbouring x.
__global__ void __launch_bounds__(256) k_ft_z(const uint8_t *__restrict__ mask, uint16_t *__restrict__ fz, long long nlines, int Z,
                                              double s0) {
    for (long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x; line < nlines; line += (long long)gridDim.x * blockDim.x) {
        const uint8_t *m = mask + line;
        uint16_t *o = fz + line;
        int cur = 0;
        while (cur < Z && m[(long long)cur * nlines] != 0) ++cur;
        if (cur == Z) {
            for (int i = 0; i < Z; ++i) o[(long long)i * nlines] = (uint16_t)FT_NONE;
            continue;
        }
        int nxt = cur + 1;
        while (nxt < Z && m[(long long)nxt * nlines] != 0) ++nxt;
        for (int i = 0; i < Z; ++i) {
            double d1 = ft_sq(ft_t(cur, i, s0));
            while (nxt < Z) {
                const double d2 = ft_sq(ft_t(nxt, i, s0));
                if (d1 <= d2) break;
                d1 = d2;
                cur = nxt++;
                while (nxt < Z && m[(long long)nxt * nlines] != 0) ++nxt;
            }
            o[(long long)i * nlines] = (uint16_t)cur;
        }
    }
}

// pass y: one thread per (z, x) line, lanes on neighbouring x.  A site carries (its feature's z, y).  The stack lives in
// scratch laid out like the volume (entry q of line (z, x) at (z, q, x): lanes at the same depth touch one row segment);
// the two top entries and their squared z-distances stay in registers.  Inputs are fetched eight steps ahead, stack
// entries of the query four at a time.
__global__ void __launch_bounds__(128) k_ft_y(const uint16_t *__restrict__ fz, uint32_t *__restrict__ fy, uint32_t *__restrict__ stack,
                                              int Z, int Y, int X, double s0, double s1) {
    const long long nlines = (long long)Z * X;
    for (long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x; line < nlines; line += (long long)gridDim.x * blockDim.x) {
        const int z = (int)(line / X), x = (int)(line % X);
        const long long base = (long long)z * Y * X + x;
        const uint16_t *in = fz + base;
        uint32_t *st = stack + base, *out = fy + base;
        int q = -1;  // depth - 1
        int uy = 0, uz = 0, vy = 0, vz = 0;
        double uR = 0.0, vR = 0.0;
        constexpr int PF = 8;
        for (int i0 = 0; i0 < Y; i0 += PF) {
            uint16_t pre[PF];
#pragma unroll
            for (int k = 0; k < PF; ++k) pre[k] = i0 + k < Y ? in[(long long)(i0 + k) * X] : (uint16_t)FT_NONE;
#pragma unroll
            for (int k = 0; k < PF; ++k) {
                const int f0 = pre[k], i = i0 + k;
                if (f0 == (int)FT_NONE) continue;  // also every step beyond the line's end
                const double wR = ft_sq(ft_t(f0, z, s0));
                while (q >= 1 && ft_pop(uy, vy, i, uR, vR, wR, s1)) {
                    --q;
                    vy = uy; vz = uz; vR = uR;
                    if (q >= 1) {
                        const uint32_t e = st[(long long)(q - 1) * X];
                        uy = (int)(e & 0xFFFFu); uz = (int)(e >> 16); uR = ft_sq(ft_t(uz, z, s0));
                    }
                }
                ++q;
                st[(long long)q * X] = (uint32_t)i | ((uint32_t)f0 << 16);
                uy = vy; uz = vz; uR = vR;
                vy = i; vz = f0; vR = wR;
            }
        }
        if (q < 0) {  // no site on this line: SciPy leaves it without features
            for (int i = 0; i < Y; ++i) out[(long long)i * X] = FT_NONE;
            continue;
        }
        const int maxl = q;
        constexpr int PB = 4;
        uint32_t pe[PB];  // entries l+1 .. l+have
        int have = 0, l = 0;
        int cy = (int)(st[0] & 0xFFFFu), cz = (int)(st[0] >> 16);
        double cR = ft_sq(ft_t(cz, z, s0));
        for (int i = 0; i < Y; ++i) {
            double d1 = __dadd_rn(cR, ft_sq(ft_t(cy, i, s1)));
            while (l < maxl) {
                if (have == 0) {
#pragma unroll
                    for (int j = 0; j < PB; ++j) pe[j] = st[(long long)min(l + 1 + j, maxl) * X];
                    have = min(PB, maxl - l);
                }
                const int ny = (int)(pe[0] & 0xFFFFu), nz = (int)(pe[0] >> 16);
                const double nR = ft_sq(ft_t(nz, z, s0));
                const double d2 = __dadd_rn(nR, ft_sq(ft_t(ny, i, s1)));
                if (d1 <= d2) break;
                d1 = d2; ++l; --have;
                cy = ny; cz = nz; cR = nR;
#pragma unroll
                for (int j = 0; j + 1 < PB; ++j) pe[j] = pe[j + 1];
            }
            out[(long long)i * X] = (uint32_t)cz | ((uint32_t)cy << 16);
        }
    }
}

// pass x, the last pass: the lines are the contiguous rows.  One warp owns 32 consecutive rows, one lane per row; the
// rows pass through shared memory in tiles of 32 x 32 voxels, so every global access is a coalesced row segment while
// each lane walks its own row.  Build: tiles of pass-y features in, pushes onto the lane's stack (scratch, entry q of
// lane at [q][lane] of the warp's region: x | z << 16 | y << 32).  Query: features of a tile out to shared memory, then
// written row by row as SciPy's outputs: int32 indices[3][Z][Y][X] when `idx` is set, and when `dist` is set the float64
// distance in NumPy's order, sqrt(((dz*s0)^2 + (dy*s1)^2) + (dx*s2)^2).  A row without any site means the mask has no
// zero voxel: *flag is raised.
constexpr int FT_WARPS = 4;
__global__ void __launch_bounds__(32 * FT_WARPS) k_ft_x(const uint32_t *__restrict__ fy, unsigned long long *__restrict__ stack,
                                                        int32_t *__restrict__ idx, double *__restrict__ dist, long long nrows, int Y,
                                                        int X, double s0, double s1, double s2, int *flag) {
    __shared__ unsigned long long tile[FT_WARPS][32 * 33];  // +1 column: lane r at row r of the tile hits its own bank
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned long long *to = tile[wib];
    uint32_t *ti = (uint32_t *)to;
    const long long n = nrows * X, nw = (nrows + 31) / 32;
    for (long long w = (long long)blockIdx.x * FT_WARPS + wib; w < nw; w += (long long)gridDim.x * FT_WARPS) {
        const long long r0 = w * 32, row = r0 + lane;
        const bool active = row < nrows;
        const int z = active ? (int)(row / Y) : 0, y = active ? (int)(row % Y) : 0;
        const int nr = (int)min(32LL, nrows - r0);
        unsigned long long *st = stack + r0 * X + lane;
        int q = -1;
        int ux = 0, vx = 0;
        double uR = 0.0, vR = 0.0;
        for (int c0 = 0; c0 < X; c0 += 32) {
            const int nc = min(32, X - c0);
            __syncwarp();
            if (lane < nc)
                for (int r = 0; r < nr; ++r) ti[r * 33 + lane] = fy[(r0 + r) * X + c0 + lane];
            __syncwarp();
            if (!active) continue;
            for (int k = 0; k < nc; ++k) {
                const uint32_t f = ti[lane * 33 + k];
                const int f0 = (int)(f & 0xFFFFu), f1 = (int)(f >> 16), i = c0 + k;
                if (f0 == (int)FT_NONE) continue;
                const double wR = __dadd_rn(ft_sq(ft_t(f0, z, s0)), ft_sq(ft_t(f1, y, s1)));
                while (q >= 1 && ft_pop(ux, vx, i, uR, vR, wR, s2)) {
                    --q;
                    vx = ux; vR = uR;
                    if (q >= 1) {
                        const unsigned long long e = st[(long long)(q - 1) * 32];
                        ux = (int)(e & 0xFFFFu);
                        uR = __dadd_rn(ft_sq(ft_t((int)((e >> 16) & 0xFFFFu), z, s0)), ft_sq(ft_t((int)(e >> 32), y, s1)));
                    }
                }
                ++q;
                st[(long long)q * 32] = (unsigned long long)i | ((unsigned long long)f0 << 16) | ((unsigned long long)f1 << 32);
                ux = vx; uR = vR;
                vx = i; vR = wR;
            }
        }
        const unsigned rows_ok = __ballot_sync(FULLMASK, active && q >= 0);
        if (active && q < 0) *flag = 1;
        const int maxl = q;
        constexpr int PB = 4;
        unsigned long long pe[PB], cur = 0ull;
        int have = 0, l = 0;
        double cR = 0.0;
        if (maxl >= 0) {
            cur = st[0];
            cR = __dadd_rn(ft_sq(ft_t((int)((cur >> 16) & 0xFFFFu), z, s0)), ft_sq(ft_t((int)(cur >> 32), y, s1)));
        }
        for (int c0 = 0; c0 < X; c0 += 32) {
            const int nc = min(32, X - c0);
            __syncwarp();
            if (maxl >= 0) {
                for (int k = 0; k < nc; ++k) {
                    const int i = c0 + k;
                    double d1 = __dadd_rn(cR, ft_sq(ft_t((int)(cur & 0xFFFFu), i, s2)));
                    while (l < maxl) {
                        if (have == 0) {
#pragma unroll
                            for (int j = 0; j < PB; ++j) pe[j] = st[(long long)min(l + 1 + j, maxl) * 32];
                            have = min(PB, maxl - l);
                        }
                        const double nR = __dadd_rn(ft_sq(ft_t((int)((pe[0] >> 16) & 0xFFFFu), z, s0)), ft_sq(ft_t((int)(pe[0] >> 32), y, s1)));
                        const double d2 = __dadd_rn(nR, ft_sq(ft_t((int)(pe[0] & 0xFFFFu), i, s2)));
                        if (d1 <= d2) break;
                        d1 = d2; ++l; --have;
                        cur = pe[0]; cR = nR;
#pragma unroll
                        for (int j = 0; j + 1 < PB; ++j) pe[j] = pe[j + 1];
                    }
                    to[lane * 33 + k] = cur;
                }
            }
            __syncwarp();
            if (lane >= nc) continue;
            const int x = c0 + lane;
            for (int r = 0; r < nr; ++r) {
                if (!((rows_ok >> r) & 1u)) continue;
                const unsigned long long e = to[r * 33 + lane];
                const int fx = (int)(e & 0xFFFFu), fzv = (int)((e >> 16) & 0xFFFFu), fyv = (int)(e >> 32);
                const long long p = (r0 + r) * X + x;
                if (idx) { idx[p] = fzv; idx[n + p] = fyv; idx[2 * n + p] = fx; }
                if (dist) {
                    const long long rr = r0 + r;
                    const double tz = ft_t(fzv, (int)(rr / Y), s0), ty = ft_t(fyv, (int)(rr % Y), s1), tx = ft_t(fx, x, s2);
                    dist[p] = __dsqrt_rn(__dadd_rn(__dadd_rn(ft_sq(tz), ft_sq(ty)), ft_sq(tx)));
                }
            }
        }
    }
}

// The three feature-transform passes.  Scratch: uint16 pass-z features, uint32 pass-y features, 8-byte stack slots
// (shared by the y and x passes): 14 bytes per voxel.  *flag raised when the mask has no zero voxel.  Asynchronous.
int ft_passes(const uint8_t *d_mask, const int64_t *shape, const double *s, double *dist, int32_t *idx, int *flag, cudaStream_t stream) {
    const long long Z = shape[0], Y = shape[1], X = shape[2], n = Z * Y * X, nrows = Z * Y;
    Buf fz, fy, st;
    cudaError_t e = fz.alloc(n * sizeof(uint16_t), stream);
    if (e == cudaSuccess) e = fy.alloc(n * sizeof(uint32_t), stream);
    if (e == cudaSuccess) e = st.alloc((size_t)((nrows + 31) / 32) * 32 * X * sizeof(unsigned long long), stream);
    if (e == cudaSuccess) {
        const int gz = (int)std::min<long long>((Y * X + 255) / 256, 148 * 16);
        const int gy = (int)std::min<long long>((Z * X + 127) / 128, 148 * 16);
        const int gx = (int)std::min<long long>(((nrows + 31) / 32 + FT_WARPS - 1) / FT_WARPS, 148 * 16);
        k_ft_z<<<gz, 256, 0, stream>>>(d_mask, fz.as<uint16_t>(), Y * X, (int)Z, s[0]);
        k_ft_y<<<gy, 128, 0, stream>>>(fz.as<uint16_t>(), fy.as<uint32_t>(), st.as<uint32_t>(), (int)Z, (int)Y, (int)X, s[0], s[1]);
        k_ft_x<<<gx, 32 * FT_WARPS, 0, stream>>>(fy.as<uint32_t>(), st.as<unsigned long long>(), idx, dist, nrows, (int)Y, (int)X,
                                                 s[0], s[1], s[2], flag);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        vrg_set_error_internal(cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    }
    return VRG_OK;
}

int ft_device(const uint8_t *d_mask, const int64_t *shape, const double *s, double *dist, int32_t *idx, cudaStream_t stream) {
    Buf flag;
    cudaError_t e = flag.alloc(sizeof(int), stream);
    int rc = VRG_OK;
    if (e == cudaSuccess) e = cudaMemsetAsync(flag.p, 0, sizeof(int), stream);
    if (e == cudaSuccess) {
        rc = ft_passes(d_mask, shape, s, dist, idx, flag.as<int>(), stream);
        if (rc == VRG_OK) {
            int h_flag = 0;
            e = cudaMemcpyAsync(&h_flag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e == cudaSuccess && h_flag) {
                vrg_set_error_internal("distance transform: the mask has no zero voxel");
                rc = VRG_ERR_ARG;
            }
        }
    }
    if (e != cudaSuccess) {
        vrg_set_error_internal(cudaGetErrorString(e));
        rc = e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    }
    return rc;
}

// checks the arguments of both feature-transform entry points and fills s with the spacings (1.0 without sampling)
int ft_check(const uint8_t *mask, const int64_t *shape, const double *sampling, const double *dist, const int32_t *idx, double *s) {
    if (!mask || edt_check(shape) != VRG_OK) return bad_args("feature transform: null mask or bad shape (axes 1..16384)");
    if (!dist && !idx) return bad_args("feature transform: at least one of dist / indices must be requested");
    for (int d = 0; d < 3; ++d) {
        s[d] = sampling ? sampling[d] : 1.0;
        if (!(s[d] > 0.0) || !std::isfinite(s[d])) return bad_args("feature transform: sampling must be positive and finite");
    }
    return VRG_OK;
}

}  // namespace

// shared with vrg_mask.cu: the x pass alone -- uint16 distance to the nearest zero voxel of the same row at every FOREGROUND
// voxel (0xFFFF: none in this row) and the packed foreground bits, [Z*Y][ceil(X/32)] words
int vrg_edt_rows_device_internal(const uint8_t *d_mask, const int64_t *shape, uint16_t *d1, uint32_t *bits, cudaStream_t stream) {
    const long long Z = shape[0], Y = shape[1], X = shape[2];
    const int XW = (int)((X + 31) / 32);
    k_edt_rows<<<148 * 8, 256, (size_t)8 * 3 * XW * sizeof(uint32_t), stream>>>(d_mask, d1, bits, Z * Y, (int)X, XW);
    return cudaGetLastError() == cudaSuccess ? VRG_OK : VRG_ERR_CUDA;
}

// shared with vrg_mask.cu: squared EDT of a device mask into a device int32 volume
int vrg_edt_squared_device_internal(const uint8_t *d_mask, const int64_t *shape, int *sq_out, cudaStream_t stream) {
    return edt_squared_device(d_mask, shape, sq_out, stream);
}

// mask / dist live on the device
extern "C" int vrg_edt_device(int device, const uint8_t *mask_dev, const int64_t *shape, double *dist_dev, void *cuda_stream) {
    if (!mask_dev || !dist_dev || edt_check(shape) != VRG_OK) return bad_args("distance transform: null buffer or bad shape (axes 1..16384)");
    if (cudaSetDevice(device) != cudaSuccess) return VRG_ERR_CUDA;
    vrg_scratch::pool_setup(device);
    return edt_device(mask_dev, shape, dist_dev, (cudaStream_t)cuda_stream);
}

// host buffers: mask uint8 (non-zero = foreground), dist float64, both (Z, Y, X) C order
extern "C" int vrg_edt(int device, const uint8_t *mask_host, const int64_t *shape, double *dist_host) {
    if (!mask_host || !dist_host || edt_check(shape) != VRG_OK) return bad_args("distance transform: null buffer or bad shape (axes 1..16384)");
    if (cudaSetDevice(device) != cudaSuccess) return VRG_ERR_CUDA;
    vrg_scratch::pool_setup(device);
    const size_t n = (size_t)shape[0] * shape[1] * shape[2];
    Buf d_mask, d_out;
    cudaError_t e = d_mask.alloc(n, nullptr);
    if (e == cudaSuccess) e = d_out.alloc(n * sizeof(double), nullptr);
    int rc = VRG_OK;
    if (e == cudaSuccess) e = cudaMemcpy(d_mask.p, mask_host, n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = edt_device(d_mask.as<uint8_t>(), shape, d_out.as<double>(), nullptr);
        if (rc == VRG_OK) e = cudaMemcpy(dist_host, d_out.p, n * sizeof(double), cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) {
        vrg_set_error_internal(cudaGetErrorString(e));
        rc = e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    }
    return rc;
}

// mask / dist / indices live on the device; sampling (3 doubles or NULL) on the host
extern "C" int vrg_edt_ft_device(int device, const uint8_t *mask_dev, const int64_t *shape, const double *sampling, double *dist_dev,
                                 int32_t *indices_dev, void *cuda_stream) {
    double s[3];
    const int rc = ft_check(mask_dev, shape, sampling, dist_dev, indices_dev, s);
    if (rc != VRG_OK) return rc;
    if (cudaSetDevice(device) != cudaSuccess) return VRG_ERR_CUDA;
    vrg_scratch::pool_setup(device);
    return ft_device(mask_dev, shape, s, dist_dev, indices_dev, (cudaStream_t)cuda_stream);
}

// host buffers: mask uint8 (Z, Y, X), dist float64 (Z, Y, X), indices int32 (3, Z, Y, X), all C order
extern "C" int vrg_edt_ft(int device, const uint8_t *mask_host, const int64_t *shape, const double *sampling, double *dist_host,
                          int32_t *indices_host) {
    double s[3];
    int rc = ft_check(mask_host, shape, sampling, dist_host, indices_host, s);
    if (rc != VRG_OK) return rc;
    if (cudaSetDevice(device) != cudaSuccess) return VRG_ERR_CUDA;
    vrg_scratch::pool_setup(device);
    const size_t n = (size_t)shape[0] * shape[1] * shape[2];
    Buf d_mask, d_dist, d_idx;
    cudaError_t e = d_mask.alloc(n, nullptr);
    if (e == cudaSuccess && dist_host) e = d_dist.alloc(n * sizeof(double), nullptr);
    if (e == cudaSuccess && indices_host) e = d_idx.alloc(3 * n * sizeof(int32_t), nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(d_mask.p, mask_host, n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = ft_device(d_mask.as<uint8_t>(), shape, s, d_dist.as<double>(), d_idx.as<int32_t>(), nullptr);
        if (rc == VRG_OK && dist_host) e = cudaMemcpy(dist_host, d_dist.p, n * sizeof(double), cudaMemcpyDeviceToHost);
        if (rc == VRG_OK && e == cudaSuccess && indices_host) e = cudaMemcpy(indices_host, d_idx.p, 3 * n * sizeof(int32_t), cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) {
        vrg_set_error_internal(cudaGetErrorString(e));
        rc = e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA;
    }
    return rc;
}

// hands the cached scratch blocks of the handle-less entry points (EDT, labelling, vessel mask) back to the driver
extern "C" int vrg_release_scratch(int device) {
    if (cudaSetDevice(device) != cudaSuccess) return VRG_ERR_CUDA;
    cudaDeviceSynchronize();
    vrg_scratch::pool_trim(device);
    return VRG_OK;
}
