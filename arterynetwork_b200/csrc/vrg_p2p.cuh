// Multi-GPU exchange over NVLink peer memory (one process per GPU, buffers shared through CUDA IPC).
//
// The z-slab protocol has exactly two exchanges per iteration (DESIGN.md section 7):
//   halo  -- the 2 boundary planes of the executed-flip plane F (and of C, E when the input has label 4) go to each
//            neighbour slab;
//   stats -- a SUM all-reduce of the int64 statistics vector (region histograms + counters).
// Both are done by kernels of THIS library on the run's own stream: the producer stores straight into the peer's
// receive buffer / mailbox over NVLink, fences system-wide, and raises a sequence-numbered flag in the peer's memory;
// the consumer spins on its own flag (acquire) and unpacks.  No host round trip, no NCCL call in the loop, so the host
// enqueues a whole batch of iterations at once exactly as on one GPU.  Sequence numbers come from device state
// (run epoch << 32 | sweep + 1), identical on every rank, and only grow, so flags never need a reset.
//
// Hazards (who may run ahead of whom) are argued in DESIGN.md section 7; in short a rank can be at most one statistics
// exchange ahead of any other, hence the mailbox is double-buffered by sequence parity, and halo data goes through a
// receive buffer because the receiver's own sweep writes (raw) flip words into the same halo planes.
#pragma once
#include "vrg_kernels.cuh"

namespace vrg {

constexpr int P2P_MAX_WORLD = 8;
constexpr int P2P_KINDS = 3;  // F, C, E
enum { PK_F = 0, PK_C = 1, PK_E = 2 };
constexpr long long EXIT_PEER_TIMEOUT = 99;
constexpr long long P2P_SPIN_LIMIT = 40000000000ll;          // ~20 s of SM clocks: a dead peer must not hang the box

// flag words of one rank's mailbox (unsigned long long each)
//   [0 .. 2*P2P_KINDS)                      halo flags: kind * 2 + side (0 = from the lower neighbour, 1 = from the upper)
//   [HALO_FLAGS .. +2*world)                stats flags: parity * world + source rank
//   [DONE_BASE .. +4)                       block-completion counters of this rank's own push kernels (local use)
constexpr int HALO_FLAGS = 2 * P2P_KINDS;
constexpr int STATS_FLAGS = HALO_FLAGS;
constexpr int DONE_BASE = STATS_FLAGS + 2 * P2P_MAX_WORLD;
constexpr int FLAG_WORDS = DONE_BASE + 8;

struct P2P {
    int rank, world;
    int slot_words;                                  // int64 words per statistics slot (capacity, >= 2L + ST_EXTRA)
    unsigned long long *flags;                       // my flag words
    long long *slots;                                // my mailbox: [2 parities][world][slot_words]
    uint32_t *recv;                                  // my halo receive buffer: [2 parities][P2P_KINDS][2 sides][HALO][plane_words]
                                                     // uint32, then [2 parities][2 sides][HALO][plane_words] tagged 8-byte slots
    unsigned long long *peer_flags[P2P_MAX_WORLD];   // every rank's flag words (mine included)
    long long *peer_slots[P2P_MAX_WORLD];
    uint32_t *peer_recv[2];                          // lower / upper neighbour's receive buffer (nullptr at the ends)
};

__device__ __forceinline__ unsigned long long p2p_seq(const Params &p) {
    return ((unsigned long long)p.ctrl[C_EPOCH] << 32) | (unsigned long long)(p.ctrl[C_SWEEPS] + 1);
}
__device__ __forceinline__ void st_release_sys(unsigned long long *addr, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *addr) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long *addr, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long *addr) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(addr) : "memory");
    return v;
}
// the receive buffer's second part: tagged 8-byte slots [2 parities][2 sides][n] of the pipelined run's halo exchange
// (n = HALO * plane_words); it starts behind the [2][P2P_KINDS][2][n] uint32 words of the flag-based exchange
__device__ __forceinline__ unsigned long long *p2p_ll_region(uint32_t *recv, long long n) {
    return (unsigned long long *)(recv + 2 * P2P_KINDS * 2 * n);
}
// spin until *flag >= seq; false on timeout (the caller raises the peer-timeout exit)
__device__ __forceinline__ bool p2p_wait(const unsigned long long *flag, unsigned long long seq) {
    const long long t0 = clock64();
    while (ld_acquire_sys(flag) < seq) {
        if (clock64() - t0 > P2P_SPIN_LIMIT) return false;
        __nanosleep(64);
    }
    return true;
}
// the last block of a push kernel to finish raises the flags (all data of all blocks is then fenced)
__device__ __forceinline__ bool p2p_last_block(unsigned long long *counter) {
    __shared__ bool last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long done = atomicAdd(counter, 1ull) + 1ull;
        last = done == gridDim.x;
        if (last) *counter = 0ull;
    }
    __syncthreads();
    return last;
}

// ---- halo --------------------------------------------------------------------------------------------------------
// kinds: bit mask over PK_*.  `running_only`: loop exchanges obey the run status; the one after init does not.
// Loop exchanges take their sequence number and their go / no-go from the snapshot k_cancel left in the control block
// (C_HALO_SEQ, C_HALO_GO), which holds the iteration k_cancel applied until the next k_cancel; C_SWEEPS / C_STATUS move on
// with the statistics exchange's bookkeeping.  The receive buffer is double-buffered by sequence parity, because a
// neighbour that is one iteration ahead may push its next planes while this rank still unpacks the current ones.
__device__ __forceinline__ bool p2p_halo_seq(const Params &p, int seq_zero, unsigned long long &seq) {
    if (seq_zero) { seq = (unsigned long long)p.ctrl[C_EPOCH] << 32; return true; }
    seq = (unsigned long long)p.ctrl[C_HALO_SEQ];
    return p.ctrl[C_HALO_GO] != 0;
}

__global__ void __launch_bounds__(BLOCK) k_p2p_push_halo(Params p, P2P q, int kinds, int seq_zero) {
    unsigned long long seq;
    if (!p2p_halo_seq(p, seq_zero, seq)) return;
    const long long n = (long long)HALO * p.plane_words;
    const long long par_off = (long long)(seq & 1ull) * P2P_KINDS * 2 * n;
    const long long tid = (long long)blockIdx.x * BLOCK + threadIdx.x, nth = (long long)gridDim.x * BLOCK;
    for (int kind = 0; kind < P2P_KINDS; ++kind) {
        if (!(kinds & (1 << kind))) continue;
        const uint32_t *plane = kind == PK_F ? p.F : kind == PK_C ? p.C : p.E;
        if (plane == nullptr) continue;
        for (int side = 0; side < 2; ++side) {  // side 0: to the lower neighbour, side 1: to the upper
            uint32_t *dst = q.peer_recv[side];
            if (dst == nullptr) continue;
            // my first own planes land in the lower neighbour's "from above" region (its side 1) and vice versa
            dst += par_off + ((long long)kind * 2 + (side ^ 1)) * n;
            const uint32_t *src = plane + (long long)(side == 0 ? p.own_lo : p.own_hi - HALO) * p.plane_words;
            for (long long i = tid; i < n; i += nth) dst[i] = src[i];
        }
    }
    if (p2p_last_block(q.flags + DONE_BASE + 0) && threadIdx.x == 0) {
        for (int kind = 0; kind < P2P_KINDS; ++kind) {
            if (!(kinds & (1 << kind))) continue;
            if (q.peer_recv[0]) st_release_sys(q.peer_flags[q.rank - 1] + kind * 2 + 1, seq);
            if (q.peer_recv[1]) st_release_sys(q.peer_flags[q.rank + 1] + kind * 2 + 0, seq);
        }
    }
}

// `flip`: the unpacked executed-flip words are applied to the halo copy of the segmented plane in the same pass
// (what k_flip_halo does on the collective path).
__global__ void __launch_bounds__(BLOCK) k_p2p_wait_unpack_halo(Params p, P2P q, int kinds, int seq_zero, int flip) {
    unsigned long long seq;
    if (!p2p_halo_seq(p, seq_zero, seq)) return;
    __shared__ int ok;
    if (threadIdx.x == 0) {
        ok = 1;
        for (int kind = 0; kind < P2P_KINDS && ok; ++kind) {
            if (!(kinds & (1 << kind))) continue;
            if (q.peer_recv[0] && !p2p_wait(q.flags + kind * 2 + 0, seq)) ok = 0;
            if (ok && q.peer_recv[1] && !p2p_wait(q.flags + kind * 2 + 1, seq)) ok = 0;
        }
        if (!ok) { p.ctrl[C_PEER_TIMEOUT] = 1; p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
        __threadfence_system();
    }
    __syncthreads();
    if (!ok) return;
    const long long n = (long long)HALO * p.plane_words;
    const long long par_off = (long long)(seq & 1ull) * P2P_KINDS * 2 * n;
    const long long tid = (long long)blockIdx.x * BLOCK + threadIdx.x, nth = (long long)gridDim.x * BLOCK;
    for (int kind = 0; kind < P2P_KINDS; ++kind) {
        if (!(kinds & (1 << kind))) continue;
        uint32_t *plane = kind == PK_F ? p.F : kind == PK_C ? p.C : p.E;
        if (plane == nullptr) continue;
        for (int side = 0; side < 2; ++side) {  // side 0: data from the lower neighbour -> my lower halo planes
            if (q.peer_recv[side] == nullptr) continue;
            const uint32_t *src = q.recv + par_off + ((long long)kind * 2 + side) * n;
            uint32_t *dst = plane + (long long)(side == 0 ? p.own_lo - HALO : p.own_hi) * p.plane_words;
            if (kind == PK_F && flip) {
                uint32_t *sdst = p.S + (long long)(side == 0 ? p.own_lo - HALO : p.own_hi) * p.plane_words;
                const int z0 = side == 0 ? p.own_lo - HALO : p.own_hi;
                for (long long i = tid; i < n; i += nth) {
                    const uint32_t f = __ldcg(src + i);
                    dst[i] = f;
                    if (f) {
                        sdst[i] ^= f;
                        const int zl = z0 + (int)(i / p.plane_words), y = (int)((i % p.plane_words) / p.WP), c = (int)(i % p.WP);
                        p.unitmap[unit_index(p, zl, y, c)] = 1;
                    }
                }
            } else {
                for (long long i = tid; i < n; i += nth) dst[i] = __ldcg(src + i);
            }
        }
    }
}

// ---- statistics all-reduce (+ the loop bookkeeping) -----------------------------------------------------------------
// One block: store my vector into every rank's mailbox, fence, raise the flags, wait for everybody's, sum the slots in
// rank order (integers: any order gives the same bits) into the global statistics and, in the loop, run the exit
// tests of k_advance right away -- the whole tail of an iteration is a single launch.
constexpr int STATS_BLOCK = 1024;
__device__ __forceinline__ void advance_state(const Params &p);  // defined with k_advance in vrg_kernels.cuh

// seq_zero: 0 = loop exchange (obeys the run status, ends with the loop bookkeeping); 1 = the exchange after init (sequence
// number 0 of the epoch); 2 = one more exchange after the exit, on every rank alike, which brings the counters that trail the
// loop's last exchange (k_quirks of the last applied update runs beside it) into the global statistics.
__global__ void __launch_bounds__(STATS_BLOCK) k_p2p_stats(Params p, P2P q, long long *gstats, int seq_zero) {
    if (!seq_zero && p.ctrl[C_STATUS] != RUNNING) return;
    const unsigned long long seq = seq_zero == 1 ? ((unsigned long long)p.ctrl[C_EPOCH] << 32) : p2p_seq(p);
    const int par = (int)(seq & 1ull), n = 2 * p.L + ST_EXTRA;
    for (int r = 0; r < q.world; ++r) {
        long long *dst = q.peer_slots[r] + ((long long)par * q.world + q.rank) * q.slot_words;
        for (int i = threadIdx.x; i < n; i += STATS_BLOCK) dst[i] = p.lstats[i];
    }
    __threadfence_system();
    __syncthreads();
    __shared__ int ok;
    if (threadIdx.x == 0) ok = 1;
    if (threadIdx.x < q.world) st_release_sys(q.peer_flags[threadIdx.x] + STATS_FLAGS + par * P2P_MAX_WORLD + q.rank, seq);
    __syncthreads();
    if (threadIdx.x < q.world && !p2p_wait(q.flags + STATS_FLAGS + par * P2P_MAX_WORLD + threadIdx.x, seq)) ok = 0;
    __threadfence_system();
    __syncthreads();
    if (!ok) {
        if (threadIdx.x == 0) { p.ctrl[C_PEER_TIMEOUT] = 1; if (seq_zero != 2) p.ctrl[C_STATUS] = EXIT_PEER_TIMEOUT; }
        return;
    }
    const long long *base = q.slots + (long long)par * q.world * q.slot_words;
    for (int i = threadIdx.x; i < n; i += STATS_BLOCK) {
        long long sum = 0;
        for (int r = 0; r < q.world; ++r) sum += __ldcg(base + (long long)r * q.slot_words + i);
        gstats[i] = sum;
    }
    if (seq_zero) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) advance_state(p);
}

}  // namespace vrg
