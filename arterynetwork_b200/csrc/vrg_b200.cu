// Host side of the C-ABI declared in include/vrg_b200.h (no torch types, no CPU fallback:
// every compute entry point launches the sm_100a kernels in vrg_kernels.cuh or fails).
#include "../../include/vrg_b200.h"
#include "vrg_kernels.cuh"
#include "vrg_p2p.cuh"
#include "vrg_tail.cuh"
#include "vrg_parzen.cuh"
#include "vrg_scratch.cuh"

#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace vrg;

static thread_local std::string g_err;
static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(e_ == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                   \
    } while (0)

struct vrg_handle {
    vrg_config cfg;
    Params p;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sms = 148;
    int64_t nz_own = 0, ext_lo = 0, ext_hi = 0;  // extended slab in global z
    size_t plane_bytes = 0;                      // one bit-plane buffer (all local planes)
    size_t rowflag_bytes = 0;
    double *d_data = nullptr;
    uint8_t *d_vm = nullptr, *d_rowflag = nullptr, *d_labels = nullptr, *d_unitmap = nullptr;
    size_t unitmap_bytes = 0;
    int *d_front = nullptr, *d_dirty = nullptr, *d_stamp = nullptr;
    uint16_t *d_index = nullptr;
    uint32_t *d_S = nullptr, *d_E = nullptr, *d_F = nullptr, *d_C = nullptr;
    uint32_t *d_Dc = nullptr;  // F64_DENSE: the decision bit-plane of the sweeps between refreshes (vrg_kernels.cuh, dense_refresh)
    double *d_levels = nullptr, *d_pin = nullptr, *d_pout = nullptr, *d_kmat = nullptr;
    uint32_t *d_dbits = nullptr;
    long long *d_lstats = nullptr, *d_gstats = nullptr, *d_ctrl = nullptr, *d_trace = nullptr;
    unsigned long long stage_seq = 0;       // chunks staged so far (buffer = parity)
    char *h_stage[2] = {nullptr, nullptr};  // pinned staging buffers of vrg_upload (pageable sources)
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    long long *h_ctrl = nullptr;  // pinned
    long long *h_poll = nullptr;  // pinned, 2 x C_WORDS: the control block as it stood behind the last two batches of vrg_run
    cudaEvent_t ev_poll[2] = {nullptr, nullptr};
    unsigned long long *d_hash = nullptr, *d_hkeys = nullptr;
    int *d_hcount = nullptr;
    std::vector<double> levels;  // distinct levels seen (sorted)
    int64_t n_distinct = 0;
    bool have_data = false, have_levels = false, inited = false, separate_gstats = false;
    int64_t launches = 0;
    int grid = 148 * 8;
    bool no_dcache = false;  // A/B switch VRG_NO_DCACHE: no decision bit-plane, every dense sweep reads the fp64 volume
    bool dense_attr_set = false, hist_attr_set = false, attached = false;
    const void *vm_base = nullptr;  // valueMap as indexed by local plane (own uint8 buffer, or attached in its own dtype)
    int vm_dtype = VRG_DTYPE_U8;
    // optional per-kernel timing (CUDA events on the launch stream), see vrg_profile
    bool prof = false;
    std::vector<cudaEvent_t> ev;   // 4 events per enqueued iteration: decide begin/end, cancel begin/end
    size_t ev_used = 0;
    int64_t prof_sweeps0 = 0;      // C_SWEEPS when the pending events started
    double prof_ms[2] = {0, 0};
    int64_t prof_n[2] = {0, 0};
    // peer-memory transport (multi-GPU, see vrg_p2p.cuh)
    bool p2p_on = false;
    P2P q;
    uint32_t *d_recv = nullptr;
    unsigned long long *d_flags = nullptr;
    long long *d_slots = nullptr;
    std::vector<void *> ipc_opened;
    long long epoch = 0;
    // second stream of the pipelined run: the statistics exchange + next decision table beside the next sweep
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // continuous-intensity mode (vrg_parzen.cuh)
    Cont cq;
    bool cont_alloc = false;
    // CUDA graph of one batch of iterations (vrg_run)
    cudaGraphExec_t gexec = nullptr;
    uint64_t gsig = 0;
    int64_t glaunches = 0;
    bool graph_ok = true;
    // fused tail of an iteration (vrg_tail.cuh): one cooperative launch per iteration behind the sweep
    unsigned int *d_gbar = nullptr;   // device-wide barrier words
    unsigned long long *d_tail_dbg = nullptr;  // phase timings of the tail kernel (profiling runs)
    bool tail_ok = true;              // A/B switch VRG_NO_FUSED_TAIL, or the cooperative launch is not available
    bool tail_checked = false;
    int pipe_mode = -1;               // statistics + next table beside the next sweep (vrg_tail.cuh): -1 = on slabs (where the
                                      // all-to-all exchange is worth hiding), 0 = never, 1 = always (switch VRG_PIPELINE=0|1)
    bool async_pending = false;       // the second stream holds work the next tail kernel has to wait for
};

static const int HASH_CAP = 1 << 18;

// The large per-run buffers (intensity copy, valueMap, level index, label staging) come from the device's stream-ordered pool,
// which keeps freed blocks (vrg_scratch.cuh): a drop-in call that creates and destroys a handle paid up to a second in
// cudaMalloc / cudaFree at C3; vrg_release_scratch() hands the cached blocks back to the driver.
static cudaError_t big_alloc(vrg_handle *h, void **ptr, size_t bytes) {
    vrg_scratch::pool_setup(h->cfg.device);
    return cudaMallocAsync(ptr, bytes ? bytes : 1, h->stream);
}

// kernel<MODE, LATTICE> dispatch on the two run-time switches
#define LAUNCH_ML(KERNEL, GRID, BLK, SMEM, ...)                                                           \
    do {                                                                                                  \
        const bool idx_ = h->cfg.intensity_mode == VRG_INTENSITY_INDEX, lat_ = h->p.lattice != 0;         \
        if (idx_ && lat_) KERNEL<MODE_INDEX, true><<<GRID, BLK, SMEM, h->stream>>>(__VA_ARGS__);          \
        else if (idx_) KERNEL<MODE_INDEX, false><<<GRID, BLK, SMEM, h->stream>>>(__VA_ARGS__);            \
        else if (lat_) KERNEL<MODE_F64_BAND, true><<<GRID, BLK, SMEM, h->stream>>>(__VA_ARGS__);          \
        else KERNEL<MODE_F64_BAND, false><<<GRID, BLK, SMEM, h->stream>>>(__VA_ARGS__);                   \
    } while (0)

static size_t dense_smem_bytes(const Params &p, bool wide = false) {
    return (size_t)((p.LW * 4 + 127) & ~127) + ((DENSE_WARPS * (DENSE_STAGES * 8 + UNIT_RING * 4) + 127) & ~127) +
           (size_t)DENSE_WARPS * DENSE_STAGES * (wide ? WIDE_STAGE_BYTES : STAGE_BYTES);
}
// rows of 31 / 32 words (two 16-word segments): one warp per whole row in the dense sweep, if its 8 KB stages fit
static bool dense_wide(const Params &p) {
    return p.nseg == 2 && p.segw == 16 && dense_smem_bytes(p, true) <= 227 * 1024;
}

static cudaEvent_t prof_event(vrg_handle *h) {
    if (h->ev_used == h->ev.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->ev.push_back(e);
    }
    return h->ev[h->ev_used++];
}
// fold finished event pairs into the totals; only launches that did real work count (no-op launches
// after the exit would drag the average down).  Call after a stream synchronise.
static void prof_collect(vrg_handle *h, int64_t sweeps_now) {
    const int64_t real = sweeps_now - h->prof_sweeps0;
    for (size_t i = 0; i + 3 < h->ev_used; i += 4) {
        if ((int64_t)(i / 4) >= real) break;
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]) == cudaSuccess) { h->prof_ms[0] += ms; h->prof_n[0]++; }
        if (cudaEventElapsedTime(&ms, h->ev[i + 2], h->ev[i + 3]) == cudaSuccess) { h->prof_ms[1] += ms; h->prof_n[1]++; }
    }
    h->ev_used = 0;
    h->prof_sweeps0 = sweeps_now;
}

const char *vrg_last_error(void) { return g_err.c_str(); }
void vrg_set_error_internal(const char *msg) { g_err = msg ? msg : ""; }  // for the other translation units of the library
int vrg_version(void) { return 101; }

static void free_levels(vrg_handle *h) {
    cudaFree(h->d_levels); cudaFree(h->d_pin); cudaFree(h->d_pout); cudaFree(h->d_dbits); cudaFree(h->d_kmat);
    h->d_kmat = nullptr;
    cudaFree(h->d_lstats);
    if (h->separate_gstats) cudaFree(h->d_gstats);
    h->d_levels = h->d_pin = h->d_pout = nullptr; h->d_dbits = nullptr; h->d_lstats = h->d_gstats = nullptr;
}

int vrg_create(const vrg_config *cfg, vrg_handle **out) {
    if (!cfg || !out) return fail(VRG_ERR_ARG, "null argument");
    const int64_t Z = cfg->shape[0], Y = cfg->shape[1], X = cfg->shape[2];
    if (Z <= 0 || Y <= 0 || X <= 0 || cfg->z_begin < 0 || cfg->z_end > Z || cfg->z_begin >= cfg->z_end)
        return fail(VRG_ERR_ARG, "bad shape or slab [%lld,%lld) of Z=%lld", (long long)cfg->z_begin, (long long)cfg->z_end, (long long)Z);
    if (Y > 0x7FFFFFF0 || X > 0x7FFFFFF0) return fail(VRG_ERR_ARG, "axis too long");
    if (cfg->intensity_mode < 0 || cfg->intensity_mode > 3) return fail(VRG_ERR_ARG, "bad intensity_mode");
    if (!(cfg->H > 0) || cfg->iter_max < 1) return fail(VRG_ERR_ARG, "bad H or iter_max");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(VRG_ERR_ARG, "device %d of %d", cfg->device, ndev);
    CK(cudaSetDevice(cfg->device));
    vrg_handle *h = new vrg_handle();
    h->cfg = *cfg;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, cfg->device));
    h->sms = prop.multiProcessorCount;
    h->grid = h->sms * 8;
    h->no_dcache = getenv("VRG_NO_DCACHE") != nullptr;
    h->tail_ok = getenv("VRG_NO_FUSED_TAIL") == nullptr;  // A/B switch: the separate kernels behind the sweep
    if (const char *e = getenv("VRG_PIPELINE")) h->pipe_mode = atoi(e) != 0;  // A/B switch (default: pipelined on slabs only)
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
    Params &p = h->p;
    memset(&p, 0, sizeof p);
    h->nz_own = cfg->z_end - cfg->z_begin;
    p.Y = (int)Y; p.X = (int)X;
    p.XW = (int)((X + 31) / 32);
    p.WP = (p.XW + 3) & ~3;
    p.nseg = (p.XW + WORDS_PER_WARP - 1) / WORDS_PER_WARP;
    p.segw = (p.XW + p.nseg - 1) / p.nseg;  // equal-width segments
    p.nzl = (int)h->nz_own + 2 * HALO;
    p.own_lo = HALO; p.own_hi = HALO + (int)h->nz_own;
    h->ext_lo = std::max<int64_t>(0, cfg->z_begin - HALO);
    h->ext_hi = std::min<int64_t>(Z, cfg->z_end + HALO);
    p.valid_lo = (int)(h->ext_lo - (cfg->z_begin - HALO));
    p.valid_hi = (int)(h->ext_hi - (cfg->z_begin - HALO));
    p.tail_mask = (X % 32) ? ((1u << (X % 32)) - 1u) : 0xFFFFFFFFu;
    p.plane_words = (long long)Y * p.WP;
    p.plane_vox = (long long)Y * X;
    p.mhH = -0.5 * cfg->H;
    p.dirty_lists = cfg->intensity_mode == VRG_INTENSITY_F64_BAND || cfg->intensity_mode == VRG_INTENSITY_INDEX ||
                    (cfg->intensity_mode == VRG_INTENSITY_F64_DENSE && !h->no_dcache);  // without Dc every dense sweep is a refresh
    {   // rows per work unit of the dense sweep: long units on large volumes (fewer window restarts), short ones on thin slabs
        const long long rows_per_warp = (long long)(h->nz_own + 2) * Y * (p.nseg == 2 && p.segw == 16 ? 1 : p.nseg) / ((long long)h->sms * DENSE_WARPS);
        p.dense_rows = rows_per_warp >= 96 ? 8 : 4;  // measured: profiles/README.md (r2b, r2c)
    }
    h->plane_bytes = (size_t)p.nzl * p.plane_words * sizeof(uint32_t);
    h->rowflag_bytes = (size_t)p.nzl * Y * p.nseg;
    const size_t nvox = (size_t)p.nzl * p.plane_vox;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **ptr, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(ptr, bytes); };
    alloc((void **)&h->d_S, h->plane_bytes);
    alloc((void **)&h->d_E, h->plane_bytes);
    alloc((void **)&h->d_F, h->plane_bytes);
    alloc((void **)&h->d_C, h->plane_bytes);
    if (cfg->intensity_mode == VRG_INTENSITY_F64_DENSE && !h->no_dcache) alloc((void **)&h->d_Dc, h->plane_bytes);
    alloc((void **)&h->d_rowflag, h->rowflag_bytes);
    h->unitmap_bytes = (size_t)p.nzl * ((Y + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT) * p.nseg;
    alloc((void **)&h->d_unitmap, h->unitmap_bytes);
    p.front_cap = 1 + (int)((size_t)h->nz_own * Y * p.nseg);
    alloc((void **)&h->d_front, 2 * (size_t)p.front_cap * sizeof(int));
    alloc((void **)&h->d_dirty, 2 * (size_t)p.front_cap * sizeof(int));
    alloc((void **)&h->d_stamp, h->rowflag_bytes * sizeof(int));
    alloc((void **)&h->d_ctrl, C_WORDS * sizeof(long long));
    alloc((void **)&h->d_trace, 3 * (cfg->iter_max + 2) * sizeof(long long));
    alloc((void **)&h->d_hash, (size_t)HASH_CAP * sizeof(unsigned long long));
    alloc((void **)&h->d_hkeys, (size_t)VRG_MAX_LEVELS * sizeof(unsigned long long));
    alloc((void **)&h->d_hcount, 4 * sizeof(int));
    alloc((void **)&h->d_gbar, 4 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(h->d_gbar, 0, 4 * sizeof(unsigned int));
    alloc((void **)&h->d_tail_dbg, (16 + 2 * (size_t)h->sms) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(h->d_tail_dbg, 0, (16 + 2 * (size_t)h->sms) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&h->h_ctrl, C_WORDS * sizeof(long long));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&h->h_poll, 2 * C_WORDS * sizeof(long long));
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&h->ev_poll[i], cudaEventDisableTiming);
    if (e != cudaSuccess) {
        int code = fail(e == cudaErrorMemoryAllocation ? VRG_ERR_NOMEM : VRG_ERR_CUDA, "allocation: %s", cudaGetErrorString(e));
        vrg_destroy(h);
        return code;
    }
    (void)nvox;  // the input buffers are allocated on the first vrg_upload*; vrg_attach_device needs none
    p.S = h->d_S; p.F = h->d_F; p.Cq = h->d_C; p.rowflag = h->d_rowflag; p.front = h->d_front; p.unitmap = h->d_unitmap; p.dirty = h->d_dirty; p.stamp = h->d_stamp;
    p.data = h->d_data;
    p.Dc = h->d_Dc;
    p.ctrl = h->d_ctrl; p.trace = h->d_trace;
    *out = h;
    return VRG_OK;
}

int vrg_destroy(vrg_handle *h) {
    if (!h) return VRG_OK;
    cudaSetDevice(h->cfg.device);
    cudaStreamSynchronize(h->stream);  // also a caller's stream set by vrg_set_stream, the legacy default one (NULL) included
    for (void *big : {(void *)h->d_data, (void *)h->d_vm, (void *)h->d_index, (void *)h->d_labels})
        if (big) cudaFreeAsync(big, h->stream);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_S); cudaFree(h->d_E); cudaFree(h->d_F); cudaFree(h->d_C); cudaFree(h->d_Dc); cudaFree(h->d_rowflag); cudaFree(h->d_front); cudaFree(h->d_unitmap); cudaFree(h->d_dirty); cudaFree(h->d_stamp);
    cudaFree(h->d_ctrl); cudaFree(h->d_trace); cudaFree(h->d_hash); cudaFree(h->d_hkeys); cudaFree(h->d_hcount); cudaFree(h->d_gbar); cudaFree(h->d_tail_dbg);
    free_levels(h);
    if (h->cont_alloc) {
        cudaFree(h->cq.pin); cudaFree(h->cq.pout); cudaFree(h->cq.B); cudaFree(h->cq.newlist); cudaFree(h->cq.oldlist);
        cudaFree(h->cq.rowlist); cudaFree(h->cq.count); cudaFree(h->cq.partial); cudaFree(h->cq.abrowlist); cudaFree(h->cq.AB);
    }
    if (h->gexec) cudaGraphExecDestroy(h->gexec);
    if (h->side_stream) { cudaStreamSynchronize(h->side_stream); cudaStreamDestroy(h->side_stream); }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (void *o : h->ipc_opened) cudaIpcCloseMemHandle(o);
    cudaFree(h->d_recv); cudaFree(h->d_flags); cudaFree(h->d_slots);
    if (h->h_ctrl) cudaFreeHost(h->h_ctrl);
    if (h->h_poll) cudaFreeHost(h->h_poll);
    for (int i = 0; i < 2; ++i) { if (h->h_stage[i]) cudaFreeHost(h->h_stage[i]); if (h->ev_stage[i]) cudaEventDestroy(h->ev_stage[i]); }
    for (int i = 0; i < 2; ++i) if (h->ev_poll[i]) cudaEventDestroy(h->ev_poll[i]);
    for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return VRG_OK;
}

int vrg_set_stream(vrg_handle *h, void *s) {
    if (!h) return fail(VRG_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    h->stream = (cudaStream_t)s;
    h->graph_ok = true;  // a new stream may be capturable where the last one was not
    return VRG_OK;
}

static int ensure_input_buffers(vrg_handle *h) {
    const size_t nvox = (size_t)h->p.nzl * h->p.plane_vox;
    if (!h->d_data) {
        CK(big_alloc(h, (void **)&h->d_data, nvox * sizeof(double)));
        CK(cudaMemsetAsync(h->d_data, 0, nvox * sizeof(double), h->stream));
    }
    if (!h->d_vm) {
        CK(big_alloc(h, (void **)&h->d_vm, nvox));
        CK(cudaMemsetAsync(h->d_vm, 3, nvox, h->stream));
    }
    return VRG_OK;
}

static int upload_impl(vrg_handle *h, const double *data, const uint8_t *vm, cudaMemcpyKind kind) {
    if (!h) return fail(VRG_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->cfg.device));
    Params &p = h->p;
    const size_t off = (size_t)p.valid_lo * p.plane_vox, n = (size_t)(p.valid_hi - p.valid_lo) * p.plane_vox;
    if (h->attached && !(data && vm)) return fail(VRG_ERR_ARG, "inputs are attached: upload both buffers or attach again");
    { int rc_ = ensure_input_buffers(h); if (rc_ != VRG_OK) return rc_; }
    h->attached = false;
    p.data = h->d_data;
    h->vm_base = h->d_vm;
    h->vm_dtype = VRG_DTYPE_U8;
    if (data) {
        CK(cudaMemcpyAsync(h->d_data + off, data, n * sizeof(double), kind, h->stream));
        h->have_data = true;
        h->have_levels = false;
    }
    if (vm) CK(cudaMemcpyAsync(h->d_vm + off, vm, n, kind, h->stream));
    h->inited = false;
    return VRG_OK;
}
// Host -> device copy of a large PAGEABLE buffer: the driver stages such a copy through its own pinned buffer on one thread
// (11 GB/s for the 4.5 GB of config C3); here several host threads fill two pinned staging buffers in turn while the DMA
// engine drains the other one.  Pinned sources (cudaHostAlloc / cudaHostRegister) go straight through.
static int staged_h2d(vrg_handle *h, void *dst, const void *src, size_t bytes) {
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (pinned || bytes < ((size_t)64 << 20)) {
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
        return VRG_OK;
    }
    const size_t CH = (size_t)32 << 20;
    if (!h->h_stage[0]) {
        for (int i = 0; i < 2; ++i) {
            CK(cudaMallocHost((void **)&h->h_stage[i], CH));
            CK(cudaEventCreateWithFlags(&h->ev_stage[i], cudaEventDisableTiming));
        }
    }
    const int nthreads = (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2));
    size_t off = 0;
    for (; off < bytes; off += CH) {
        const int b = (int)(h->stage_seq & 1);
        const size_t len = std::min(CH, bytes - off);
        // the copy that last used this buffer has to be done -- also one of an earlier call (the valueMap follows the intensities
        // through the same two buffers)
        if (h->stage_seq >= 2) CK(cudaEventSynchronize(h->ev_stage[b]));
        ++h->stage_seq;
        const char *s0 = (const char *)src + off;
        char *d0 = (char *)h->h_stage[b];
        std::vector<std::thread> th;
        const size_t part = (len + nthreads - 1) / nthreads;
        for (int t = 1; t < nthreads; ++t) {
            const size_t a = std::min(len, part * t), e = std::min(len, part * (t + 1));
            if (e > a) th.emplace_back([=]() { memcpy(d0 + a, s0 + a, e - a); });
        }
        memcpy(d0, s0, std::min(len, part));
        for (auto &t : th) t.join();
        CK(cudaMemcpyAsync((char *)dst + off, d0, len, cudaMemcpyHostToDevice, h->stream));
        CK(cudaEventRecord(h->ev_stage[b], h->stream));
    }
    return VRG_OK;
}

int vrg_upload(vrg_handle *h, const double *d, const uint8_t *vm) {
    if (!d || !vm) return fail(VRG_ERR_ARG, "null buffer");
    if (!h) return fail(VRG_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->cfg.device));
    Params &p = h->p;
    if (h->attached) { h->attached = false; }
    { int rc_ = ensure_input_buffers(h); if (rc_ != VRG_OK) return rc_; }
    p.data = h->d_data;
    h->vm_base = h->d_vm;
    h->vm_dtype = VRG_DTYPE_U8;
    const size_t off = (size_t)p.valid_lo * p.plane_vox, n = (size_t)(p.valid_hi - p.valid_lo) * p.plane_vox;
    { int rc_ = staged_h2d(h, h->d_data + off, d, n * sizeof(double)); if (rc_ != VRG_OK) return rc_; }
    { int rc_ = staged_h2d(h, h->d_vm + off, vm, n); if (rc_ != VRG_OK) return rc_; }
    h->have_data = true;
    h->have_levels = false;
    h->inited = false;
    CK(cudaStreamSynchronize(h->stream));  // caller may free its buffers
    return VRG_OK;
}
int vrg_upload_device(vrg_handle *h, const double *d, const uint8_t *vm) {
    if (!d && !vm) return fail(VRG_ERR_ARG, "null buffer");
    return upload_impl(h, d, vm, cudaMemcpyDeviceToDevice);
}
static size_t dtype_size(int dtype) {
    switch (dtype) {
        case VRG_DTYPE_U8: case VRG_DTYPE_I8: return 1;
        case VRG_DTYPE_I16: return 2;
        case VRG_DTYPE_I32: case VRG_DTYPE_F32: return 4;
        case VRG_DTYPE_I64: case VRG_DTYPE_F64: return 8;
        default: return 0;
    }
}
// Zero-copy: run on the caller's device-resident extended slab (read-only; must stay alive until the run ends).
int vrg_attach_device(vrg_handle *h, const double *data_dev, const uint8_t *vm_dev) {
    return vrg_attach_device_typed(h, data_dev, vm_dev, VRG_DTYPE_U8);
}
// same, with the valueMap in any vrg_dtype: vrg_init reads it as it is (no conversion pass)
int vrg_attach_device_typed(vrg_handle *h, const double *data_dev, const void *vm_dev, int32_t vm_dtype) {
    if (!h || !data_dev || !vm_dev) return fail(VRG_ERR_ARG, "null argument");
    const size_t es = dtype_size(vm_dtype);
    if (!es) return fail(VRG_ERR_ARG, "unknown valueMap dtype %d", (int)vm_dtype);
    if ((uintptr_t)vm_dev % es) return fail(VRG_ERR_ARG, "valueMap buffer not aligned to its element size");
    CK(cudaSetDevice(h->cfg.device));
    Params &p = h->p;
    const long long off = (long long)p.valid_lo * p.plane_vox;  // kernels index by local plane; only valid planes are read
    p.data = (const double *)((uintptr_t)data_dev - (uintptr_t)off * sizeof(double));
    h->vm_base = (const void *)((uintptr_t)vm_dev - (uintptr_t)off * es);
    h->vm_dtype = vm_dtype;
    h->attached = true;
    h->have_data = true;
    h->have_levels = false;
    h->inited = false;
    return VRG_OK;
}
template <typename T>
static void launch_state(vrg_handle *h, const void *map, long long n, int seg_pass) {
    const long long off = (long long)h->p.valid_lo * h->p.plane_vox;
    k_state_from_map<T><<<h->grid, BLOCK, 0, h->stream>>>((const T *)map, h->d_vm + off, n, seg_pass);
    h->launches++;
}
static int state_pass(vrg_handle *h, const void *map, int dtype, int seg_pass) {
    const long long n = (long long)(h->p.valid_hi - h->p.valid_lo) * h->p.plane_vox;
    switch (dtype) {
        case VRG_DTYPE_I8: launch_state<int8_t>(h, map, n, seg_pass); break;
        case VRG_DTYPE_I16: launch_state<int16_t>(h, map, n, seg_pass); break;
        case VRG_DTYPE_I32: launch_state<int32_t>(h, map, n, seg_pass); break;
        case VRG_DTYPE_I64: launch_state<int64_t>(h, map, n, seg_pass); break;
        case VRG_DTYPE_F32: launch_state<float>(h, map, n, seg_pass); break;
        case VRG_DTYPE_F64: launch_state<double>(h, map, n, seg_pass); break;
        default: launch_state<uint8_t>(h, map, n, seg_pass); break;
    }
    CK(cudaGetLastError());
    return VRG_OK;
}
// update()'s inputs on the device: the intensities attached zero-copy, the state built into the handle's own uint8 valueMap
// from segmentedMap (== 1: segmented) and valueMap (== 4: excluded), each read in its own dtype
int vrg_attach_state_typed(vrg_handle *h, const double *data_dev, const void *seg_dev, int32_t seg_dtype, const void *vm_dev,
                           int32_t vm_dtype) {
    if (!h || !data_dev || !seg_dev || !vm_dev) return fail(VRG_ERR_ARG, "null argument");
    const size_t es = dtype_size(seg_dtype), ev = dtype_size(vm_dtype);
    if (!es || !ev) return fail(VRG_ERR_ARG, "unknown map dtype %d / %d", (int)seg_dtype, (int)vm_dtype);
    if ((uintptr_t)seg_dev % es || (uintptr_t)vm_dev % ev) return fail(VRG_ERR_ARG, "map buffer not aligned to its element size");
    CK(cudaSetDevice(h->cfg.device));
    Params &p = h->p;
    if (!h->d_vm) {
        CK(big_alloc(h, (void **)&h->d_vm, (size_t)p.nzl * p.plane_vox));
        CK(cudaMemsetAsync(h->d_vm, 3, (size_t)p.nzl * p.plane_vox, h->stream));
    }
    { int rc_ = state_pass(h, vm_dev, vm_dtype, 0); if (rc_ != VRG_OK) return rc_; }
    { int rc_ = state_pass(h, seg_dev, seg_dtype, 1); if (rc_ != VRG_OK) return rc_; }
    p.data = (const double *)((uintptr_t)data_dev - (uintptr_t)p.valid_lo * p.plane_vox * sizeof(double));
    h->vm_base = h->d_vm;
    h->vm_dtype = VRG_DTYPE_U8;
    h->attached = true;
    h->have_data = true;
    h->have_levels = false;
    h->inited = false;
    return VRG_OK;
}
int vrg_upload_value_map(vrg_handle *h, const uint8_t *vm) {
    if (!vm) return fail(VRG_ERR_ARG, "null buffer");
    int rc = upload_impl(h, nullptr, vm, cudaMemcpyHostToDevice);
    if (rc == VRG_OK) CK(cudaStreamSynchronize(h->stream));
    return rc;
}

// ---- levels -----------------------------------------------------------------------------------
int vrg_scan_levels(vrg_handle *h, int64_t *n_levels) {
    if (!h || !h->have_data) return fail(VRG_ERR_ARG, "upload data first");
    CK(cudaSetDevice(h->cfg.device));
    const Params &p = h->p;
    CK(cudaMemsetAsync(h->d_hash, 0xFF, (size_t)HASH_CAP * sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(h->d_hcount, 0, 4 * sizeof(int), h->stream));
    const long long n = (long long)(p.valid_hi - p.valid_lo) * p.plane_vox;
    k_scan_levels<<<h->grid, BLOCK, 0, h->stream>>>(p.data + (size_t)p.valid_lo * p.plane_vox, n, h->d_hash, HASH_CAP - 1,
                                                     h->d_hcount, VRG_MAX_LEVELS, h->d_hcount + 1);
    h->launches++;
    CK(cudaGetLastError());
    k_compact_levels<<<h->sms, BLOCK, 0, h->stream>>>(h->d_hash, HASH_CAP, h->d_hkeys, h->d_hcount + 3, VRG_MAX_LEVELS);
    h->launches++;
    int hc[4];
    CK(cudaMemcpyAsync(hc, h->d_hcount, sizeof hc, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (hc[1]) return fail(VRG_ERR_NONFINITE, "intensity volume holds NaN or Inf");
    if (hc[2] || hc[0] > VRG_MAX_LEVELS || hc[3] > VRG_MAX_LEVELS)
        return fail(VRG_ERR_LEVELS, "more than %d distinct intensity levels: continuous data needs the brute-force Parzen path", VRG_MAX_LEVELS);
    std::vector<unsigned long long> keys((size_t)hc[3]);
    if (hc[3]) CK(cudaMemcpy(keys.data(), h->d_hkeys, keys.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    h->levels.clear();
    for (unsigned long long k : keys) { double v; memcpy(&v, &k, 8); h->levels.push_back(v); }
    std::sort(h->levels.begin(), h->levels.end());
    h->n_distinct = (int64_t)h->levels.size();
    if (n_levels) *n_levels = h->n_distinct;
    return VRG_OK;
}

int vrg_get_levels(vrg_handle *h, double *out, int64_t cap) {
    if (!h || !out) return fail(VRG_ERR_ARG, "null argument");
    if ((int64_t)h->levels.size() > cap) return fail(VRG_ERR_ARG, "levels buffer too small");
    memcpy(out, h->levels.data(), h->levels.size() * sizeof(double));
    return VRG_OK;
}

int vrg_set_levels(vrg_handle *h, const double *lv, int64_t n) {
    if (!h || !lv || n < 1) return fail(VRG_ERR_ARG, "bad levels");
    if (n > VRG_MAX_LEVELS) return fail(VRG_ERR_LEVELS, "more than %d distinct intensity levels", VRG_MAX_LEVELS);
    CK(cudaSetDevice(h->cfg.device));
    std::vector<double> s(lv, lv + n);
    std::sort(s.begin(), s.end());
    s.erase(std::unique(s.begin(), s.end()), s.end());
    n = (int64_t)s.size();
    Params &p = h->p;
    // lattice detection: every level sits on lev0 + k*step with k < 65536 -> O(1) voxel->level mapping
    p.lattice = 0; p.lev0 = s[0]; p.inv_step = 0.0;
    std::vector<double> table = s;
    if (n >= 2) {
        double step = s[1] - s[0];
        for (int64_t i = 2; i < n; ++i) step = std::min(step, s[i] - s[i - 1]);
        const double inv = 1.0 / step;
        const double span = (s[n - 1] - s[0]) * inv;
        bool ok = std::isfinite(inv) && span < (double)VRG_MAX_LEVELS - 0.5;
        std::vector<int64_t> ks(n);
        for (int64_t i = 0; ok && i < n; ++i) {
            const double t = (s[i] - s[0]) * inv;
            ks[i] = (int64_t)std::llrint(t);
            if (std::fabs(t - (double)ks[i]) > 1e-6 || (i && ks[i] <= ks[i - 1])) ok = false;
        }
        if (ok) {
            const int64_t K = ks[n - 1] + 1;
            table.assign(K, 0.0);
            for (int64_t k = 0; k < K; ++k) table[k] = s[0] + (double)k * step;
            for (int64_t i = 0; i < n; ++i) table[ks[i]] = s[i];
            p.lattice = 1; p.inv_step = inv;
        }
    } else {
        p.lattice = 1; p.inv_step = 1.0;
    }
    h->levels = s;
    h->n_distinct = n;
    // same table size as last time: keep every buffer (stable device pointers: hosts may hold CUDA graphs over them)
    const bool keep = h->d_levels != nullptr && p.L == (int)table.size();
    p.L = (int)table.size();
    p.LW = (p.L + 31) / 32;
    const size_t sb = (size_t)(2 * p.L + ST_EXTRA) * sizeof(long long);
    if (!keep) {
        free_levels(h);
        h->separate_gstats = false;
        CK(cudaMalloc((void **)&h->d_levels, p.L * sizeof(double)));
        CK(cudaMalloc((void **)&h->d_pin, p.L * sizeof(double)));
        CK(cudaMalloc((void **)&h->d_pout, p.L * sizeof(double)));
        CK(cudaMalloc((void **)&h->d_dbits, 2 * (size_t)p.LW * sizeof(uint32_t)));
        CK(cudaMemsetAsync(h->d_dbits, 0, 2 * (size_t)p.LW * sizeof(uint32_t), h->stream));
        CK(cudaMalloc((void **)&h->d_lstats, sb));
        h->d_gstats = h->d_lstats;
        if (p.L <= 2048) CK(cudaMalloc((void **)&h->d_kmat, (size_t)p.L * p.L * sizeof(double)));
    }
    CK(cudaMemcpyAsync(h->d_levels, table.data(), p.L * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->d_pin, 0, p.L * sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->d_pout, 0, p.L * sizeof(double), h->stream));
    CK(cudaStreamSynchronize(h->stream));  // `table` is a local
    p.levels = h->d_levels; p.pin = h->d_pin; p.pout = h->d_pout; p.dbits = h->d_dbits;
    p.lstats = h->d_lstats; p.gstats = h->d_gstats;
    p.kmat = nullptr;
    if (h->d_kmat) {
        k_kmat<<<h->grid, BLOCK, 0, h->stream>>>(p, h->d_kmat);
        h->launches++;
        CK(cudaGetLastError());
        p.kmat = h->d_kmat;
    }
    h->have_levels = true;
    h->inited = false;
    if (h->cfg.intensity_mode == VRG_INTENSITY_INDEX) {
        const size_t nvox = (size_t)p.nzl * p.plane_vox, voff = (size_t)p.valid_lo * p.plane_vox;
        const long long nval = (long long)(p.valid_hi - p.valid_lo) * p.plane_vox;
        if (!h->d_index) {
            CK(big_alloc(h, (void **)&h->d_index, nvox * sizeof(uint16_t)));
            CK(cudaMemsetAsync(h->d_index, 0, nvox * sizeof(uint16_t), h->stream));
        }
        if (p.lattice) k_build_index<true><<<h->grid, BLOCK, 0, h->stream>>>(p, p.data + voff, h->d_index + voff, nval);
        else k_build_index<false><<<h->grid, BLOCK, 0, h->stream>>>(p, p.data + voff, h->d_index + voff, nval);
        h->launches++;
        CK(cudaGetLastError());
        p.index = h->d_index;
    }
    return VRG_OK;
}

int vrg_use_separate_global_stats(vrg_handle *h) {
    if (!h || !h->have_levels) return fail(VRG_ERR_ARG, "set levels first");
    if (h->separate_gstats) return VRG_OK;
    CK(cudaSetDevice(h->cfg.device));
    const size_t sb = (size_t)(2 * h->p.L + ST_EXTRA) * sizeof(long long);
    CK(cudaMalloc((void **)&h->d_gstats, sb));
    CK(cudaMemsetAsync(h->d_gstats, 0, sb, h->stream));
    h->separate_gstats = true;
    h->p.gstats = h->d_gstats;
    return VRG_OK;
}

// ---- init -------------------------------------------------------------------------------------
static int launch_init_hist(vrg_handle *h) {
    const Params &p = h->p;
    // lane-private shared histograms (64 B per level per warp)
    const size_t per_warp = (size_t)((p.L + 1) & ~1) * 32 * sizeof(uint16_t);
    if (!h->hist_attr_set) {
        CK(cudaFuncSetAttribute(k_init_hist_private<MODE_INDEX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_private<MODE_INDEX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_private<MODE_F64_BAND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_private<MODE_F64_BAND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_shared<MODE_INDEX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_shared<MODE_INDEX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_shared<MODE_F64_BAND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CK(cudaFuncSetAttribute(k_init_hist_shared<MODE_F64_BAND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        h->hist_attr_set = true;
    }
    // TMA-staged: the level source streams through a per-warp ring (16-byte aligned row segments only), one shared-memory
    // histogram per warp (atomics), many warps per SM
    const size_t elem = h->cfg.intensity_mode == VRG_INTENSITY_INDEX ? sizeof(uint16_t) : sizeof(double);
    const uintptr_t src_base = h->cfg.intensity_mode == VRG_INTENSITY_INDEX ? (uintptr_t)p.index : (uintptr_t)p.data;
    if (((size_t)p.X * elem) % 16 == 0 && (src_base & 15) == 0) {
        const size_t stage_bytes = ((size_t)p.segw * 32 * elem + 127) & ~(size_t)127;
        const size_t per_w = (size_t)((p.L + 1) & ~1) * sizeof(unsigned int);
        const size_t per = per_w + HIST_STAGES * stage_bytes + HIST_STAGES * 8;
        // the kernel evaluates whole batches of 10 words: on a short row the last batch reads (and ignores) up to 2560 bytes
        // behind its stage, which must still be shared memory of this block
        const size_t slack = 10 * 32 * sizeof(double);
        const int hw = (int)std::min<size_t>(16, (227 * 1024 - 256 - slack) / per);
        if (hw >= 8) {
            const size_t smem = (((size_t)hw * HIST_STAGES * 8 + 127) & ~(size_t)127) + (size_t)hw * HIST_STAGES * stage_bytes + hw * per_w + slack;
            LAUNCH_ML(k_init_hist_shared, h->sms, hw * 32, smem, p, hw, (int)stage_bytes);
            return VRG_OK;
        }
    }
    const int hw = (int)std::min<size_t>(16, (220 * 1024) / per_warp);
    if (hw >= 4) {
        LAUNCH_ML(k_init_hist_private, h->sms, hw * 32, hw * per_warp, p, hw);
        return VRG_OK;
    }
    const size_t one = (size_t)2 * p.L * sizeof(unsigned int);
    const int copies = (int)std::min<size_t>(WARPS, (48 * 1024) / one);
    LAUNCH_ML(k_init_hist, h->grid, BLOCK, copies * one, p, copies);
    return VRG_OK;
}

static int cont_alloc(vrg_handle *h) {
    if (h->cont_alloc) return VRG_OK;
    const Params &p = h->p;
    const size_t nvox = (size_t)p.nzl * p.plane_vox;
    if (nvox >= 0x7FFFFFFFull) return fail(VRG_ERR_ARG, "continuous mode: volume too large (%zu voxels)", nvox);
    Cont &q = h->cq;
    memset(&q, 0, sizeof q);
    q.cap = (int)std::min<size_t>(nvox, (size_t)1 << 18);
    const size_t ntiles = ((size_t)q.cap + CONT_TILE - 1) / CONT_TILE;
    CK(cudaMalloc((void **)&q.pin, nvox * sizeof(double)));
    CK(cudaMalloc((void **)&q.pout, nvox * sizeof(double)));
    CK(cudaMalloc((void **)&q.B, h->plane_bytes));
    CK(cudaMalloc((void **)&q.newlist, (size_t)q.cap * sizeof(int)));
    CK(cudaMalloc((void **)&q.oldlist, (size_t)q.cap * sizeof(int)));
    CK(cudaMalloc((void **)&q.rowlist, h->rowflag_bytes * sizeof(int)));
    CK(cudaMalloc((void **)&q.abrowlist, h->rowflag_bytes * sizeof(int)));
    CK(cudaMalloc((void **)&q.AB, h->plane_bytes));
    CK(cudaMalloc((void **)&q.count, CC_WORDS * sizeof(int)));
    CK(cudaMalloc((void **)&q.partial, ntiles * CONT_SPLIT * CONT_TILE * 2 * sizeof(double)));
    h->cont_alloc = true;
    return VRG_OK;
}

// bit-planes from the valueMap, read in its own dtype (vrg_attach_device_typed)
static void launch_init_planes(vrg_handle *h) {
    const Params &p = h->p;
    switch (h->vm_dtype) {
        case VRG_DTYPE_I8: k_init_planes<int8_t><<<h->grid, BLOCK, 0, h->stream>>>(p, (const int8_t *)h->vm_base, h->d_E); break;
        case VRG_DTYPE_I16: k_init_planes<int16_t><<<h->grid, BLOCK, 0, h->stream>>>(p, (const int16_t *)h->vm_base, h->d_E); break;
        case VRG_DTYPE_I32: k_init_planes<int32_t><<<h->grid, BLOCK, 0, h->stream>>>(p, (const int32_t *)h->vm_base, h->d_E); break;
        case VRG_DTYPE_I64: k_init_planes<int64_t><<<h->grid, BLOCK, 0, h->stream>>>(p, (const int64_t *)h->vm_base, h->d_E); break;
        case VRG_DTYPE_F32: k_init_planes<float><<<h->grid, BLOCK, 0, h->stream>>>(p, (const float *)h->vm_base, h->d_E); break;
        case VRG_DTYPE_F64: k_init_planes<double><<<h->grid, BLOCK, 0, h->stream>>>(p, (const double *)h->vm_base, h->d_E); break;
        default: k_init_planes<uint8_t><<<h->grid, BLOCK, 0, h->stream>>>(p, (const uint8_t *)h->vm_base, h->d_E); break;
    }
}

// init of the continuous mode: no level table; region sizes by counting, every band voxel gets its full sums
static int cont_init(vrg_handle *h) {
    Params &p = h->p;
    if (p.valid_lo != p.own_lo || p.valid_hi != p.own_hi) return fail(VRG_ERR_ARG, "continuous mode runs on a single slab");
    if (!h->d_lstats || p.L != 0) {
        free_levels(h);
        h->separate_gstats = false;
        p.L = 0; p.LW = 0; p.lattice = 0; p.levels = nullptr; p.kmat = nullptr; p.dbits = nullptr; p.pin = p.pout = nullptr;
        CK(cudaMalloc((void **)&h->d_lstats, ST_EXTRA * sizeof(long long)));
        h->d_gstats = h->d_lstats;
        p.lstats = h->d_lstats; p.gstats = h->d_gstats;
    }
    { int rc_ = cont_alloc(h); if (rc_ != VRG_OK) return rc_; }
    Cont &q = h->cq;
    const size_t nvox = (size_t)p.nzl * p.plane_vox;
    CK(cudaMemsetAsync(h->d_S, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_E, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_F, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(q.B, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(q.pin, 0, nvox * sizeof(double), h->stream));
    CK(cudaMemsetAsync(q.pout, 0, nvox * sizeof(double), h->stream));
    CK(cudaMemsetAsync(q.count, 0, CC_WORDS * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_rowflag, 0, h->rowflag_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_front, 0, 2 * (size_t)p.front_cap * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_dirty, 0, 2 * (size_t)p.front_cap * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_stamp, 0xFF, h->rowflag_bytes * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_unitmap, 0, h->unitmap_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_lstats, 0, ST_EXTRA * sizeof(long long), h->stream));
    CK(cudaMemsetAsync(h->d_trace, 0, 3 * (h->cfg.iter_max + 2) * sizeof(long long), h->stream));
    long long c[C_WORDS];
    memset(c, 0, sizeof c);
    c[C_STATUS] = RUNNING; c[C_ITER] = 1; c[C_ITER_MAX] = h->cfg.iter_max; c[C_MAX_SEG] = h->cfg.max_segment_size;
    c[C_TRACE_N] = 1; c[C_FULL_SWEEP] = 1; c[C_EPOCH] = ++h->epoch;
    memcpy(h->h_ctrl, c, sizeof c);
    CK(cudaMemcpyAsync(h->d_ctrl, h->h_ctrl, sizeof c, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->d_C, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(q.AB, 0, h->plane_bytes, h->stream));
    p.E = h->d_E; p.C = h->d_C;
    launch_init_planes(h);
    k_init_bands<<<h->grid, BLOCK, 0, h->stream>>>(p);  // E = Eraw & ~dil26(S), VRG:137
    k_cont_count<<<h->grid, BLOCK, 0, h->stream>>>(p);
    k_cont_band<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    k_cont_full1<<<dim3(h->sms, CONT_SPLIT), BLOCK, 0, h->stream>>>(p, q);
    k_cont_full2<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    h->launches += 6;
    CK(cudaGetLastError());
    long long ex[ST_EXTRA];
    int cc[CC_WORDS];
    CK(cudaMemcpyAsync(ex, h->d_lstats, sizeof ex, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(cc, q.count, sizeof cc, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ex[ST_BAD_LABEL]) return fail(VRG_ERR_LABEL, "initial valueMap may only hold labels 0 (seed), 3 (outside) and 4 (excluded)");
    if (ex[ST_N_EXCL] == 0) { p.E = nullptr; p.C = nullptr; }  // no label 4: skip the absorb path
    if (ex[ST_N_IN] == 0) return fail(VRG_ERR_EMPTY_SEED, "no seed voxel (label 0) in valueMap");
    if (ex[ST_N_BAND] == 0) return fail(VRG_ERR_NO_BAND, "seed has no boundary: every voxel is inside");
    if (cc[CC_OVERFLOW]) return fail(VRG_ERR_ARG, "continuous mode: more than %d band voxels entered at once", q.cap);
    long long row[3] = {-1, ex[ST_N_IN], ex[ST_N_OUT]};
    CK(cudaMemcpyAsync(h->d_trace, row, sizeof row, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->inited = true;
    h->ev_used = 0;
    h->prof_sweeps0 = 0;
    return VRG_OK;
}

static int cont_enqueue_iteration(vrg_handle *h) {
    const Params &p = h->p;
    const Cont &q = h->cq;
    k_cont_begin<<<1, 32, 0, h->stream>>>(p, q);
    k_cont_decide<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    k_cancel<MODE_CONT, false><<<h->grid, BLOCK, 0, h->stream>>>(p);
    k_quirks<<<h->grid, BLOCK, 0, h->stream>>>(p);
    h->launches++;
    if (p.E != nullptr) {  // label 4: absorb around the flips, and remember which voxels joined the outside region
        CK(cudaMemsetAsync(q.AB, 0, h->plane_bytes, h->stream));
        k_absorb<MODE_CONT, false><<<h->grid, BLOCK, 0, h->stream>>>(p, q.AB);
        k_cont_rows<<<1, 1024, 0, h->stream>>>(p, q, 1);
        h->launches += 2;
    }
    k_advance<<<1, 32, 0, h->stream>>>(p);
    k_cont_rows<<<1, 1024, 0, h->stream>>>(p, q, 0);
    k_cont_band<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    k_cont_incr<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    k_cont_full1<<<dim3(h->sms, CONT_SPLIT), BLOCK, 0, h->stream>>>(p, q);
    k_cont_full2<<<h->grid, BLOCK, 0, h->stream>>>(p, q);
    h->launches += 9;
    CK(cudaGetLastError());
    return VRG_OK;
}

int vrg_init(vrg_handle *h) {
    if (!h || !h->have_data) return fail(VRG_ERR_ARG, "upload first");
    CK(cudaSetDevice(h->cfg.device));
    if (h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS) return cont_init(h);
    if (!h->have_levels) {
        int64_t n = 0;
        int rc = vrg_scan_levels(h, &n);
        if (rc != VRG_OK) return rc;
        std::vector<double> lv = h->levels;
        rc = vrg_set_levels(h, lv.data(), (int64_t)lv.size());
        if (rc != VRG_OK) return rc;
    }
    if (h->p2p_on) { int rc_ = vrg_use_separate_global_stats(h); if (rc_ != VRG_OK) return rc_; }
    Params &p = h->p;
    CK(cudaMemsetAsync(h->d_S, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_E, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_F, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_C, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_rowflag, 0, h->rowflag_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_front, 0, 2 * (size_t)p.front_cap * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_stamp, 0xFF, h->rowflag_bytes * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_unitmap, 0, h->unitmap_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_dirty, 0, 2 * (size_t)p.front_cap * sizeof(int), h->stream));
    CK(cudaMemsetAsync(h->d_lstats, 0, (size_t)(2 * p.L + ST_EXTRA) * sizeof(long long), h->stream));
    CK(cudaMemsetAsync(h->d_trace, 0, 3 * (h->cfg.iter_max + 2) * sizeof(long long), h->stream));
    long long c[C_WORDS];
    memset(c, 0, sizeof c);
    c[C_STATUS] = RUNNING; c[C_ITER] = 1; c[C_ITER_MAX] = h->cfg.iter_max; c[C_MAX_SEG] = h->cfg.max_segment_size;
    c[C_TRACE_N] = 1;
    c[C_FULL_SWEEP] = 1;  // the first sweep (index 0) is a full one
    c[C_EPOCH] = ++h->epoch;  // same on every rank: sequence numbers of the peer exchanges
    memcpy(h->h_ctrl, c, sizeof c);
    CK(cudaMemcpyAsync(h->d_ctrl, h->h_ctrl, sizeof c, cudaMemcpyHostToDevice, h->stream));
    p.E = h->d_E; p.C = h->d_C;
    launch_init_planes(h);
    k_init_bands<<<h->grid, BLOCK, 0, h->stream>>>(p);
    { int rc_ = launch_init_hist(h); if (rc_ != VRG_OK) return rc_; }
    h->launches += 3;
    CK(cudaGetLastError());
    if (h->p2p_on) {  // slabs: excluded halo planes and the global statistics, over peer memory
        k_p2p_push_halo<<<h->sms, BLOCK, 0, h->stream>>>(p, h->q, 1 << PK_E, 1);
        k_p2p_wait_unpack_halo<<<h->sms, BLOCK, 0, h->stream>>>(p, h->q, 1 << PK_E, 1, 0);
        k_p2p_stats<<<1, STATS_BLOCK, 0, h->stream>>>(p, h->q, h->d_gstats, 1);
        h->launches += 3;
        CK(cudaGetLastError());
    }
    // the init row of the trace and the error checks need the counters on the host
    std::vector<long long> ex(ST_EXTRA);
    const long long *src_stats = h->p2p_on ? h->d_gstats : h->d_lstats;
    CK(cudaMemcpyAsync(ex.data(), src_stats + 2 * p.L, ST_EXTRA * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, C_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_ctrl[C_STATUS] == EXIT_PEER_TIMEOUT) return fail(VRG_ERR_CUDA, "peer GPU did not answer during init (p2p timeout)");
    if (ex[ST_BAD_LABEL]) return fail(VRG_ERR_LABEL, "initial valueMap may only hold labels 0 (seed), 3 (outside) and 4 (excluded)");
    if (ex[ST_N_EXCL] == 0 && (!h->separate_gstats || h->p2p_on)) { p.E = nullptr; p.C = nullptr; }  // no label 4: skip the absorb path
    h->inited = true;
    h->ev_used = 0;
    h->prof_sweeps0 = 0;
    if (!h->separate_gstats || h->p2p_on) {  // the global view is known here (single slab, or slabs over peer memory)
        if (ex[ST_N_IN] == 0) return fail(VRG_ERR_EMPTY_SEED, "no seed voxel (label 0) in valueMap");
        if (ex[ST_N_BAND] == 0) return fail(VRG_ERR_NO_BAND, "seed has no boundary: every voxel is inside");
        long long row[3] = {-1, ex[ST_N_IN], ex[ST_N_OUT]};
        CK(cudaMemcpyAsync(h->d_trace, row, sizeof row, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return VRG_OK;
}

// ---- iteration ----------------------------------------------------------------------------------
#define NEED_INIT() \
    if (!h || !h->inited) return fail(VRG_ERR_ARG, "init first"); \
    CK(cudaSetDevice(h->cfg.device))

// slim: the pipelined run's sweep, which leaves room for the statistics / table kernels beside it (vrg_tail.cuh)
static int enqueue_sweep(vrg_handle *h, bool slim = false) {
    const Params &p = h->p;
    const size_t smem = (size_t)p.LW * sizeof(uint32_t);
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    if (h->cfg.intensity_mode == VRG_INTENSITY_F64_DENSE) {
        const bool wide = dense_wide(p);
        const size_t dsm = dense_smem_bytes(p, wide);
        if ((p.X & 1) == 0 && (((uintptr_t)p.data) & 15) == 0 && dsm <= 227 * 1024) {  // TMA ring: 16-byte aligned row segments
            if (!h->dense_attr_set) {
                CK(cudaFuncSetAttribute(k_sweep_dense<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense_slim<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense_slim<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense_slim<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                CK(cudaFuncSetAttribute(k_sweep_dense_slim<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                h->dense_attr_set = true;
            }
            if (slim) {
                if (wide && p.lattice) k_sweep_dense_slim<true, true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
                else if (wide) k_sweep_dense_slim<false, true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
                else if (p.lattice) k_sweep_dense_slim<true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
                else k_sweep_dense_slim<false><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
            } else if (wide && p.lattice) k_sweep_dense<true, true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
            else if (wide) k_sweep_dense<false, true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
            else if (p.lattice) k_sweep_dense<true><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
            else k_sweep_dense<false><<<h->sms, DENSE_WARPS * 32, dsm, h->stream>>>(p);
        } else if (p.lattice) k_sweep_dense_ldg<true><<<h->grid, BLOCK, smem, h->stream>>>(p);
        else k_sweep_dense_ldg<false><<<h->grid, BLOCK, smem, h->stream>>>(p);
        if (p.Dc != nullptr) {  // every sweep the refresh kernel above returns from at once: D from Dc, no shared memory
            // 4 blocks of 256 threads x 48 registers per SM: one wave (8 would not all be resident: a second wave behind the
            // first), half the SM's threads free for the pipelined run's statistics / table kernels
            k_sweep_band<MODE_F64_DENSE, false><<<h->sms * 4, BLOCK, 0, h->stream>>>(p);
            h->launches++;
        }
    } else {
        LAUNCH_ML(k_sweep_band, h->grid, BLOCK, smem, p);
    }
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_decide(vrg_handle *h) {
    NEED_INIT();
    k_table<<<h->p.LW, TABLE_BLOCK, 0, h->stream>>>(h->p, 0);
    h->launches++;
    return enqueue_sweep(h);
}
int vrg_enqueue_cancel(vrg_handle *h) {
    NEED_INIT();
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    LAUNCH_ML(k_cancel, h->grid, BLOCK, 0, h->p);
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_absorb(vrg_handle *h) {
    NEED_INIT();
    if (!h->p.E) return VRG_OK;
    LAUNCH_ML(k_absorb, h->grid, BLOCK, 0, h->p, nullptr);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_flip(vrg_handle *h) {
    NEED_INIT();
    // own planes were flipped inside k_cancel; only a slab with neighbours has halo planes to follow
    if (!(h->p.valid_lo == h->p.own_lo && h->p.valid_hi == h->p.own_hi)) {
        k_flip_halo<<<h->sms, BLOCK, 0, h->stream>>>(h->p);
        h->launches++;
    }
    k_quirks<<<h->grid, BLOCK, 0, h->stream>>>(h->p);  // order-dependence counters: needs the flipped halo planes
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_table(vrg_handle *h) {
    NEED_INIT();
    if (h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS) return fail(VRG_ERR_ARG, "the continuous mode has no table");
    k_table<<<h->p.LW, TABLE_BLOCK, 0, h->stream>>>(h->p, 0);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_advance(vrg_handle *h) {
    NEED_INIT();
    k_advance<<<1, 32, 0, h->stream>>>(h->p);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}

// ---- peer-memory transport ---------------------------------------------------------------------------
// phase 0: executed flips (and cancelled flips when label 4 is present) after cancel; phase 1: excluded plane after flip
int vrg_enqueue_p2p_halo(vrg_handle *h, int phase) {
    NEED_INIT();
    if (!h->p2p_on) return fail(VRG_ERR_ARG, "p2p transport not connected");
    const int kinds = phase == 0 ? ((1 << PK_F) | (h->p.E ? (1 << PK_C) : 0)) : (h->p.E ? (1 << PK_E) : 0);
    if (!kinds) return VRG_OK;
    k_p2p_push_halo<<<h->sms, BLOCK, 0, h->stream>>>(h->p, h->q, kinds, 0);
    k_p2p_wait_unpack_halo<<<h->sms, BLOCK, 0, h->stream>>>(h->p, h->q, kinds, 0, phase == 0);
    h->launches += 2;
    if (phase == 0) {
        k_quirks<<<h->grid, BLOCK, 0, h->stream>>>(h->p);
        h->launches++;
    }
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_enqueue_p2p_stats(vrg_handle *h) {
    NEED_INIT();
    if (!h->p2p_on) return fail(VRG_ERR_ARG, "p2p transport not connected");
    k_p2p_stats<<<1, STATS_BLOCK, 0, h->stream>>>(h->p, h->q, h->d_gstats, 0);  // includes the advance step
    h->launches += 1;
    CK(cudaGetLastError());
    return VRG_OK;
}

// Allocates this rank's receive buffer, flag words and statistics mailbox and returns their three CUDA IPC handles
// (3 x 64 bytes).  Every rank then passes all ranks' handles, in rank order, to vrg_p2p_connect.
int vrg_p2p_export(vrg_handle *h, int world, void *handles_out) {
    if (!h || !handles_out || world < 2 || world > P2P_MAX_WORLD) return fail(VRG_ERR_ARG, "world must be 2..%d", P2P_MAX_WORLD);
    CK(cudaSetDevice(h->cfg.device));
    const Params &p = h->p;
    const int slot_words = 2 * VRG_MAX_LEVELS + ST_EXTRA;
    if (!h->d_recv) {
        const size_t rb = (size_t)2 * P2P_KINDS * 2 * HALO * p.plane_words * sizeof(uint32_t)   // two sequence parities
                          + (size_t)2 * 2 * HALO * p.plane_words * sizeof(unsigned long long);      // + the tagged slots (p2p_ll_region)
        const size_t sb = (size_t)2 * world * slot_words * sizeof(long long);
        CK(cudaMalloc((void **)&h->d_recv, rb));
        CK(cudaMalloc((void **)&h->d_flags, FLAG_WORDS_ALL * sizeof(unsigned long long)));
        CK(cudaMalloc((void **)&h->d_slots, sb));
        CK(cudaMemset(h->d_recv, 0, rb));
        CK(cudaMemset(h->d_flags, 0, FLAG_WORDS_ALL * sizeof(unsigned long long)));
        CK(cudaMemset(h->d_slots, 0, sb));
    }
    cudaIpcMemHandle_t *out = (cudaIpcMemHandle_t *)handles_out;
    CK(cudaIpcGetMemHandle(&out[0], h->d_recv));
    CK(cudaIpcGetMemHandle(&out[1], h->d_flags));
    CK(cudaIpcGetMemHandle(&out[2], h->d_slots));
    h->q.slot_words = slot_words;
    h->q.world = world;
    return VRG_OK;
}

int vrg_p2p_connect(vrg_handle *h, int rank, int world, const void *all_handles) {
    if (!h || !all_handles || !h->d_recv || world != h->q.world || rank < 0 || rank >= world)
        return fail(VRG_ERR_ARG, "export first, then connect with the same world size");
    CK(cudaSetDevice(h->cfg.device));
    const cudaIpcMemHandle_t *hs = (const cudaIpcMemHandle_t *)all_handles;
    P2P &q = h->q;
    q.rank = rank; q.world = world;
    q.flags = h->d_flags; q.slots = h->d_slots; q.recv = h->d_recv;
    q.peer_recv[0] = q.peer_recv[1] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { q.peer_flags[r] = h->d_flags; q.peer_slots[r] = h->d_slots; continue; }
        void *pf = nullptr, *ps = nullptr;
        CK(cudaIpcOpenMemHandle(&pf, hs[3 * r + 1], cudaIpcMemLazyEnablePeerAccess));
        CK(cudaIpcOpenMemHandle(&ps, hs[3 * r + 2], cudaIpcMemLazyEnablePeerAccess));
        h->ipc_opened.push_back(pf); h->ipc_opened.push_back(ps);
        q.peer_flags[r] = (unsigned long long *)pf; q.peer_slots[r] = (long long *)ps;
        if (r == rank - 1 || r == rank + 1) {
            void *pr = nullptr;
            CK(cudaIpcOpenMemHandle(&pr, hs[3 * r + 0], cudaIpcMemLazyEnablePeerAccess));
            h->ipc_opened.push_back(pr);
            q.peer_recv[r == rank - 1 ? 0 : 1] = (uint32_t *)pr;
        }
    }
    h->p2p_on = true;
    h->inited = false;
    return VRG_OK;
}

// The same transport for N handles of ONE process (one per device): peer access instead of CUDA IPC mappings.
int vrg_p2p_connect_local(vrg_handle **hs, int world) {
    if (!hs || world < 2 || world > P2P_MAX_WORLD) return fail(VRG_ERR_ARG, "world must be 2..%d", P2P_MAX_WORLD);
    for (int r = 0; r < world; ++r) {
        if (!hs[r]) return fail(VRG_ERR_ARG, "null handle");
        if (r && (hs[r]->cfg.z_begin != hs[r - 1]->cfg.z_end || hs[r]->cfg.device == hs[r - 1]->cfg.device))
            return fail(VRG_ERR_ARG, "handles must own consecutive z-slabs on distinct devices, in rank order");
    }
    for (int r = 0; r < world; ++r) {
        unsigned char dummy[VRG_P2P_HANDLE_BYTES];
        int rc = vrg_p2p_export(hs[r], world, dummy);  // allocates the receive buffer, flag words and mailbox
        if (rc != VRG_OK) return rc;
        CK(cudaSetDevice(hs[r]->cfg.device));
        for (int o = 0; o < world; ++o) {
            if (o == r) continue;
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, hs[r]->cfg.device, hs[o]->cfg.device));
            if (!can) return fail(VRG_ERR_ARG, "device %d cannot access device %d's memory", hs[r]->cfg.device, hs[o]->cfg.device);
            const cudaError_t e = cudaDeviceEnablePeerAccess(hs[o]->cfg.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
            cudaGetLastError();
        }
    }
    for (int r = 0; r < world; ++r) {
        vrg_handle *h = hs[r];
        CK(cudaSetDevice(h->cfg.device));
        P2P &q = h->q;
        q.rank = r; q.world = world;
        q.flags = h->d_flags; q.slots = h->d_slots; q.recv = h->d_recv;
        for (int o = 0; o < world; ++o) { q.peer_flags[o] = hs[o]->d_flags; q.peer_slots[o] = hs[o]->d_slots; }
        q.peer_recv[0] = r > 0 ? hs[r - 1]->d_recv : nullptr;
        q.peer_recv[1] = r + 1 < world ? hs[r + 1]->d_recv : nullptr;
        h->p2p_on = true;
        h->inited = false;
    }
    return VRG_OK;
}

int vrg_poll(vrg_handle *h, vrg_result *res) {
    NEED_INIT();
    long long ex[ST_EXTRA];
    CK(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, C_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(ex, h->p.gstats + 2 * h->p.L, sizeof ex, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->prof) prof_collect(h, h->h_ctrl[C_SWEEPS]);
    if (res) {
        res->iterations = h->h_ctrl[C_ITER];
        res->exit_reason = h->h_ctrl[C_STATUS];
        res->n_in = ex[ST_N_IN]; res->n_out = ex[ST_N_OUT]; res->n_excluded = ex[ST_N_EXCL];
        res->n_levels = h->p.L;
        res->sweeps = h->h_ctrl[C_SWEEPS];
        res->kernel_launches = h->launches;
        res->q_cancelled = ex[ST_Q_CANCELLED]; res->q_add_to_inside = ex[ST_Q_ADD_INSIDE];
        res->q_remove_to_outside = ex[ST_Q_REM_OUTSIDE]; res->q_cancel_repromoted = ex[ST_Q_REPROMOTED];
        res->redone_sweeps = h->h_ctrl[C_REDOS];
    }
    return VRG_OK;
}

int vrg_dense_refresh_sweeps(vrg_handle *h, int64_t *n) {
    if (!h || !n) return fail(VRG_ERR_ARG, "null argument");
    *n = h->inited ? h->h_ctrl[C_REFRESHES] : 0;  // the control block as the last vrg_poll read it
    return VRG_OK;
}

static int enqueue_table(vrg_handle *h) {
    k_table<<<h->p.LW, TABLE_BLOCK, 0, h->stream>>>(h->p, 0);
    h->launches++;
    return VRG_OK;
}

// The fused tail serves the table modes without label 4, on a whole volume or on a slab with the peer-memory transport.
static bool tail_applies(vrg_handle *h) {
    if (!h->tail_ok || h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS || h->p.E != nullptr) return false;
    if (h->separate_gstats && !h->p2p_on) return false;  // slab driven by a host-side collective transport
    if (!h->tail_checked) {
        int coop = 0, nb = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->cfg.device);
        const int smem_max = TAIL_STAGE_LEVELS * 2 * (int)sizeof(double);
        cudaFuncSetAttribute(k_tail<MODE_INDEX, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_INDEX, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_F64_BAND, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_F64_BAND, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_INDEX, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_INDEX, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_F64_BAND, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaFuncSetAttribute(k_tail<MODE_F64_BAND, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_tail<MODE_F64_BAND, true, false>, TAIL_BLOCK, smem_max);
        if (!coop || nb < 1 || h->sms < 2) h->tail_ok = false;
        cudaGetLastError();
        h->tail_checked = true;
    }
    return h->tail_ok;
}

static int enqueue_tail(vrg_handle *h) {
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(h->sms); cfg.blockDim = dim3(TAIL_BLOCK); cfg.dynamicSmemBytes = 0; cfg.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const bool idx = h->cfg.intensity_mode == VRG_INTENSITY_INDEX, lat = h->p.lattice != 0;
    const int p2p = h->p2p_on ? 1 : 0;
    const int stage = h->p.L <= TAIL_STAGE_LEVELS ? 1 : 0;
    cfg.dynamicSmemBytes = stage ? (size_t)2 * h->p.L * sizeof(double) : 0;
    unsigned long long *dbg = h->prof ? h->d_tail_dbg : nullptr;
    cudaError_t e;
#define TAIL_LAUNCH(M, LAT)                                                                                                   \
    (dbg ? cudaLaunchKernelEx(&cfg, k_tail<M, LAT, true>, h->p, h->q, h->d_gstats, h->d_gbar, p2p, stage, dbg)               \
         : cudaLaunchKernelEx(&cfg, k_tail<M, LAT, false>, h->p, h->q, h->d_gstats, h->d_gbar, p2p, stage, dbg))
    if (idx && lat) e = TAIL_LAUNCH(MODE_INDEX, true);
    else if (idx) e = TAIL_LAUNCH(MODE_INDEX, false);
    else if (lat) e = TAIL_LAUNCH(MODE_F64_BAND, true);
    else e = TAIL_LAUNCH(MODE_F64_BAND, false);
#undef TAIL_LAUNCH
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    h->launches++;
    CK(e);
    return VRG_OK;
}

// second stream + events of the pipelined run
static int ensure_side_stream(vrg_handle *h) {
    if (!h->side_stream) {
        CK(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    return VRG_OK;
}

static int enqueue_tail_pipe(vrg_handle *h) {
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(h->sms); cfg.blockDim = dim3(TAIL_BLOCK); cfg.dynamicSmemBytes = 0; cfg.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const bool idx = h->cfg.intensity_mode == VRG_INTENSITY_INDEX, lat = h->p.lattice != 0;
    const int p2p = h->p2p_on ? 1 : 0;
    unsigned long long *dbg = h->prof ? h->d_tail_dbg : nullptr;
    cudaError_t e;
#define TAIL_LAUNCH(M, LAT)                                                                              \
    (dbg ? cudaLaunchKernelEx(&cfg, k_tail_pipe<M, LAT, true>, h->p, h->q, h->d_gbar, p2p, dbg)         \
         : cudaLaunchKernelEx(&cfg, k_tail_pipe<M, LAT, false>, h->p, h->q, h->d_gbar, p2p, dbg))
    if (idx && lat) e = TAIL_LAUNCH(MODE_INDEX, true);
    else if (idx) e = TAIL_LAUNCH(MODE_INDEX, false);
    else if (lat) e = TAIL_LAUNCH(MODE_F64_BAND, true);
    else e = TAIL_LAUNCH(MODE_F64_BAND, false);
#undef TAIL_LAUNCH
    if (h->prof) cudaEventRecord(prof_event(h), h->stream);
    h->launches++;
    CK(e);
    return VRG_OK;
}

// One pipelined iteration: the sweep goes first, only then does the main stream wait for the statistics / table kernels of
// the previous update (they have been running beside this sweep), then the tail kernel; the statistics + table kernels of
// this update are forked to the second stream.
static int enqueue_pipelined(vrg_handle *h) {
    int rc;
    if ((rc = enqueue_sweep(h, true)) != VRG_OK) return rc;
    if (h->async_pending) {
        CK(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
        h->async_pending = false;
    }
    if ((rc = enqueue_tail_pipe(h)) != VRG_OK) return rc;
    CK(cudaEventRecord(h->ev_fork, h->stream));
    CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    k_async_stats<<<1, ASYNC_BLOCK, 0, h->side_stream>>>(h->p, h->q, h->d_gstats, h->p2p_on ? 1 : 0);
    k_async_table<<<h->p.LW, ASYNC_BLOCK, 0, h->side_stream>>>(h->p);
    h->launches += 2;
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev_join, h->side_stream));
    h->async_pending = true;
    return VRG_OK;
}

static int join_async(vrg_handle *h) {
    if (h->async_pending) {
        CK(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
        h->async_pending = false;
    }
    return VRG_OK;
}

static int enqueue_batch(vrg_handle *h, int n) {
    const bool fused = tail_applies(h);
    const bool piped = fused && (h->pipe_mode < 0 ? h->p2p_on : h->pipe_mode != 0);
    if (piped) { int rc_ = ensure_side_stream(h); if (rc_ != VRG_OK) return rc_; }
    for (int k = 0; k < n; ++k) {
        int rc;
        if (h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS) {
            if ((rc = cont_enqueue_iteration(h)) != VRG_OK) return rc;
            continue;
        }
        if (piped) {
            if ((rc = enqueue_pipelined(h)) != VRG_OK) return rc;
            continue;
        }
        if (fused) {  // the table of this sweep was computed by the previous tail (the first one: vrg_run)
            if ((rc = enqueue_sweep(h)) != VRG_OK) return rc;
            if ((rc = enqueue_tail(h)) != VRG_OK) return rc;
            continue;
        }
        if ((rc = vrg_enqueue_decide(h)) != VRG_OK) return rc;
        if ((rc = vrg_enqueue_cancel(h)) != VRG_OK) return rc;
        if (h->p2p_on && (rc = vrg_enqueue_p2p_halo(h, 0)) != VRG_OK) return rc;
        if ((rc = vrg_enqueue_absorb(h)) != VRG_OK) return rc;
        if (h->p2p_on) {  // halo flips were applied while unpacking; the statistics kernel also advances the loop
            if ((rc = vrg_enqueue_p2p_halo(h, 1)) != VRG_OK) return rc;
            if ((rc = vrg_enqueue_p2p_stats(h)) != VRG_OK) return rc;
        } else {
            if ((rc = vrg_enqueue_flip(h)) != VRG_OK) return rc;
            if ((rc = vrg_enqueue_advance(h)) != VRG_OK) return rc;
        }
    }
    return join_async(h);  // a batch ends joined: it may be a captured graph, and the host polls the main stream
}

static uint64_t run_signature(const vrg_handle *h) {
    uint64_t x = 1469598103934665603ull;
    auto mix = [&](const void *ptr, size_t n) {
        const unsigned char *b = (const unsigned char *)ptr;
        for (size_t i = 0; i < n; ++i) { x ^= b[i]; x *= 1099511628211ull; }
    };
    mix(&h->p, sizeof(Params));
    if (h->p2p_on) mix(&h->q, sizeof(P2P));
    const int64_t extra[5] = {h->cfg.intensity_mode, h->p2p_on, h->tail_ok, h->pipe_mode, h->no_dcache};
    mix(extra, sizeof extra);
    return x;
}

// The loop of VRG:58-117.  The host enqueues batches of 8 iterations and reads the device-side status word after each;
// kernels launched after the exit see the status and return at once.  From the second batch on the batch is a CUDA
// graph (captured once per parameter set, replayed), which removes the launch gaps between the short kernels.
int vrg_run(vrg_handle *h, vrg_result *res) {
    NEED_INIT();
    vrg_result r;
    const int check_every = 8;
    const auto t0 = std::chrono::steady_clock::now();
    bool use_graph = !h->prof && h->graph_ok;
    bool first = true, time_flagged = false;
    long long nbatch = 0;
    if (h->cfg.intensity_mode != VRG_INTENSITY_CONTINUOUS) {
        // the decision table + bookkeeping in front of the first sweep; every later one is the last phase of the tail kernel
        // (the separate-kernel path recomputes it in front of each sweep: same stats, same table)
        int rc = enqueue_table(h);
        if (rc != VRG_OK) return rc;
    }
    while (true) {
        bool launched = false;
        if (use_graph && !first) {
            const uint64_t sig = run_signature(h);
            if (!h->gexec || h->gsig != sig) {
                if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
                if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                    const int64_t l0 = h->launches;
                    const int rc = enqueue_batch(h, check_every);
                    cudaGraph_t g = nullptr;
                    const cudaError_t e = cudaStreamEndCapture(h->stream, &g);
                    h->glaunches = h->launches - l0;
                    h->launches = l0;
                    if (rc == VRG_OK && e == cudaSuccess && cudaGraphInstantiate(&h->gexec, g, 0) == cudaSuccess) h->gsig = sig;
                    else {
                        h->gexec = nullptr; h->graph_ok = false;
                        if (getenv("VRG_VERBOSE")) fprintf(stderr, "vrg_b200: CUDA graph capture failed (%s / %s): plain stream launches\n",
                                                           cudaGetErrorString(e), rc == VRG_OK ? "enqueue ok" : vrg_last_error());
                    }
                    if (g) cudaGraphDestroy(g);
                } else h->graph_ok = false;  // e.g. the legacy default stream cannot be captured: stay eager
                cudaGetLastError();
                use_graph = h->graph_ok;
            }
            if (use_graph && h->gexec) {
                CK(cudaGraphLaunch(h->gexec, h->stream));
                h->launches += h->glaunches;
                launched = true;
            }
        }
        if (!launched) {
            const int rc = enqueue_batch(h, check_every);
            if (rc != VRG_OK) return rc;
        }
        first = false;
        // The status word of this batch travels to the host behind it.  With graph replay the host does not wait for it: it
        // queues the next batch first and only then looks at the previous one, so the device never idles between batches (a
        // stream synchronise + a poll + a graph launch cost about 30 us per batch of 8 iterations); the price is one batch of
        // no-op launches after the exit.
        const int slot = (int)(nbatch & 1);
        CK(cudaMemcpyAsync(h->h_poll + slot * C_WORDS, h->d_ctrl, C_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev_poll[slot], h->stream));
        ++nbatch;
        const bool ahead = use_graph && h->gexec != nullptr;
        if (ahead && nbatch < 2) continue;  // nothing older to look at yet
        const int look = ahead ? (int)((nbatch - 2) & 1) : slot;
        CK(cudaEventSynchronize(h->ev_poll[look]));
        const long long st = h->h_poll[look * C_WORDS + C_STATUS];
        if (st == EXIT_PEER_TIMEOUT) return fail(VRG_ERR_CUDA, "peer GPU did not answer (p2p timeout)");
        if (st == EXIT_CONT_OVERFLOW) return fail(VRG_ERR_ARG, "continuous mode: band list overflow (%d voxels)", h->cq.cap);
        if (st != VRG_EXIT_RUNNING) break;
        if (h->cfg.max_seconds > 0 &&
            std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() >= h->cfg.max_seconds) {
            // VRG:97: stop before applying the next flips; the state is that of the last applied update
            if (h->p2p_on) {
                // slabs: the ranks' clocks differ, so the exit is taken collectively -- this rank raises a flag in its own
                // statistics vector, the next exchange sums it, and every rank leaves at the same update (advance_state)
                if (!time_flagged) {
                    static const long long one = 1;
                    CK(cudaMemcpyAsync(h->d_lstats + 2 * h->p.L + ST_TIME_UP, &one, sizeof one, cudaMemcpyHostToDevice, h->stream));
                    time_flagged = true;
                }
                continue;
            }
            CK(cudaStreamSynchronize(h->stream));  // a batch queued ahead finishes first
            CK(cudaMemcpy(h->h_ctrl, h->d_ctrl, sizeof(long long), cudaMemcpyDeviceToHost));
            if (h->h_ctrl[C_STATUS] == VRG_EXIT_RUNNING) {
                h->h_ctrl[C_STATUS] = VRG_EXIT_MAX_TIME;
                CK(cudaMemcpyAsync(h->d_ctrl, h->h_ctrl, sizeof(long long), cudaMemcpyHostToDevice, h->stream));
                CK(cudaStreamSynchronize(h->stream));
            }
            break;
        }
    }
    {   // drain whatever was queued ahead and read the final state
        int rc = vrg_poll(h, &r);
        if (rc != VRG_OK) return rc;
        if (r.exit_reason == EXIT_PEER_TIMEOUT) return fail(VRG_ERR_CUDA, "peer GPU did not answer (p2p timeout)");
        if (r.exit_reason == EXIT_CONT_OVERFLOW) return fail(VRG_ERR_ARG, "continuous mode: band list overflow (%d voxels)", h->cq.cap);
    }
    if (h->p2p_on) {
        // every rank left the loop at the same update: one more statistics exchange folds in what trailed the last one
        k_p2p_stats<<<1, STATS_BLOCK, 0, h->stream>>>(h->p, h->q, h->d_gstats, 2);
        h->launches++;
        CK(cudaGetLastError());
        int rc = vrg_poll(h, &r);
        if (rc != VRG_OK) return rc;
        if (h->h_ctrl[C_PEER_TIMEOUT]) return fail(VRG_ERR_CUDA, "peer GPU did not answer (p2p timeout)");
    }
    if (h->cfg.intensity_mode != VRG_INTENSITY_CONTINUOUS) {  // vrg_get_table: the sums of the state the run leaves behind
        k_table<<<h->p.LW, TABLE_BLOCK, 0, h->stream>>>(h->p, 1);
        h->launches++;
        CK(cudaGetLastError());
    }
    if (res) *res = r;
    return VRG_OK;
}

// ---- update() with caller-chosen flips (VRG:124, flipedPoints given) -----------------------------------------
static int flips_args(vrg_handle *h, const void *coords, int64_t n) {
    if (n < 0 || (n > 0 && !coords)) return fail(VRG_ERR_ARG, "bad flip list");
    const Params &p = h->p;
    if (h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS) return fail(VRG_ERR_ARG, "vrg_apply_flips needs a level-table mode");
    if (h->p2p_on || p.valid_lo != p.own_lo || p.valid_hi != p.own_hi) return fail(VRG_ERR_ARG, "vrg_apply_flips runs on a whole-volume handle");
    return VRG_OK;
}
static int fail_flip_outside(int64_t i, int64_t z, int64_t y, int64_t x) {
    return fail(VRG_ERR_ARG, "flip %lld = (%lld, %lld, %lld) lies outside the volume", (long long)i, (long long)z, (long long)y, (long long)x);
}
// the band state machine on validated device rows (n may be 0)
static int apply_flips_rows(vrg_handle *h, const long long *d_coords, int64_t n, vrg_result *res) {
    const Params &p = h->p;
    CK(cudaMemsetAsync(h->d_F, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_C, 0, h->plane_bytes, h->stream));
    CK(cudaMemsetAsync(h->d_rowflag, 0, h->rowflag_bytes, h->stream));
    k_prepare_apply<<<1, 32, 0, h->stream>>>(p);
    if (n) k_set_flips<<<h->grid, BLOCK, 0, h->stream>>>(p, d_coords, n, h->cfg.z_begin);
    k_mask_flips<<<h->grid, BLOCK, 0, h->stream>>>(p);
    h->launches += 3;
    CK(cudaGetLastError());
    int rc = vrg_enqueue_cancel(h);
    if (rc == VRG_OK) rc = vrg_enqueue_absorb(h);
    if (rc == VRG_OK) rc = vrg_enqueue_flip(h);
    if (rc == VRG_OK) rc = vrg_enqueue_advance(h);
    if (rc == VRG_OK) rc = vrg_enqueue_table(h);  // the sums of the new state; its incremental hint does not hold for foreign flips:
    if (rc == VRG_OK) {
        k_force_full_sweep<<<1, 32, 0, h->stream>>>(h->p);
        h->launches++;
        rc = vrg_poll(h, res);
    }
    return rc;
}
int vrg_apply_flips(vrg_handle *h, const int64_t *coords, int64_t n, vrg_result *res) {
    NEED_INIT();
    { int rc_ = flips_args(h, coords, n); if (rc_ != VRG_OK) return rc_; }
    const Params &p = h->p;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t z = coords[3 * i], y = coords[3 * i + 1], x = coords[3 * i + 2];
        if (z < h->cfg.z_begin || z >= h->cfg.z_end || y < 0 || y >= p.Y || x < 0 || x >= p.X) return fail_flip_outside(i, z, y, x);
    }
    long long *d_coords = nullptr;
    if (n) {
        CK(cudaMalloc((void **)&d_coords, (size_t)n * 3 * sizeof(long long)));
        CK(cudaMemcpyAsync(d_coords, coords, (size_t)n * 3 * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    }
    const int rc = apply_flips_rows(h, d_coords, n, res);
    if (d_coords) { cudaStreamSynchronize(h->stream); cudaFree(d_coords); }
    return rc;
}
// the same with the rows in device memory: validated on the device (one synchronisation for the verdict) before anything changes
int vrg_apply_flips_device(vrg_handle *h, const int64_t *rows_dev, int64_t n, vrg_result *res) {
    NEED_INIT();
    { int rc_ = flips_args(h, rows_dev, n); if (rc_ != VRG_OK) return rc_; }
    if ((uintptr_t)rows_dev % sizeof(int64_t)) return fail(VRG_ERR_ARG, "flip rows not aligned to 8 bytes");
    const long long *d_coords = (const long long *)rows_dev;
    if (n) {
        unsigned long long *d_out = (unsigned long long *)h->d_hcount;  // 16 bytes of scratch: count, first row outside
        CK(cudaMemsetAsync(d_out, 0, sizeof(unsigned long long), h->stream));
        CK(cudaMemsetAsync(d_out + 1, 0xFF, sizeof(unsigned long long), h->stream));
        const long long blocks = std::min<long long>(h->grid, (n + BLOCK - 1) / BLOCK);
        k_check_flips<<<(int)blocks, BLOCK, 0, h->stream>>>(h->p, d_coords, n, h->cfg.z_begin, d_out);
        h->launches++;
        CK(cudaGetLastError());
        unsigned long long v[2];
        CK(cudaMemcpyAsync(v, d_out, sizeof v, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (v[0]) {
            long long r[3];
            CK(cudaMemcpy(r, d_coords + 3 * v[1], sizeof r, cudaMemcpyDeviceToHost));
            return fail_flip_outside((int64_t)v[1], r[0], r[1], r[2]);
        }
    }
    return apply_flips_rows(h, d_coords, n, res);
}

// FNV-1a over the kernel parameter block: a host that replays captured launches (CUDA graphs) re-captures when it moves
int vrg_params_signature(vrg_handle *h, uint64_t *sig) {
    if (!h || !sig) return fail(VRG_ERR_ARG, "null argument");
    uint64_t x = 1469598103934665603ull;
    const unsigned char *b = (const unsigned char *)&h->p;
    for (size_t i = 0; i < sizeof(Params); ++i) { x ^= b[i]; x *= 1099511628211ull; }
    *sig = x ^ (uint64_t)h->cfg.intensity_mode;
    return VRG_OK;
}

// fp64 Parzen-kernel evaluations per second this device sustains (k_exp_peak): the continuous mode's roofline
int vrg_exp_peak(int device, double *evals_per_second) {
    if (!evals_per_second) return fail(VRG_ERR_ARG, "null argument");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int grid = prop.multiProcessorCount * 8, iters = 4096;
    double *out = nullptr;
    CK(cudaMalloc((void **)&out, (size_t)grid * BLOCK * sizeof(double)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    k_exp_peak<<<grid, BLOCK>>>(-1.125, 64, out);  // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(e0));
        k_exp_peak<<<grid, BLOCK>>>(-1.125, iters, out);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best = std::min(best, ms);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *evals_per_second = (double)grid * BLOCK * iters * 8.0 / ((double)best * 1e-3);
    return VRG_OK;
}
int vrg_get_exp_evals(vrg_handle *h, int64_t *evals) {
    NEED_INIT();
    if (!evals) return fail(VRG_ERR_ARG, "null argument");
    long long v = 0;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(&v, h->d_lstats + 2 * h->p.L + ST_EXP_EVALS, sizeof v, cudaMemcpyDeviceToHost));
    *evals = v;
    return VRG_OK;
}

int vrg_profile(vrg_handle *h, int enable) {
    if (!h) return fail(VRG_ERR_ARG, "null handle");
    h->prof = enable != 0;
    if (enable) cudaMemsetAsync(h->d_tail_dbg, 0, (16 + 2 * (size_t)h->sms) * sizeof(unsigned long long), h->stream);
    h->ev_used = 0;
    h->prof_ms[0] = h->prof_ms[1] = 0;
    h->prof_n[0] = h->prof_n[1] = 0;
    return VRG_OK;
}
// phase timings of the tail kernel, collected while vrg_profile is on: us[0..6] = mean microseconds block 0 spent in
// phase 1 (cancel rule + flips), the first device-wide barrier, phase 2 (in-order run: statistics exchange + exit tests, halo
// exchange on the other blocks; pipelined run: halo wait + unpack), the second barrier, phase 3, and for the pipelined run the
// halo push and the counters (the first two parts of its phase 2); us[7..13] the same for the last block of the grid.
int vrg_get_tail_profile(vrg_handle *h, double *us, int64_t *launches) {
    if (!h || !us || !launches) return fail(VRG_ERR_ARG, "null argument");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long d[16];
    CK(cudaMemcpy(d, h->d_tail_dbg, sizeof d, cudaMemcpyDeviceToHost));
    *launches = (int64_t)d[0];
    if (getenv("VRG_VERBOSE") && d[0]) {  // per-block spread of phase 1 and phase 3
        std::vector<unsigned long long> b(2 * (size_t)h->sms);
        CK(cudaMemcpy(b.data(), h->d_tail_dbg + 16, b.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (int ph = 0; ph < 2; ++ph) {
            fprintf(stderr, "vrg_b200: tail phase %d per block (us):", ph ? 3 : 1);
            for (int i = 0; i < h->sms; ++i) fprintf(stderr, " %.1f", (double)b[(size_t)ph * h->sms + i] / (double)d[0] * 1e-3);
            fprintf(stderr, "\n");
        }
    }
    for (int i = 0; i < 7; ++i) {
        us[i] = d[0] ? (double)d[1 + i] / (double)d[0] * 1e-3 : 0.0;
        us[7 + i] = d[0] ? (double)d[9 + i] / (double)d[0] * 1e-3 : 0.0;
    }
    return VRG_OK;
}
int vrg_get_profile(vrg_handle *h, double *ms_total, int64_t *launches) {
    if (!h || !ms_total || !launches) return fail(VRG_ERR_ARG, "null argument");
    for (int i = 0; i < 2; ++i) { ms_total[i] = h->prof_ms[i]; launches[i] = h->prof_n[i]; }
    return VRG_OK;
}

// ---- buffers for a multi-GPU host ------------------------------------------------------------------
int vrg_buffer_info(vrg_handle *h, int which, void **ptr, int64_t *bytes) {
    if (!h || !ptr || !bytes) return fail(VRG_ERR_ARG, "null argument");
    const int64_t sb = (int64_t)(2 * h->p.L + ST_EXTRA) * sizeof(long long);
    switch (which) {
        case VRG_BUF_SEG: *ptr = h->d_S; *bytes = (int64_t)h->plane_bytes; break;
        case VRG_BUF_EXCL: *ptr = h->d_E; *bytes = (int64_t)h->plane_bytes; break;
        case VRG_BUF_FLIPS: *ptr = h->d_F; *bytes = (int64_t)h->plane_bytes; break;
        case VRG_BUF_CANCELLED: *ptr = h->d_C; *bytes = (int64_t)h->plane_bytes; break;
        case VRG_BUF_LOCAL_STATS: *ptr = h->d_lstats; *bytes = sb; break;
        case VRG_BUF_GLOBAL_STATS: *ptr = h->d_gstats; *bytes = sb; break;
        case VRG_BUF_CTRL: *ptr = h->d_ctrl; *bytes = C_WORDS * sizeof(long long); break;
        default: return fail(VRG_ERR_ARG, "unknown buffer %d", which);
    }
    return VRG_OK;
}
int vrg_plane_geometry(vrg_handle *h, int64_t *wpr, int64_t *wpp, int64_t *npl) {
    if (!h) return fail(VRG_ERR_ARG, "null handle");
    if (wpr) *wpr = h->p.WP;
    if (wpp) *wpp = h->p.plane_words;
    if (npl) *npl = h->p.nzl;
    return VRG_OK;
}

// ---- outputs ----------------------------------------------------------------------------------------
static int labels_impl(vrg_handle *h, uint8_t *dev_out, int seg_only) {
    k_labels<uint8_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, dev_out, seg_only);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
int vrg_labels_device(vrg_handle *h, uint8_t *out) {
    NEED_INIT();
    if (!out) return fail(VRG_ERR_ARG, "null buffer");
    return labels_impl(h, out, 0);
}
// labels 0..4 (or the 0/1 segmented map) of the own planes as `dtype`, into a device buffer; on the handle's stream, no sync
int vrg_labels_device_typed(vrg_handle *h, void *out, int32_t dtype, int32_t seg_only) {
    NEED_INIT();
    if (!out) return fail(VRG_ERR_ARG, "null buffer");
    const size_t es = dtype_size(dtype);
    if (!es) return fail(VRG_ERR_ARG, "unknown dtype %d", (int)dtype);
    if ((uintptr_t)out % es) return fail(VRG_ERR_ARG, "output buffer not aligned to its element size");
    const int so = seg_only ? 1 : 0;
    switch (dtype) {
        case VRG_DTYPE_I8: k_labels<int8_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (int8_t *)out, so); break;
        case VRG_DTYPE_I16: k_labels<int16_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (int16_t *)out, so); break;
        case VRG_DTYPE_I32: k_labels<int32_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (int32_t *)out, so); break;
        case VRG_DTYPE_I64: k_labels<int64_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (int64_t *)out, so); break;
        case VRG_DTYPE_F32: k_labels<float><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (float *)out, so); break;
        case VRG_DTYPE_F64: k_labels<double><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (double *)out, so); break;
        default: k_labels<uint8_t><<<h->grid, BLOCK, 0, h->stream>>>(h->p, (uint8_t *)out, so); break;
    }
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}
static int download_impl(vrg_handle *h, uint8_t *out, int seg_only) {
    NEED_INIT();
    if (!out) return fail(VRG_ERR_ARG, "null buffer");
    const size_t n = (size_t)h->nz_own * h->p.plane_vox;
    if (!h->d_labels) CK(big_alloc(h, (void **)&h->d_labels, n));
    int rc = labels_impl(h, h->d_labels, seg_only);
    if (rc != VRG_OK) return rc;
    CK(cudaMemcpyAsync(out, h->d_labels, n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return VRG_OK;
}
// position-sensitive hash of the own planes' labels (see k_hash_labels): slab hashes add up to the whole volume's
int vrg_labels_hash(vrg_handle *h, uint64_t *hash_out) {
    NEED_INIT();
    if (!hash_out) return fail(VRG_ERR_ARG, "null argument");
    const size_t n = (size_t)h->nz_own * h->p.plane_vox;
    if (!h->d_labels) CK(big_alloc(h, (void **)&h->d_labels, n));
    int rc = labels_impl(h, h->d_labels, 0);
    if (rc != VRG_OK) return rc;
    unsigned long long *d_out = (unsigned long long *)(h->d_hcount);  // 16 bytes of scratch, 8-byte aligned (cudaMalloc)
    CK(cudaMemsetAsync(d_out, 0, sizeof(unsigned long long), h->stream));
    k_hash_labels<<<h->grid, BLOCK, 0, h->stream>>>(h->d_labels, (long long)n, (long long)h->cfg.z_begin * h->p.plane_vox, d_out);
    h->launches++;
    CK(cudaGetLastError());
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, d_out, sizeof v, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *hash_out = (uint64_t)v;
    return VRG_OK;
}

// np.count_nonzero(dataArray) over the own planes, for the reference's second printed line (VRG:95): the volume is resident,
// counting it here is a 0.6 ms stream instead of half a second of host time at C3
int vrg_count_nonzero(vrg_handle *h, int64_t *count_out) {
    if (!h || !h->have_data || !count_out) return fail(VRG_ERR_ARG, "upload data first");
    CK(cudaSetDevice(h->cfg.device));
    const Params &p = h->p;
    const long long n = (long long)h->nz_own * p.plane_vox;
    unsigned long long *d_out = (unsigned long long *)(h->d_hcount);  // 16 bytes of scratch
    CK(cudaMemsetAsync(d_out, 0, sizeof(unsigned long long), h->stream));
    k_count_nonzero<<<h->grid, BLOCK, 0, h->stream>>>(p.data + (size_t)p.own_lo * p.plane_vox, n, d_out);
    h->launches++;
    CK(cudaGetLastError());
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, d_out, sizeof v, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *count_out = (int64_t)v;
    return VRG_OK;
}

// segmentedMap in the reference's dtype (VRG:45: np.full(shape, 0) is int64): expanded on the device, chunk by chunk
int vrg_download_segmented_map_i64(vrg_handle *h, int64_t *out) {
    NEED_INIT();
    if (!out) return fail(VRG_ERR_ARG, "null buffer");
    const size_t n = (size_t)h->nz_own * h->p.plane_vox;
    if (!h->d_labels) CK(big_alloc(h, (void **)&h->d_labels, n));
    int rc = labels_impl(h, h->d_labels, 1);
    if (rc != VRG_OK) return rc;
    const size_t chunk = std::min<size_t>(n, (size_t)32 << 20);  // 32 Mi voxels = 256 MiB of int64 per buffer, two buffers
    long long *stage[2] = {nullptr, nullptr};
    CK(cudaMalloc((void **)&stage[0], chunk * sizeof(long long)));
    cudaError_t e = cudaMalloc((void **)&stage[1], chunk * sizeof(long long));
    if (e != cudaSuccess) { cudaFree(stage[0]); return fail(VRG_ERR_NOMEM, "staging buffer: %s", cudaGetErrorString(e)); }
    int b = 0;
    for (size_t off = 0; off < n && e == cudaSuccess; off += chunk, b ^= 1) {
        const size_t m = std::min(chunk, n - off);
        k_expand_i64<<<h->grid, BLOCK, 0, h->stream>>>(h->d_labels + off, stage[b], (long long)m);
        h->launches++;
        // pageable destination: the copy returns once the chunk is staged, while the next chunk is being expanded
        e = cudaMemcpyAsync(out + off, stage[b], m * sizeof(long long), cudaMemcpyDeviceToHost, h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(stage[0]); cudaFree(stage[1]);
    if (e != cudaSuccess) return fail(VRG_ERR_CUDA, "segmented map download: %s", cudaGetErrorString(e));
    return VRG_OK;
}
int vrg_download_labels(vrg_handle *h, uint8_t *out) { return download_impl(h, out, 0); }
int vrg_download_segmented_map(vrg_handle *h, uint8_t *out) { return download_impl(h, out, 1); }

int vrg_download_segmented(vrg_handle *h, int64_t *coords, int64_t cap, int64_t *n_out) {
    NEED_INIT();
    if (!n_out) return fail(VRG_ERR_ARG, "null argument");
    const Params &p = h->p;
    const size_t words = (size_t)h->nz_own * p.plane_words;
    std::vector<uint32_t> plane(words);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(plane.data(), h->d_S + (size_t)p.own_lo * p.plane_words, words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    int64_t n = 0;
    for (int64_t zl = 0; zl < h->nz_own; ++zl)
        for (int64_t y = 0; y < p.Y; ++y) {
            const uint32_t *row = plane.data() + (size_t)zl * p.plane_words + (size_t)y * p.WP;
            for (int c = 0; c < p.XW; ++c) {
                uint32_t w = row[c];
                while (w) {
                    const int b = __builtin_ctz(w); w &= w - 1;
                    if (coords && n < cap) { coords[3 * n] = h->cfg.z_begin + zl; coords[3 * n + 1] = y; coords[3 * n + 2] = (int64_t)c * 32 + b; }
                    ++n;
                }
            }
        }
    *n_out = n;
    return VRG_OK;
}

template <int WHICH>
static cudaError_t launch_rows(vrg_handle *h, long long *counts, const long long *offs, int64_t *rows_dev, int64_t cap) {
    if (counts) k_seg_count<WHICH><<<h->grid, BLOCK, 0, h->stream>>>(h->p, counts);
    else k_seg_scatter<WHICH><<<h->grid, BLOCK, 0, h->stream>>>(h->p, offs, (long long *)rows_dev, (long long)cap,
                                                                  (long long)h->cfg.z_begin);
    return cudaGetLastError();
}
static cudaError_t launch_rows(vrg_handle *h, int which, long long *counts, const long long *offs, int64_t *rows_dev, int64_t cap) {
    if (which == 1) return launch_rows<1>(h, counts, offs, rows_dev, cap);
    if (which == 2) return launch_rows<2>(h, counts, offs, rows_dev, cap);
    return launch_rows<0>(h, counts, offs, rows_dev, cap);
}
// the rows of the segmented voxels (which = 0), the inner band (1) or the outer band (2), compacted on the device: popcounts per
// row segment, an exclusive scan (CUB), a scatter of the triples.  The count travels to the host (the one synchronisation); rows
// beyond `cap` are not written.
int vrg_band_rows_device(vrg_handle *h, int32_t which, int64_t *rows_dev, int64_t cap, int64_t *n_out) {
    NEED_INIT();
    if (!n_out || which < 0 || which > 2) return fail(VRG_ERR_ARG, "bad argument");
    if (rows_dev && (uintptr_t)rows_dev % sizeof(int64_t)) return fail(VRG_ERR_ARG, "rows buffer not aligned to 8 bytes");
    const Params &p = h->p;
    const long long nslots_ll = (long long)h->nz_own * p.Y * p.nseg;
    if (nslots_ll >= (1LL << 31) - 1) return fail(VRG_ERR_ARG, "too many rows for the device compaction");
    const int nslots = (int)nslots_ll;
    size_t tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const long long *)nullptr, (long long *)nullptr, nslots + 1, h->stream));
    const size_t cnt_bytes = ((size_t)(nslots + 1) * sizeof(long long) + 255) & ~(size_t)255;
    char *buf = nullptr;
    CK(big_alloc(h, (void **)&buf, 2 * cnt_bytes + tmp_bytes));
    long long *counts = (long long *)buf, *offs = (long long *)(buf + cnt_bytes);
    cudaError_t e = cudaMemsetAsync(counts + nslots, 0, sizeof(long long), h->stream);
    if (e == cudaSuccess) e = launch_rows(h, which, counts, nullptr, nullptr, 0);
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(buf + 2 * cnt_bytes, tmp_bytes, counts, offs, nslots + 1, h->stream);
    if (e == cudaSuccess && rows_dev && cap > 0) e = launch_rows(h, which, nullptr, offs, rows_dev, cap);
    long long n = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&n, offs + nslots, sizeof n, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFreeAsync(buf, h->stream);
    if (e != cudaSuccess) return fail(VRG_ERR_CUDA, "band rows on the device: %s", cudaGetErrorString(e));
    h->launches += 2 + (rows_dev && cap > 0);
    *n_out = n;
    return VRG_OK;
}
int vrg_segmented_device(vrg_handle *h, int64_t *rows_dev, int64_t cap, int64_t *n_out) {
    return vrg_band_rows_device(h, 0, rows_dev, cap, n_out);
}

// update()'s Parzen sum volumes of the current table (k_band_sums_dense), own planes, on the handle's stream (no synchronisation)
int vrg_band_sums_device(vrg_handle *h, double *pin_dev, double *pout_dev) {
    NEED_INIT();
    if (!pin_dev || !pout_dev) return fail(VRG_ERR_ARG, "null buffer");
    if ((uintptr_t)pin_dev % sizeof(double) || (uintptr_t)pout_dev % sizeof(double)) return fail(VRG_ERR_ARG, "sum buffers not aligned to 8 bytes");
    if (h->cfg.intensity_mode == VRG_INTENSITY_CONTINUOUS) return fail(VRG_ERR_ARG, "vrg_band_sums_device needs a level-table mode");
    if (h->p.lattice) k_band_sums_dense<true><<<h->grid, BLOCK, 0, h->stream>>>(h->p, pin_dev, pout_dev);
    else k_band_sums_dense<false><<<h->grid, BLOCK, 0, h->stream>>>(h->p, pin_dev, pout_dev);
    h->launches++;
    CK(cudaGetLastError());
    return VRG_OK;
}

int vrg_get_trace(vrg_handle *h, int64_t *rows, int64_t cap, int64_t *n_rows) {
    NEED_INIT();
    if (!n_rows) return fail(VRG_ERR_ARG, "null argument");
    CK(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, C_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const int64_t n = h->h_ctrl[C_TRACE_N];
    *n_rows = n;
    if (rows) CK(cudaMemcpy(rows, h->d_trace, (size_t)std::min(n, cap) * 3 * sizeof(long long), cudaMemcpyDeviceToHost));
    return VRG_OK;
}

int vrg_get_table(vrg_handle *h, double *pin, double *pout, int64_t cap) {
    if (!h || !h->have_levels) return fail(VRG_ERR_ARG, "no table yet");
    if (cap < h->p.L) return fail(VRG_ERR_ARG, "table buffer too small (%d levels)", h->p.L);
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    if (pin) CK(cudaMemcpy(pin, h->d_pin, h->p.L * sizeof(double), cudaMemcpyDeviceToHost));
    if (pout) CK(cudaMemcpy(pout, h->d_pout, h->p.L * sizeof(double), cudaMemcpyDeviceToHost));
    return VRG_OK;
}

// continuous mode: the normalised Parzen sums the last decision used, at every band voxel (own planes, C order)
int vrg_get_band_sums(vrg_handle *h, int64_t *vox_out, double *pin_out, double *pout_out, int64_t cap, int64_t *n_out) {
    NEED_INIT();
    if (h->cfg.intensity_mode != VRG_INTENSITY_CONTINUOUS || !n_out) return fail(VRG_ERR_ARG, "continuous mode only");
    const Params &p = h->p;
    CK(cudaStreamSynchronize(h->stream));
    const size_t words = (size_t)h->nz_own * p.plane_words, nvox = (size_t)h->nz_own * p.plane_vox;
    std::vector<uint32_t> B(words);
    std::vector<double> pin(nvox), pout(nvox);
    long long ex[ST_EXTRA];
    CK(cudaMemcpy(B.data(), h->cq.B + (size_t)p.own_lo * p.plane_words, words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pin.data(), h->cq.pin + (size_t)p.own_lo * p.plane_vox, nvox * sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pout.data(), h->cq.pout + (size_t)p.own_lo * p.plane_vox, nvox * sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ex, h->d_lstats, sizeof ex, cudaMemcpyDeviceToHost));
    int64_t n = 0;
    for (int64_t zl = 0; zl < h->nz_own; ++zl)
        for (int64_t y = 0; y < p.Y; ++y)
            for (int c = 0; c < p.XW; ++c) {
                uint32_t w = B[(size_t)zl * p.plane_words + (size_t)y * p.WP + c];
                while (w) {
                    const int b = __builtin_ctz(w); w &= w - 1;
                    const int64_t v = (zl * p.Y + y) * p.X + (int64_t)c * 32 + b;
                    if (n < cap) {
                        if (vox_out) vox_out[n] = v;
                        if (pin_out) pin_out[n] = pin[v] / (double)ex[ST_N_IN];
                        if (pout_out) pout_out[n] = pout[v] / (double)ex[ST_N_OUT];
                    }
                    ++n;
                }
            }
    *n_out = n;
    return VRG_OK;
}

int vrg_get_table_levels(vrg_handle *h, double *out, int64_t cap) {
    if (!h || !h->have_levels || !out) return fail(VRG_ERR_ARG, "no table yet");
    if (cap < h->p.L) return fail(VRG_ERR_ARG, "buffer too small");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpy(out, h->d_levels, h->p.L * sizeof(double), cudaMemcpyDeviceToHost));
    return VRG_OK;
}
