/* vrg_b200 -- C-ABI of the B200-native variational region growing (VRG) path.
 *
 * Drop-in boundary for ONE function of zjx1805/ArteryNetwork:
 *   Code/variationalRegionGrowing.py:10  variationalRegionGrowing(dataArray, valueMap, H, maxSegmentSize)
 *   Code/variationalRegionGrowing.py:124 update(...)            (init branch + band state machine)
 * The reference has no FFI of its own (it is pure Python); these entry points are
 * what a ctypes binding of that function binds (see INTEGRATION.md).  Plain C
 * types only; the caller owns every host buffer, the handle owns device memory.
 * One handle serves one host thread and one CUDA device.  Every call returns
 * VRG_OK or a negative vrg_status and never aborts; vrg_last_error() gives text.
 *
 * Volume layout: (Z, Y, X) with X fastest -- a C-ordered ndarray of shape
 * (Z, Y, X).  A handle owns planes [z_begin, z_end) of the global volume (the
 * whole volume on one GPU; one z-slab per GPU otherwise) plus VRG_HALO halo
 * planes on each side, which the caller fills from the neighbouring slabs.
 */
#ifndef VRG_B200_H
#define VRG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VRG_HALO 2 /* halo planes per side: band classification of own planes +-1 needs state at distance 2 */

typedef enum {
    VRG_OK = 0,
    VRG_ERR_CUDA = -1,       /* a CUDA call failed (text in vrg_last_error) */
    VRG_ERR_ARG = -2,        /* bad argument / call order */
    VRG_ERR_LEVELS = -3,     /* more than VRG_MAX_LEVELS distinct intensities (continuous data) */
    VRG_ERR_LABEL = -4,      /* initial valueMap holds a label above 4 (0 inside, 1 inner band, 2 outer band, 3 outside, 4 excluded) */
    VRG_ERR_EMPTY_SEED = -5, /* no voxel with label 0 (reference: IndexError at VRG:88) */
    VRG_ERR_NO_BAND = -6,    /* seed has no boundary (reference: IndexError at VRG:88) */
    VRG_ERR_NOMEM = -7,
    VRG_ERR_NONFINITE = -8   /* NaN/Inf intensity */
} vrg_status;

/* why the iteration stopped: the four exits of VRG:91-104,118-121 */
typedef enum {
    VRG_EXIT_RUNNING = -1,
    VRG_EXIT_CONVERGED = 0,   /* no voxel flipped                         VRG:91  */
    VRG_EXIT_MAX_TIME = 1,    /* wall-clock budget reached                VRG:97  */
    VRG_EXIT_MAX_SEGMENT = 2, /* len(segmented) >= maxSegmentSize         VRG:101 */
    VRG_EXIT_MAX_ITER = 3     /* iterMax = 200 updates applied            VRG:56,118 */
} vrg_exit;

/* how the per-iteration sweep reads intensities */
typedef enum {
    VRG_INTENSITY_F64_DENSE = 0, /* stream the fp64 volume: every voxel's decision, every iteration (reference dtype) */
    VRG_INTENSITY_F64_BAND = 1,  /* fp64 volume, but only 32-voxel words that hold a band voxel */
    VRG_INTENSITY_INDEX = 2,     /* uint16 level-index volume built once; band words only */
    VRG_INTENSITY_CONTINUOUS = 3 /* no level table: brute-force Parzen sums per band voxel (VRG:151-155,232-255), for data
                                    with more than VRG_MAX_LEVELS distinct intensities; single GPU, small volumes */
} vrg_intensity_mode;

#define VRG_MAX_LEVELS 65536

typedef struct {
    int64_t shape[3];       /* global volume (Z, Y, X) */
    int64_t z_begin, z_end; /* planes owned by this handle; 0, Z on a single GPU */
    int32_t device;         /* CUDA device ordinal */
    int32_t intensity_mode; /* vrg_intensity_mode */
    double H;               /* Parzen kernel precision, VRG:10,23 (default 2.25) */
    int64_t iter_max;       /* VRG:56 (200) */
    int64_t max_segment_size; /* VRG:10,101 (5000) */
    double max_seconds;     /* VRG:97 wall-clock exit (reference: 120 s); <= 0 disables it (parity runs) */
} vrg_config;

typedef struct vrg_handle vrg_handle;

typedef struct {
    int64_t iterations;  /* the number the reference prints, VRG:94 */
    int64_t exit_reason; /* vrg_exit */
    int64_t n_in;        /* #(valueMap in {0,1}) == len(segmented), VRG:49,113 */
    int64_t n_out;       /* #(valueMap in {2,3}), VRG:50,114 */
    int64_t n_excluded;  /* #(valueMap == 4) */
    int64_t n_levels;    /* size of the decision table */
    int64_t sweeps;      /* decide passes executed == iterations (voxel-updates = N * sweeps) */
    int64_t kernel_launches;
    /* Cumulative counts, over all applied updates, of the flip patterns on which the reference's sequential list
     * processing (VRG:165-233) is order-dependent -- the same sets oracle/vrg_oracle.py reports as quirk_potential.
     * q_cancelled is part of the order-free semantics (VRG:183-190 then :198); when the other three are zero the run lies
     * inside the domain where the reference's result does not depend on its list order, i.e. where bit-identity with it
     * is defined.  Non-zero: the labels returned are those of the order-free reading (DESIGN.md section 2). */
    int64_t q_cancelled;         /* outer-band voxels marked to enter whose segmented neighbours all left (Q1) */
    int64_t q_add_to_inside;     /* added voxels left without an unsegmented neighbour: stale label 1 in the reference (Q2/Q3) */
    int64_t q_remove_to_outside; /* removed voxels left without a segmented neighbour: stale label 2 in the reference (Q2/Q3) */
    int64_t q_cancel_repromoted; /* cancelled additions next to an executed addition: added by the reference if that
                                    neighbour comes first in its band list ("Q4") */
    int64_t redone_sweeps;       /* vrg_run starts each sweep on the decision table it has while the statistics of the previous
                                    update are still being exchanged; a sweep whose table turned out to have changed is repeated
                                    with the new one.  Repeats (and the one sweep in flight when the run ends) are not in `sweeps`. */
} vrg_result;

const char *vrg_last_error(void);
int vrg_version(void);

/* lifetime ---------------------------------------------------------------- */
int vrg_create(const vrg_config *cfg, vrg_handle **out);
int vrg_destroy(vrg_handle *h);
/* run every kernel on this CUDA stream (a cudaStream_t passed as void*); default: a stream the handle owns */
int vrg_set_stream(vrg_handle *h, void *cuda_stream);

/* inputs: replaces reading dataArray / valueMap, VRG:40-46 ------------------ */
/* Extended slab = planes [max(0, z_begin-VRG_HALO), min(Z, z_end+VRG_HALO)); the pointers address its first plane.
 * data: float64 intensities; value_map: uint8 labels (0 seed, 3 outside, 4 excluded).  A map an earlier run returned may
 * be fed back in: 1 (inner band) is read as segmented, 2 (outer band) as outside, and the bands are re-derived. */
int vrg_upload(vrg_handle *h, const double *data_host, const uint8_t *value_map_host);
int vrg_upload_device(vrg_handle *h, const double *data_dev, const uint8_t *value_map_dev);
int vrg_upload_value_map(vrg_handle *h, const uint8_t *value_map_host); /* new seeds, same data */
/* zero-copy: run on the caller's device-resident extended slab (read-only, must outlive the run) */
int vrg_attach_device(vrg_handle *h, const double *data_dev, const uint8_t *value_map_dev);
/* element types of a device-resident valueMap (vrg_attach_device_typed) and of the typed label outputs */
typedef enum {
    VRG_DTYPE_U8 = 0, VRG_DTYPE_I8 = 1, VRG_DTYPE_I16 = 2, VRG_DTYPE_I32 = 3, VRG_DTYPE_I64 = 4,
    VRG_DTYPE_F32 = 5, VRG_DTYPE_F64 = 6
} vrg_dtype;
/* zero-copy like vrg_attach_device, with the valueMap in any vrg_dtype: vrg_init reads it in that dtype (no conversion
 * pass); anything but an integral value in 0..4 (negative, fractional, NaN, above 4) makes vrg_init return VRG_ERR_LABEL.
 * The valueMap pointer must be aligned to its element size (any storage offset of a tensor view is). */
int vrg_attach_device_typed(vrg_handle *h, const double *data_dev, const void *value_map_dev, int32_t value_map_dtype);
/* the inputs of update() (VRG:124) on the device: data attached zero-copy like vrg_attach_device; the state built on the handle's
 * stream into the handle's own uint8 valueMap from the caller's segmentedMap (== 1: segmented) and valueMap (== 4: excluded),
 * each in its own vrg_dtype and read only by this call (every other value: outside).  Map pointers aligned to their element size. */
int vrg_attach_state_typed(vrg_handle *h, const double *data_dev, const void *seg_map_dev, int32_t seg_map_dtype,
                           const void *value_map_dev, int32_t value_map_dtype);

/* distinct intensity levels (the decision table's domain) ------------------- */
int vrg_scan_levels(vrg_handle *h, int64_t *n_levels);             /* local slab */
int vrg_get_levels(vrg_handle *h, double *levels_out, int64_t cap); /* sorted */
int vrg_set_levels(vrg_handle *h, const double *levels, int64_t n); /* union over all slabs (multi-GPU) */

/* init branch of update(), VRG:129-155: seeds, 4->3 around seeds, bands, region histograms */
int vrg_init(vrg_handle *h);

/* iteration loop, VRG:58-117.  vrg_run drives one GPU to an exit; the enqueue
 * calls are the same kernels for a host that interleaves the slab halo exchange
 * and the statistics all-reduce between them (multi-GPU), in this order:
 *   decide, cancel, [exchange FLIPS (+CANCELLED)], absorb, flip, [exchange EXCL], [all-reduce stats], advance */
int vrg_run(vrg_handle *h, vrg_result *res);
int vrg_enqueue_decide(vrg_handle *h);  /* decision table + the stencil sweep: flip flags (VRG:79-88) */
int vrg_enqueue_cancel(vrg_handle *h);  /* cancel rule, executed flips, region statistics (VRG:183-190,198,232-247) */
int vrg_enqueue_absorb(vrg_handle *h);  /* 4->3 absorption (VRG:167-168,177-179); no-op without label 4 */
int vrg_enqueue_flip(vrg_handle *h);    /* segmented ^= executed flips (VRG:173,201) */
int vrg_enqueue_advance(vrg_handle *h); /* exit tests + trace row (VRG:91-117) */
int vrg_poll(vrg_handle *h, vrg_result *res); /* synchronises the stream */
/* VRG_INTENSITY_F64_DENSE, as of the last vrg_poll / vrg_run / vrg_apply_flips: sweeps since vrg_init that evaluated every
 * voxel's decision from its intensity (the first sweep of a run, and each sweep behind a changed decision table or
 * caller-chosen flips); every other sweep takes the decisions from the bit-plane the last such sweep kept.  With the
 * environment switch VRG_NO_DCACHE=1 (read by vrg_create) every sweep is one.  0 in the other modes.  (Not a field of
 * vrg_result: callers allocate that struct, so its size stays as it is.) */
int vrg_dense_refresh_sweeps(vrg_handle *h, int64_t *n);
/* One update() call with caller-chosen flips, VRG:124,156-259 (flipedPoints given): coords = n rows of global (z, y, x).
 * Listed voxels that are in neither band are ignored; the band state machine (cancel rule, absorption, region statistics)
 * is applied once and the decision table of the NEW state is computed (vrg_get_table).  Whole-volume handles only. */
int vrg_apply_flips(vrg_handle *h, const int64_t *coords_host, int64_t n, vrg_result *res);
/* the same with the n rows in device memory (int64, 8-byte aligned): checked on the device first, one synchronisation for the
 * verdict; a row outside the volume returns VRG_ERR_ARG naming the first such row, and nothing has changed */
int vrg_apply_flips_device(vrg_handle *h, const int64_t *rows_dev, int64_t n, vrg_result *res);
/* decision table of the current state without a sweep (after vrg_init: the sums the reference's init branch stores) */
int vrg_enqueue_table(vrg_handle *h);

/* per-kernel device time (CUDA events on the launch stream) accumulated over launches that did real work:
 * index 0 = decide (the stencil sweep), 1 = what follows it (vrg_run: the fused tail kernel -- cancel rule, statistics and
 * halo exchange, exit tests, next decision table; host-driven iteration: the cancel kernel).  For roofline reporting. */
int vrg_profile(vrg_handle *h, int enable);
int vrg_get_profile(vrg_handle *h, double *ms_total /*[2]*/, int64_t *launches /*[2]*/);
/* phase timings inside the tail kernel while vrg_profile is on (device clock): us[0..6] = mean microseconds the grid's first
 * block spent in phase 1 (cancel rule, flips), the first device-wide barrier, phase 2 (in-order run: statistics exchange +
 * exit tests while the other blocks exchange halos; pipelined run: halo wait + unpack), the second barrier, phase 3 (decision
 * table / counters of the rows next to a halo plane), and for the pipelined run its halo push and its counters (the first two
 * parts of its phase 2); us[7..13] = the same for the grid's last block. */
int vrg_get_tail_profile(vrg_handle *h, double *us /*[14]*/, int64_t *launches);

/* continuous mode (VRG_INTENSITY_CONTINUOUS): Parzen kernel evaluations (fp64 exp, VRG:154,253-254) of the run so far, and the
 * rate of the same expression on an otherwise idle device -- its roofline is the exp rate, not HBM (SURVEY.md 8(f) N1) */
int vrg_get_exp_evals(vrg_handle *h, int64_t *evals);
int vrg_exp_peak(int device, double *evals_per_second);

/* device buffers a multi-GPU host exchanges between the enqueue calls ------- */
typedef enum {
    VRG_BUF_SEG = 0,          /* segmented bit-plane */
    VRG_BUF_EXCL = 1,         /* excluded (label 4) bit-plane */
    VRG_BUF_FLIPS = 2,        /* flip flags of the current iteration */
    VRG_BUF_CANCELLED = 3,    /* cancelled additions of the current iteration */
    VRG_BUF_LOCAL_STATS = 4,  /* int64[2*n_levels + 8]: this slab's histograms and counters */
    VRG_BUF_GLOBAL_STATS = 5, /* same layout, summed over slabs (aliases LOCAL on one GPU) */
    VRG_BUF_CTRL = 6
} vrg_buffer;
int vrg_buffer_info(vrg_handle *h, int which, void **dev_ptr, int64_t *bytes);
/* bit-plane geometry: words (uint32, 32 voxels along x) per row and rows*words per plane */
int vrg_plane_geometry(vrg_handle *h, int64_t *words_per_row, int64_t *words_per_plane, int64_t *n_planes_local);
int vrg_use_separate_global_stats(vrg_handle *h); /* multi-GPU: un-alias GLOBAL from LOCAL */
/* hash of the kernel parameter block: hosts that replay captured launches (CUDA graphs) re-capture when it changes */
int vrg_params_signature(vrg_handle *h, uint64_t *signature);

/* Peer-memory transport for z-slab runs on the GPUs of one box (one process per GPU): the halo planes and the
 * statistics all-reduce move by this library's own kernels over NVLink (CUDA IPC mappings), so vrg_init / vrg_run
 * drive a slab exactly like a single volume and every rank simply calls them at the same time.
 *   1. every rank: vrg_p2p_export -> 3 CUDA IPC handles (192 bytes);  2. gather all ranks' handles in rank order;
 *   3. every rank: vrg_p2p_connect;  4. host barrier;  5. vrg_init, vrg_run on every rank. */
#define VRG_P2P_HANDLE_BYTES 192
int vrg_p2p_export(vrg_handle *h, int world, void *handles_out /* VRG_P2P_HANDLE_BYTES */);
int vrg_p2p_connect(vrg_handle *h, int rank, int world, const void *all_handles /* world * VRG_P2P_HANDLE_BYTES */);
/* same transport for N handles that live in ONE process (one per device, peer access enabled here instead of CUDA IPC);
 * vrg_init / vrg_run must then be called on all of them at the same time, one host thread per handle */
int vrg_p2p_connect_local(vrg_handle **handles, int world);
int vrg_enqueue_p2p_halo(vrg_handle *h, int phase); /* 0: flips (+cancelled) after cancel, applied to the halo planes (replaces vrg_enqueue_flip); 1: excluded plane after absorb */
int vrg_enqueue_p2p_stats(vrg_handle *h);           /* statistics all-reduce + the advance step (replaces vrg_enqueue_advance) */

/* outputs: the return values of VRG:96 -------------------------------------- */
int vrg_download_labels(vrg_handle *h, uint8_t *value_map_out);   /* own planes, canonical labels 0..4 */
int vrg_download_segmented_map(vrg_handle *h, uint8_t *seg_out);  /* own planes, 0/1 */
int vrg_labels_device(vrg_handle *h, uint8_t *value_map_dev_out); /* same, into a device buffer */
/* own planes into a device buffer of that vrg_dtype: the canonical labels 0..4, or (segmented_only != 0) the 0/1 segmented map;
 * enqueued on the handle's stream, no synchronisation */
int vrg_labels_device_typed(vrg_handle *h, void *out_dev, int32_t dtype, int32_t segmented_only);
/* position-sensitive 64-bit hash of the own planes' canonical labels: sum over voxels of
 * splitmix64_finalizer((global linear voxel index << 3) | label) mod 2^64.  Additive over z-slabs: the per-rank hashes of a
 * multi-GPU run add up to the hash of the whole label volume (oracle/c_oracle.py computes the same number on the CPU). */
int vrg_labels_hash(vrg_handle *h, uint64_t *hash_out);
/* np.count_nonzero(dataArray) over the own planes, counted on the device (the reference's second printed line, VRG:95) */
int vrg_count_nonzero(vrg_handle *h, int64_t *count_out);
/* segmentedMap as the reference returns it (VRG:45-46: np.full(shape, 0) -> int64 0/1), own planes, straight into host memory */
int vrg_download_segmented_map_i64(vrg_handle *h, int64_t *seg_out);
/* segmented voxel coordinates (z,y,x) of own planes in C order; returns count via n (cap in rows) */
int vrg_download_segmented(vrg_handle *h, int64_t *coords_out, int64_t cap, int64_t *n);
/* the same rows compacted on the device into device memory (rows_dev may be NULL: count only); rows beyond cap are not
 * written; *n = their number.  Synchronises the handle's stream once, for the count. */
int vrg_segmented_device(vrg_handle *h, int64_t *rows_dev, int64_t cap, int64_t *n);
/* the same for which = 0 (segmented, == vrg_segmented_device), 1 (inner band, label 1) or 2 (outer band, label 2): rows (z,y,x)
 * of the own planes in C order, compacted on the device; one synchronisation, for the count */
int vrg_band_rows_device(vrg_handle *h, int32_t which, int64_t *rows_dev, int64_t cap, int64_t *n);
/* update()'s innerProb / outerProb (VRG:132-133,151-155) of the current decision table (after vrg_init + vrg_enqueue_table, or
 * vrg_apply_flips*): own planes, C order, float64 device buffers; pin * n_in and pout * n_out (vrg_get_table, one rounding each) at
 * every inner / outer band voxel, 0.0 elsewhere.  Enqueued on the handle's stream, no synchronisation.  Level-table modes only. */
int vrg_band_sums_device(vrg_handle *h, double *pin_dev, double *pout_dev);
int vrg_get_trace(vrg_handle *h, int64_t *rows_out, int64_t cap_rows, int64_t *n_rows); /* (n_flips,n_in,n_out) */
/* last decision table: in/out normalised Parzen sums per level (VRG:79-82), for parity checks */
int vrg_get_table(vrg_handle *h, double *pin_out, double *pout_out, int64_t cap);
int vrg_get_table_levels(vrg_handle *h, double *levels_out, int64_t cap); /* the table's level of each slot */
/* continuous mode: flat voxel index (own planes) and the normalised sums of the last decision at every band voxel */
int vrg_get_band_sums(vrg_handle *h, int64_t *vox_out, double *pin_out, double *pout_out, int64_t cap, int64_t *n);

/* ---- strict (list-order) mode, SURVEY.md section 8(f) N4 -------------------------------------------------------
 * The entry points above return the ORDER-FREE result: identical to the reference wherever the reference's own result
 * does not depend on the order of its band lists (vrg_result.q_* say when a run left that domain).  This second engine
 * reproduces the reference WITH its list order (Code/variationalRegionGrowing.py:156-259): flipped points processed in
 * allBnd order against the labels at their turn (VRG:163,169,198), band labels set without a look at the neighbours
 * (VRG:174,202), Parzen corrections selected by the labels after the call (VRG:232-233) and the drifting running sums
 * innerProb / outerProb that follow (VRG:236-247).  Outputs are the reference's: the valueMap with its stale band labels
 * and `segmented` in the reference's row order.  Single GPU, whole volume (< 2^31 voxels), <= VRG_MAX_LEVELS distinct
 * intensities, initial labels 0 / 3 / 4.  See arterynetwork_b200/csrc/vrg_strict.cu for how the list walk is parallel. */
typedef struct vrg_strict vrg_strict;
typedef struct {
    int64_t iterations;  /* the number the reference prints, VRG:94 */
    int64_t exit_reason; /* vrg_exit */
    int64_t n_in, n_out, n_excluded, n_levels;
    int64_t kernel_launches;
    int64_t skipped;     /* listed flips that were in neither band any more at their turn (VRG:169,198 both false) */
    int64_t dropped;     /* flipped voxels whose label after the call was not 1 or 2: left out of the corrections (Q3) */
    int64_t rounds;      /* wavefront rounds so far (the longest chains of order dependences, summed over iterations) */
} vrg_strict_result;
int vrg_strict_create(int device, const int64_t *shape /* Z, Y, X */, double H, int64_t iter_max, int64_t max_segment_size,
                      double max_seconds, vrg_strict **out);
int vrg_strict_destroy(vrg_strict *h);
/* dataArray + valueMap (host, whole volume) and the init branch of update(), VRG:40-50,129-155 */
int vrg_strict_init(vrg_strict *h, const double *data_host, const uint8_t *value_map_host);
int vrg_strict_step(vrg_strict *h, vrg_strict_result *res); /* one pass of the while loop, VRG:58-117 */
int vrg_strict_run(vrg_strict *h, vrg_strict_result *res);  /* to one of the exits */
/* the reference's valueMap as it stands (stale band labels included) and segmentedMap (0/1); either may be NULL */
int vrg_strict_download(vrg_strict *h, uint8_t *value_map_out, uint8_t *seg_map_out);
/* which = 0: the band in allBnd order (VRG:48,111) with innerProb/innerSize, outerProb/outerSize of every band voxel
 * (VRG:79-82; sums may be NULL); which = 1: the segmented voxels in the reference's row order (VRG:126,172,200).
 * vox_out: flat C-order voxel indices; cap in entries; *n = how many there are (VRG_ERR_ARG when cap is too small). */
int vrg_strict_list(vrg_strict *h, int which, int64_t *vox_out, double *pin_out, double *pout_out, int64_t cap, int64_t *n);
int vrg_strict_get_trace(vrg_strict *h, int64_t *rows_out, int64_t cap_rows, int64_t *n_rows); /* (n_flips,n_in,n_out) */
int vrg_strict_get_sums(vrg_strict *h, double *pin_out, double *pout_out); /* innerProb, outerProb, whole volume, unnormalised */

/* synthetic phantom generated on the device (bench configs that exceed host RAM) */
int vrg_phantom_device(int device, const int64_t *shape, int64_t z0, int64_t nz, const int64_t *segments,
                       int64_t n_segments, const int64_t *roots, int64_t n_roots, int64_t seed, int64_t quantum,
                       int64_t sigma_k, int64_t exclude_below_k, int use_exclude, double *data_dev,
                       uint8_t *value_map_dev);

/* ---- the array operations on either side of the path (SURVEY.md section 8(f), N2 / N3) -------------------------
 * Volumes are (Z, Y, X) C order; each axis <= 16384.  The *_device variants take device pointers and a cudaStream_t
 * (as void*, may be NULL) and synchronise that stream before returning. */

/* scipy.ndimage.distance_transform_edt(mask), default arguments -- Code/manualCorrectionGUI.py:248 (vessel radii from the
 * VRG output mask), Code/generateVesselVolume.py:183 (distance to the brain-mask boundary).  mask: uint8, non-zero =
 * foreground; dist: float64 Euclidean distance of every foreground voxel to the nearest zero voxel (0 on the background).
 * VRG_ERR_ARG when the mask has no zero voxel. */
int vrg_edt(int device, const uint8_t *mask_host, const int64_t *shape, double *dist_host);
int vrg_edt_device(int device, const uint8_t *mask_dev, const int64_t *shape, double *dist_dev, void *cuda_stream);
/* these entry points take their scratch memory from the device's stream-ordered pool and keep it cached between calls;
 * this hands it back to the driver */
int vrg_release_scratch(int device);

/* labelVolume, Code/generateVesselVolume.py:108-136 = skimage.measure.label(volume, return_num=True, connectivity=3):
 * 26-connected components of the non-zero voxels, numbered 1..K in raster order of each component's first voxel,
 * int32 labels (0 = background); sizes_out (optional, host) receives the voxel counts of components 1..min(K, cap).
 * The volume must hold fewer than 2^31 voxels. */
int vrg_label_components(int device, const uint8_t *binary_host, const int64_t *shape, int32_t *labels_host,
                         int64_t *n_components, int64_t *sizes_out, int64_t sizes_cap);
int vrg_label_components_device(int device, const uint8_t *binary_dev, const int64_t *shape, int32_t *labels_dev,
                                int64_t *n_components, int64_t *sizes_out, int64_t sizes_cap, void *cuda_stream);

/* vesselness volume -> vessel mask, Code/generateVesselVolume.py:183-200,216: with lo/hi the range of the vesselness
 * volume, voxels within edge_distance (10) of the brain-mask boundary and <= lo + edge_fraction (0.8) * (hi - lo) are
 * zeroed, then voxels <= lo + fraction (0.7) * (hi - lo); the non-zero rest is binarised and its 26-connected components
 * of at most min_size (150) voxels are removed.  vesselness: float64; brain_mask: uint8; mask_out: uint8 0/1.
 * info_out (optional): [0] voxels kept, [1] components kept.  thresholds_out (optional): the two cut-offs. */
int vrg_vessel_mask(int device, const double *vesselness_host, const uint8_t *brain_mask_host, const int64_t *shape,
                    double edge_distance, double edge_fraction, double fraction, int64_t min_size,
                    uint8_t *mask_out_host, int64_t *info_out, double *thresholds_out);
int vrg_vessel_mask_device(int device, const double *vesselness_dev, const uint8_t *brain_mask_dev, const int64_t *shape,
                           double edge_distance, double edge_fraction, double fraction, int64_t min_size,
                           uint8_t *mask_out_dev, int64_t *info_out, double *thresholds_out, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif
