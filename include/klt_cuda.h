/* include/klt_cuda.h -- thin C-ABI between the plain-C KLT host library and
 * the hand-written sm_100a CUDA kernels (csrc/klt_dev.cu).
 *
 * extern "C", POD arguments only, every entry point returns 0 on success or a
 * non-zero code with a message retrievable through klt_dev_error(); the C side
 * (csrc/klt_track.c, csrc/klt_select.c) funnels failures into KLTError(), the
 * reference's error convention (reference src/V1/error.c:23-33).
 *
 * Each entry point names the reference interface it replaces.  A binding from
 * another host language (cgo, JNI, ctypes ...) needs exactly these symbols;
 * see INTEGRATION.md.
 *
 * Data layout on the device: every float image is row-major with a row pitch
 * rounded up to 32 floats (128 B); one "pyramid set" holds, for each level l,
 * the smoothed image L_l and its gradients gx_l, gy_l.  A context owns two
 * sets (slots 0..2): the previous frame, the current frame and -- in the overlapped
 * resident pipeline -- the frame being built while the tracker still reads the other two.
 */
#ifndef KLT_CUDA_H
#define KLT_CUDA_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLT_DEV_MAX_TAPS   71   /* reference src/V1/convolve.c:16 MAX_KERNEL_WIDTH */
#define KLT_DEV_MAX_LEVELS 12
#define KLT_DEV_SLOTS      3    /* pyramid sets per context: previous, current, being built */

typedef struct klt_dev klt_dev;   /* opaque device context: stream, buffers */

/* One separable kernel pair for a given sigma, generated on the host exactly
 * as reference src/V1/convolve.c:60-114 (_computeKernels) does. */
typedef struct {
  int   gauss_width;                 /* odd */
  int   deriv_width;                 /* odd */
  float gauss[KLT_DEV_MAX_TAPS];     /* normalised Gaussian            */
  float deriv[KLT_DEV_MAX_TAPS];     /* normalised derivative of Gauss */
} klt_dev_taps;

/* What to build from one u8 frame.
 * replaces: _KLTToFloatImage + _KLTComputeSmoothedImage + _KLTComputePyramid +
 * per-level _KLTComputeGradients as sequenced in reference
 * src/V1/trackFeatures.c:1309-1321 (and selectGoodFeatures.c:354-363 when
 * nlevels_built == 1). */
typedef struct {
  int ncols, nrows;            /* frame size                                    */
  int nlevels;                 /* pyramid levels of the context geometry        */
  int subsampling;             /* 2,4,8,16,32                                   */
  int nlevels_built;           /* 1 for selection, nlevels for tracking         */
  int smooth;                  /* 0: level 0 = (float) pixels, no pre-smoothing */
  int exact;                   /* 1: reference-order, non-fused mul/add (bit-exact
                                  against the CPU reference); 0: FMA (default)  */
  klt_dev_taps smooth_taps;    /* sigma = smooth_sigma_fact * max(window)       */
  klt_dev_taps pyramid_taps;   /* sigma = subsampling * pyramid_sigma_fact      */
  klt_dev_taps grad_taps;      /* sigma = grad_sigma                            */
} klt_dev_build_desc;

/* replaces the scalar arguments of _trackFeature / KLTTrackFeatures
 * (reference src/V1/trackFeatures.c:381-399, :1364-1376, :1396). */
typedef struct {
  int   window_width, window_height;
  float step_factor;
  int   max_iterations;
  float min_determinant;
  float min_displacement;
  float max_residue;
  int   borderx, bordery;
  int   exact;
  int   lighting_insensitive;  /* tc->lighting_insensitive: gain / bias normalised windows
                                  (reference src/V1/trackFeatures.c:125-220, :433-437, :466-468) */
  float fb_max_error;          /* > 0: forward-backward check in the same launch (klt_dev_fb_results);
                                  0: off */
  int   predict;               /* motion prior: 0 none, 1 constant velocity (klt_dev_prediction_results) */
} klt_dev_track_params;

/* replaces the scalar arguments of _KLTSelectGoodFeatures /
 * _enforceMinimumDistance (reference src/V1/selectGoodFeatures.c:297-453). */
typedef struct {
  int window_width, window_height;
  int borderx, bordery;
  int nSkippedPixels;
  int mindist;
  int min_eigenvalue;
  int overwrite_all;           /* 1 = SELECTING_ALL, 0 = REPLACING_SOME */
} klt_dev_select_params;

/* ---- lifetime ---------------------------------------------------------- */
int  klt_dev_count(void);                                /* visible CUDA devices, 0 if none */
int  klt_dev_create(int device, klt_dev **out);          /* device < 0: current device      */
void klt_dev_destroy(klt_dev *d);
const char *klt_dev_error(const klt_dev *d);             /* text of the last failure        */
const char *klt_dev_create_error(void);                  /* text when klt_dev_create failed */
int  klt_dev_device(const klt_dev *d);
void *klt_dev_stream(const klt_dev *d);                  /* the cudaStream_t all work runs on */

/* ---- pyramids ---------------------------------------------------------- */
/* Build slot's pyramids from a frame.  img_is_device == 0: img is a host
 * pointer (pageable or pinned), copied H2D on the context stream;
 * != 0: img is a device pointer with row pitch img_pitch bytes.
 * Asynchronous with respect to the host unless img is pageable. */
int klt_dev_build(klt_dev *d, int slot, const unsigned char *img,
                  int img_is_device, size_t img_pitch,
                  const klt_dev_build_desc *desc);
/* Selection keys are truncated integers: a replacement that reuses the level-0 gradients of a
 * slot built in fma arithmetic could rank differently from the reference
 * (src/V1/selectGoodFeatures.c:342-348, :421).  Returns in *slot_out a slot whose level 0 is in
 * exact arithmetic: `slot` itself when it was built that way, else level 0 is rebuilt (exact,
 * same taps) from the u8 frame still on the device into the slot the next frame overwrites.
 * A caller-owned device frame must still be valid. */
int klt_dev_exact_level0(klt_dev *d, int slot, int *slot_out);
int klt_dev_slot_valid(const klt_dev *d, int slot);      /* 1 if slot holds a full pyramid set */
void klt_dev_invalidate(klt_dev *d, int slot);           /* slot < 0: both */
int klt_dev_geometry(const klt_dev *d, int *ncols, int *nrows, int *nlevels, int *subsampling);

/* ---- tracking ---------------------------------------------------------- */
/* replaces the feature loop of KLTTrackFeatures (reference
 * src/V1/trackFeatures.c:1343-1437): x,y,val are host arrays of n features,
 * updated in place; features with val < 0 are left untouched.  Synchronous. */
int klt_dev_track(klt_dev *d, int slot_prev, int slot_cur,
                  const klt_dev_track_params *p, int n,
                  float *x, float *y, int *val);

/* Device-resident variant for pipelined drivers: the feature arrays stay in
 * HBM between calls; nothing is copied and the host is not synchronised. */
int klt_dev_features_upload(klt_dev *d, int n, const float *x, const float *y, const int *val);
int klt_dev_track_resident(klt_dev *d, int slot_prev, int slot_cur,
                           const klt_dev_track_params *p);
int klt_dev_features_download(klt_dev *d, int n, float *x, float *y, int *val);   /* synchronises */
/* Forward-backward check (fb_max_error > 0): after the forward leg of a feature the same warp tracks
 * the result back from frame 2 into frame 1; the feature is kept when that leg ends KLT_TRACKED within
 * fb_max_error pixels of the start, else it is recorded as (-1, -1, KLT_B200_FB_INCONSISTENT).
 * klt_dev_fb_results copies the per-feature records of the last klt_dev_track* call into the non-NULL
 * arrays: where the backward leg ended (xb, yb; -1 when it lost the feature), the distance from the
 * start (err; -1 when the backward leg lost it) and its status (back_val); xb = yb = err = -1,
 * back_val = 1 for a feature the check did not run on.  Fails unless that call ran the check on
 * exactly n features.  Synchronises. */
int klt_dev_fb_results(klt_dev *d, int n, float *xb, float *yb, float *err, int *back_val);
/* Motion prior: a feature with a guess g of its frame-2 position starts its pyramid descent from g
 * (scaled through the levels as its own position is) instead of from zero motion; everything else is
 * the reference loop.  A feature uses, in this order, its explicit guess (klt_dev_set_guesses; both
 * coordinates finite, NaN = none), or with predict = 1 its constant-velocity guess x0 + (dx, dy): the
 * device keeps one record {px, py, dx, dy} per feature index, written by every call with the prior
 * as {xout, yout, xout - x0, yout - y0} for a feature that ends KLT_TRACKED (after the
 * forward-backward check, before the affine check) and invalid for every other one; a feature uses
 * it when its input val is KLT_TRACKED and it still starts at (px, py).  Records are invalid when
 * allocated, after a call without the prior and after a change of frame geometry.  With the
 * forward-backward check, the backward leg of a feature that used g starts from xout - (g - x0).
 * klt_dev_set_guesses queues n guesses for the next klt_dev_track* call, which consumes them and
 * fails unless it has n features: host arrays are staged and copied H2D, device arrays (on_device != 0)
 * D2D on the library's copy stream, so they must be complete when this is called.  Two sets of
 * guesses can be in flight: queuing a third waits until the tracking call that read the first has
 * finished on the device, so a pipelined driver may queue guesses for step k + 1 before step k ran.
 * klt_dev_prediction_results copies the per-feature records of the last klt_dev_track* call into the
 * non-NULL arrays: the guess (gx, gy) and its source (0 none, 1 velocity, 2 explicit); -1, -1, 0
 * without a guess.  Fails unless that call ran with prediction on exactly n features.  Synchronises. */
int klt_dev_set_guesses(klt_dev *d, int n, const float *gx, const float *gy, int on_device);
/* the number of guesses queued for the next klt_dev_track* call, -1 when none are */
int klt_dev_guesses_pending(const klt_dev *d);
int klt_dev_prediction_results(klt_dev *d, int n, float *gx, float *gy, int *source);
/* Ring of pinned snapshots of the resident features for pipelined drivers
 * (KLTTrackFeaturesSequence): klt_dev_snapshot_ring sizes it (depth <= 64 slots),
 * klt_dev_snapshot_push queues a copy of the current x | y | val into a slot behind the work
 * queued so far (no synchronisation), klt_dev_snapshot_wait blocks until that copy has landed and
 * returns pointers into the slot (valid until the slot is pushed again). */
int klt_dev_features_capacity(const klt_dev *d);
int klt_dev_snapshot_ring(klt_dev *d, int depth);
int klt_dev_snapshot_push(klt_dev *d, int slot);
int klt_dev_snapshot_wait(klt_dev *d, int slot, const float **x, const float **y, const int **val);
/* 7x7 fma tracking runs on track7w_kernel (one warp per feature; default) or, with
 * klt_dev_disable_track7w(d, 1) / env KLT_B200_TRACK7W=0, on track_fast_kernel<7> (8 lanes per feature) */
void klt_dev_disable_track7w(klt_dev *d, int on);
/* zero-copy variant for the C host layer: pack the feature list straight into the
 * context's pinned staging area, commit it (async H2D), and after the work fetch the
 * results back into the same area (D2H + synchronise). */
int klt_dev_features_staging(klt_dev *d, int n, float **x, float **y, int **val);
int klt_dev_features_commit(klt_dev *d, int n);
int klt_dev_features_fetch(klt_dev *d, int n);
/* record mode, for feature lists that live in pinned host memory (klt_dev_host_alloc: what
 * KLTCreateFeatureList uses when a CUDA device is present): first_record points at an array of n
 * records of stride_bytes each with x | y | val (float, float, int) in their first 12 bytes -- the
 * layout of KLT_FeatureRec.  One H2D copy mirrors them, the next tracker reads the mirror and
 * writes x | y | val of every live feature straight into the caller's records (posted PCIe
 * writes); klt_dev_features_fetch then only synchronises.  No pack / unpack on the host. */
int klt_dev_features_commit_records(klt_dev *d, int n, void *first_record, size_t stride_bytes);
void *klt_dev_host_alloc(size_t bytes);     /* portable pinned host memory; NULL without a device */
void klt_dev_host_free(void *p);

/* ---- affine consistency check ------------------------------------------ */
/* replaces the tc->affineConsistencyCheck >= 0 branch of KLTTrackFeatures and its _am_* helpers
 * (reference src/V1/trackFeatures.c:506-1224, :1438-1497).  Exact reference arithmetic always. */
typedef struct {
  int   check;                    /* tc->affineConsistencyCheck: 0 translation, 1 similarity, 2 affine */
  int   window_width, window_height;       /* tc->affine_window_* */
  int   max_iterations;           /* tc->affine_max_iterations */
  float max_residue;              /* tc->affine_max_residue */
  float min_displacement;         /* tc->affine_min_displacement */
  float max_displacement_differ;  /* tc->affine_max_displacement_differ */
} klt_dev_affine_params;
typedef struct {                  /* the aff_* members of KLT_FeatureRec (klt.h:97-105) */
  int   has;                      /* aff_img != NULL: the device holds this feature's template */
  float aff_x, aff_y, Axx, Ayx, Axy, Ayy;
  int   flags;                    /* out: 1 = template created by this call, 2 = template released */
} klt_dev_affine_state;
/* One call: features committed through the staging area -> klt_dev_affine_begin (hands out the pinned
 * state array of n records for the host to fill) -> klt_dev_affine_put_template for every feature
 * whose template the device does not hold yet -> klt_dev_track_resident -> klt_dev_affine_check
 * -> klt_dev_features_fetch (synchronises) -> read the state array, fetch created templates. */
int klt_dev_affine_begin(klt_dev *d, int n, const klt_dev_affine_params *ap, klt_dev_affine_state **staging);
int klt_dev_affine_put_template(klt_dev *d, int i, const float *img, const float *gx, const float *gy);
int klt_dev_affine_check(klt_dev *d, int slot_prev, int slot_cur, const klt_dev_track_params *tp,
                         const klt_dev_affine_params *ap);
/* The check inside the resident / sequence pipeline (KLTTrackFeaturesSequence): the per-feature state
 * stays on the device between frames.  Set up with klt_dev_affine_begin + the staging array +
 * klt_dev_affine_put_template as above, then klt_dev_affine_upload_states ONCE; per frame
 * klt_dev_affine_keep_positions (before the tracker), klt_dev_track_resident,
 * klt_dev_affine_check_resident; klt_dev_affine_fetch_states (synchronises) hands the states back in
 * the staging array at the end; templates through klt_dev_affine_get_template(s). */
int klt_dev_affine_upload_states(klt_dev *d, int n);
int klt_dev_affine_keep_positions(klt_dev *d);
int klt_dev_affine_check_resident(klt_dev *d, int slot_prev, int slot_cur, const klt_dev_track_params *tp,
                                  const klt_dev_affine_params *ap);
int klt_dev_affine_fetch_states(klt_dev *d, int n, klt_dev_affine_state **staging);
int klt_dev_affine_get_template(klt_dev *d, int i, float *img, float *gx, float *gy);
int klt_dev_affine_get_templates(klt_dev *d, int n, float *all);

/* ---- selection --------------------------------------------------------- */
/* replaces the eigenvalue loop, _sortPointList and _enforceMinimumDistance of
 * _KLTSelectGoodFeatures (reference src/V1/selectGoodFeatures.c:373-446) on
 * the level-0 gradients of `slot`.  Ties in the ranking are resolved in raster
 * order (== the reference built with -DKLT_USE_QSORT on glibc).  Synchronous. */
int klt_dev_select(klt_dev *d, int slot, const klt_dev_select_params *p,
                   int n, float *x, float *y, int *val);
/* the same on the device-resident feature arrays (klt_dev_features_upload ...): no copies, no
 * synchronisation; with p->overwrite_all == 0 this is KLTReplaceLostFeatures */
int klt_dev_select_resident(klt_dev *d, int slot, const klt_dev_select_params *p);

/* ---- introspection (parity tests, debugging) --------------------------- */
/* which: 0 image, 1 gradx, 2 grady.  out: dense ncols*nrows floats of that level. */
int klt_dev_read_level(klt_dev *d, int slot, int which, int level, float *out);
int klt_dev_level_dims(const klt_dev *d, int level, int *ncols, int *nrows);
/* int min-eigenvalue of every candidate pixel in raster order (the pointlist
 * `val` column of reference selectGoodFeatures.c:396-423); returns the count
 * through *npoints; out may be NULL to query the count only. */
int klt_dev_eigen_map(klt_dev *d, int slot, const klt_dev_select_params *p,
                      int *out, int *npoints);
int klt_dev_sync(klt_dev *d);
/* 1: the tracker and the feature copies run on a second stream, ordered against the
 * pyramid builds with events, so build(k+1) overlaps track(k) (KLTB200Resident*);
 * 0 (default): one stream, strictly in order.  Drains both streams. */
int klt_dev_set_overlap(klt_dev *d, int on);
int klt_dev_slots(void);
/* number of kernels this context has launched so far */
unsigned long long klt_dev_launch_count(const klt_dev *d);
/* 1 if the last klt_dev_build used the fused tiled kernels, 0 if it took the
 * generic (any radius / any subsampling) kernels */
int klt_dev_last_build_path(const klt_dev *d);
/* force the generic kernels (cross-check of the tiled ones); default 0 */
void klt_dev_force_generic(klt_dev *d, int on);
/* keep the tiled kernels but not the fused TMA level-0 kernel (cross-check); default 0 */
void klt_dev_disable_fused(klt_dev *d, int on);
/* Debug aid (compute-sanitizer's stand-in): guard mode (env KLT_B200_GUARD=1 or klt_dev_set_guard
 * before the next build) puts a 4 KB canary band in front of every plane of the pyramid arena and
 * behind the last one; klt_dev_check_guards synchronises and counts the canary words a kernel has
 * damaged (0 = no store left its plane) and names the first damaged band. */
void klt_dev_set_guard(klt_dev *d, int on);
int klt_dev_check_guards(klt_dev *d, long long *damaged_words, int *first_band);
/* (for the guard test) device address of a plane (which: 0 image, 1 gradx, 2 grady), NULL if not
 * allocated; a synchronous raw host-to-device write */
void *klt_dev_plane_address(const klt_dev *d, int slot, int which, int level);
int klt_dev_poke(klt_dev *d, void *device_dst, const void *host_src, size_t bytes);
/* which level-0 kernel the fused path uses, process wide (env KLT_B200_L0_TILE at first use):
 * 0: l0_fused_kernel with 64x64 tiles, 1 (default): 64x48 tiles, 2: l0_march_kernel (column strips
 * marched down by three-warp teams; same results, measured slower -- kept as a cross-check) */
void klt_dev_set_l0_kernel(int variant);
int klt_dev_l0_kernel(void);
/* number of pyramid levels the last klt_dev_build produced with the fused TMA kernels
 * (level 0: l0_fused_kernel, coarser levels: level_fused_kernel); 0 if none */
int klt_dev_last_build_fused(const klt_dev *d);
/* Host frames are uploaded in bands of `rows` image rows (rounded up to 64) on a copy stream and
 * the fused kernels are launched over the tile rows each band completes, so the PCIe transfer
 * hides the image pipeline; rows == 0: one copy, then the kernels; rows < 0 (default, or env
 * KLT_B200_BAND_ROWS): automatic -- frames of >= 4 MB in two bands (60 % / 40 %), smaller ones in
 * one copy.  klt_dev_last_build_bands: copies the last klt_dev_build issued (0 for a
 * device-resident frame). */
void klt_dev_set_band_rows(klt_dev *d, int rows);
int klt_dev_last_build_bands(const klt_dev *d);
/* Pageable frame buffers: a driver that reuses its malloc'ed images for the whole run (reference
 * src/V3/example3.c:45-46,75) hands the same pageable pointers in again and again.  The second
 * time a buffer of >= 1 MB (same address, same size) arrives it is page-locked in place
 * (cudaHostRegister) and from then on copied by DMA directly, as a pinned frame is; up to 32
 * buffers per context.  The registrations are dropped by klt_dev_forget_host_frames -- called by
 * KLTStopSequentialMode and KLTFreeTrackingContext -- and by klt_dev_destroy.  A registered
 * buffer must not be freed while the registration lives (call KLTStopSequentialMode first, or
 * switch the cache off: env KLT_B200_REGISTER_FRAMES=0 / klt_dev_set_register_frames(d, 0)). */
int klt_dev_forget_host_frames(klt_dev *d);
int klt_dev_registered_host_frames(const klt_dev *d);
void klt_dev_set_register_frames(klt_dev *d, int on);
/* Pageable host frames of >= 1 MB are copied into a pinned staging buffer by n host threads
 * (OpenMP; default 4, env KLT_B200_STAGE_THREADS; 0 = leave the staging to cudaMemcpyAsync), ~1 MB
 * chunk by chunk ahead of the DMA.  klt_dev_last_build_staged: 1 if the last build did that. */
void klt_dev_set_stage_threads(klt_dev *d, int n);
int klt_dev_last_build_staged(const klt_dev *d);
/* device time between the two calls, measured with CUDA events recorded on the
 * context's own stream (the stream the kernels run on) */
int klt_dev_timer_start(klt_dev *d);
int klt_dev_timer_stop(klt_dev *d, float *ms);
/* per-kernel device time: between begin and end every kernel launch of this
 * context is bracketed by CUDA events on the context stream and accumulated by
 * kernel class; klt_dev_profile_get returns the class name (NULL past the end) */
int klt_dev_profile_begin(klt_dev *d);
int klt_dev_profile_end(klt_dev *d);
int klt_dev_profile_kernels(void);
const char *klt_dev_profile_get(const klt_dev *d, int kid, unsigned long long *launches, double *total_ms);
/* timeline of the same profiling session: record i (launch order as folded) = class name, start
 * and end in ms since klt_dev_profile_begin; also covers the frame / feature copies ("copy_h2d",
 * "copy_d2h"), which are timed but never counted as kernel launches.  NULL past the end. */
int klt_dev_trace_count(const klt_dev *d);
const char *klt_dev_trace_get(const klt_dev *d, int i, float *t0_ms, float *t1_ms);
/* number of features that entered klt_dev_track* with val >= 0 since the last
 * reset, counted on the device (the metric's numerator for resident pipelines) */
int klt_dev_live_total(klt_dev *d, unsigned long long *out, int reset);

#ifdef __cplusplus
}
#endif

#endif
