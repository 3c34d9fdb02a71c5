/* include/klt_b200.h -- extensions of the KLT C API that only make sense for
 * the GPU library.  Nothing here is needed by the reference's drivers; they
 * exist for multi-GPU placement, parity testing and pipelined benches. */
#ifndef KLT_B200_H
#define KLT_B200_H

#include <stddef.h>
#include "klt.h"
#include "klt_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* val of a feature the forward-backward check rejected (KLTB200SetForwardBackward) */
#define KLT_B200_FB_INCONSISTENT  -6

/* val of a feature the global motion check rejected (KLTB200SetMotionCheck) */
#define KLT_B200_MOTION_OUTLIER  -7

/* CUDA device the context's work runs on.  Default: environment variable
 * KLT_B200_DEVICE, else the calling thread's current device.  Must be called
 * before the first Select/Track call on tc. */
void KLTB200SetDevice(KLT_TrackingContext tc, int device);

/* 1: tracking pyramids and the tracker use reference-order, separately rounded
 * multiply/add (bit-identical to the CPU reference); 0 (default, or env
 * KLT_B200_EXACT unset/0): fused multiply-add, within 1e-4 relative.
 * KLTSelectGoodFeatures always builds its images in exact mode, because its
 * ranking keys are truncated integers. */
void KLTB200SetExact(KLT_TrackingContext tc, int exact);
int  KLTB200GetExact(KLT_TrackingContext tc);

/* Forward-backward check of every tracking call on tc (KLTTrackFeatures, KLTTrackFeaturesDevice,
 * KLTB200Resident*, KLTTrackFeaturesSequence).  Each feature the translation tracker keeps is
 * tracked back from frame 2 into frame 1 with the same parameters; it stays KLT_TRACKED, at the
 * position it has with the check off, when the backward leg tracks and ends no more than max_error
 * pixels from where the feature started.  Otherwise it is lost as x = y = -1,
 * val = KLT_B200_FB_INCONSISTENT, before the affine consistency check, so that
 * KLTReplaceLostFeatures refills the slot.  max_error <= 0 switches the check off; INFINITY drops
 * only the features whose backward leg fails.  Default: environment variable KLT_B200_FB_MAX_ERROR
 * when tc's state is created, else off.  NaN ends in KLTError. */
void  KLTB200SetForwardBackward(KLT_TrackingContext tc, float max_error);
float KLTB200GetForwardBackward(KLT_TrackingContext tc);
/* Per feature of the last tracking call on tc (the last frame of a sequence or resident step), into
 * the non-NULL arrays: where the backward leg ended (xb, yb), its distance from the start position
 * (err) and its status (back_val); -1 in xb, yb and err when the backward leg lost the feature, and
 * xb = yb = err = -1, back_val = 1 for a feature the check did not run on.  Synchronises.  KLTError
 * when that call did not run the check or had a number of features other than n. */
void KLTB200ForwardBackwardResult(KLT_TrackingContext tc, int n, float *xb, float *yb, float *err,
                                  int *back_val);

/* Motion prior of every tracking call on tc (the calls above).  A feature with a guess g of its position
 * in frame 2 starts its pyramid descent from g instead of from zero motion, so that it can be found
 * farther away than the pyramid alone reaches; everything else, the status codes included, is the
 * reference's loop, and a guess equal to the feature's position changes nothing.  A guess whose window
 * leaves a level loses the feature as KLT_OOB.  Guesses come from:
 *   KLT_B200_PREDICT_VELOCITY: the feature's last displacement, for a feature whose val is KLT_TRACKED
 *     and which still sits where the last tracking call on tc left it (so not for features that were
 *     just selected or replaced, or that the caller moved).  The displacement is recorded after the
 *     forward-backward check and before the affine check by every call that runs with the prior
 *     (velocity mode, or explicit guesses in any mode), and forgotten by a call with neither and by
 *     a change of frame size.
 *   KLTB200SetGuesses: explicit guesses for the next KLTTrackFeatures, KLTTrackFeaturesDevice or
 *     KLTB200ResidentStep on tc, one per feature (NaN: none for that feature); they take precedence
 *     over the velocity.  That call ends in KLTError unless it has n features, and so does
 *     KLTTrackFeaturesSequence while guesses are set (through this call or klt_dev_set_guesses: they
 *     share one queue).  gx, gy are host arrays, or device arrays when on_device != 0; a device
 *     array must be complete when this is called.  Guesses for the next KLTB200ResidentStep may be
 *     set before the previous step has run; a third set waits until the device has finished the
 *     step that read the first.
 * With the forward-backward check, the backward leg of a feature that used g starts from the mirrored
 * prior xout - (g - x0).  Default mode: environment variable KLT_B200_PREDICT (none | velocity) when
 * tc's state is created, else none; any other value ends in KLTError. */
#define KLT_B200_PREDICT_NONE      0
#define KLT_B200_PREDICT_VELOCITY  1
void KLTB200SetPrediction(KLT_TrackingContext tc, int mode);
int  KLTB200GetPrediction(KLT_TrackingContext tc);
void KLTB200SetGuesses(KLT_TrackingContext tc, int n, const float *gx, const float *gy, int on_device);
/* Per feature of the last tracking call on tc (the last frame of a sequence or resident step), into the
 * non-NULL arrays: the guess it started from and its source (0 none, 1 velocity, 2 explicit);
 * gx = gy = -1 without one.  Synchronises.  KLTError when that call ran without prediction or had a
 * number of features other than n. */
void KLTB200PredictionResult(KLT_TrackingContext tc, int n, float *gx, float *gy, int *source);

/* Global motion check of every tracking call on tc (the calls above; each frame of
 * KLTTrackFeaturesSequence counts as one call).  After the tracker and the forward-backward check, and
 * before the affine check, a RANSAC homography is fitted on the device to the call's correspondences:
 * the features that entered with val >= 0 and are KLT_TRACKED, from where they started to where they
 * were tracked.  `hypotheses` fixed samples of 4 correspondences are solved and scored, the one with
 * the most inliers (reprojection distance <= max_error pixels) wins, and a least-squares fit over its
 * inliers refines it.  When the final model keeps at least 8 features, every other correspondence is
 * lost as x = y = -1, val = KLT_B200_MOTION_OUTLIER, so that KLTReplaceLostFeatures refills the slot
 * and the affine check releases its template; the features it keeps are exactly as with the check off.
 * With fewer, nothing is dropped.  The arithmetic is the same in both arithmetic modes.
 * max_error <= 0 switches the check off; hypotheses == 0 means 1024, else 1 .. 65536.  NaN or a
 * hypothesis count out of range ends in KLTError.  Default: environment variable
 * KLT_B200_MOTION_MAX_ERROR when tc's state is created, else off.  The check makes the tracker write
 * its results on the device, so the per-call API downloads them instead of receiving posted writes. */
typedef struct {
  float H[9];       /* row-major, maps frame-1 pixel coordinates to frame 2, H[8] = 1; NaN when !valid */
  int   valid;      /* 1: a model was found and applied                                            */
  int   tracked;    /* features that entered the check (val == KLT_TRACKED after the tracker / FB)  */
  int   inliers;    /* features kept by the final model                                             */
  int   hypothesis; /* index of the winning hypothesis, -1 when none                                */
} KLT_B200_MotionModel;
void  KLTB200SetMotionCheck(KLT_TrackingContext tc, float max_error, int hypotheses);
float KLTB200GetMotionCheck(KLT_TrackingContext tc, int *hypotheses);
/* Per feature of the last tracking call on tc (the last frame of a sequence or resident step): its
 * reprojection distance under the final model, -1 for a feature the check did not evaluate, +inf for
 * one the model maps behind the camera.  Synchronises.  KLTError when that call ran without the check
 * or had a number of features other than n. */
void  KLTB200MotionResult(KLT_TrackingContext tc, int n, float *err);
/* The models of the last `count` tracking calls on tc that ran the check, oldest first, with no
 * per-frame synchronisation in between (a sequence call yields one per frame).  The device keeps the
 * last 4096; a call without the check clears them.  Synchronises.  KLTError when count is larger
 * than recorded. */
void  KLTB200MotionModels(KLT_TrackingContext tc, int count, KLT_B200_MotionModel *out);

/* the device context behind tc (created on demand) */
klt_dev *KLTB200Device(KLT_TrackingContext tc);
/* slot (0/1) holding tc's previous-frame pyramids, -1 if none */
int KLTB200LastSlot(KLT_TrackingContext tc);

/* KLTTrackFeatures with the new frame already resident in HBM (row pitch in
 * bytes).  img1 is only used when no previous pyramid is held, as in the
 * reference (src/V1/trackFeatures.c:1285-1308); it may be NULL otherwise. */
void KLTTrackFeaturesDevice(KLT_TrackingContext tc, const KLT_PixelType *d_img1,
                            const KLT_PixelType *d_img2, size_t pitch,
                            int ncols, int nrows, KLT_FeatureList fl);

/* Resident-feature tracking for pipelined drivers: the feature arrays stay on
 * the device between frames, no host synchronisation per frame.
 *   KLTB200ResidentBegin  uploads fl and (if needed) builds the first pyramid
 *   KLTB200ResidentStep   builds pyramids of one more frame and tracks into it
 *   KLTB200ResidentEnd    downloads the features into fl (synchronises)
 * frames are host pointers when on_device == 0 (pinned memory recommended). */
void KLTB200ResidentBegin(KLT_TrackingContext tc, const KLT_PixelType *img1, int on_device,
                          size_t pitch, int ncols, int nrows, KLT_FeatureList fl);
void KLTB200ResidentStep(KLT_TrackingContext tc, const KLT_PixelType *img2, int on_device,
                         size_t pitch, int ncols, int nrows);
void KLTB200ResidentEnd(KLT_TrackingContext tc, KLT_FeatureList fl);

/* Batched driver API (SURVEY 8f N1): track fl through a whole sequence of HOST frames in one call.
 * Equivalent, result for result, to the reference's driver loop (src/V3/example3.c:54-76)
 *
 *     for (k = 1; k < nframes; k++) {
 *       KLTTrackFeatures(tc, frames[k-1], frames[k], ncols, nrows, fl);
 *       if (replace) KLTReplaceLostFeatures(tc, frames[k], ncols, nrows, fl);
 *       if (ft) KLTStoreFeatureList(fl, ft, first_frame + k);
 *     }
 *
 * with tc->sequentialMode = TRUE, but nothing waits for a frame's result before the next frame is
 * queued: frame k+1 crosses PCIe (two device staging buffers) while frame k's pyramids are built
 * and its features tracked, the features stay in HBM, every frame's x | y | val snapshot is copied
 * into pinned memory behind the tracker, and the host synchronises once at the end.  frames[0] is
 * only read when tc holds no previous pyramid (as img1 in KLTTrackFeatures) and may then not be
 * NULL.  ft may be NULL; column first_frame + k receives frame k (column first_frame is not
 * written: the caller stores the selection itself, as example3 does).  On return fl holds the
 * state after the last frame and tc is in sequential mode with the last frame's pyramids held.
 * tc->affineConsistencyCheck >= 0 is honoured (reference trackFeatures.c:1438-1497): the per-feature
 * affine state and templates live on the device during the call and are attached to fl at its end,
 * exactly as the loop above leaves them. */
void KLTTrackFeaturesSequence(KLT_TrackingContext tc, KLT_PixelType *const *frames, int nframes,
                              int ncols, int nrows, KLT_FeatureList fl, KLT_FeatureTable ft,
                              int first_frame, int replace);

#ifdef __cplusplus
}
#endif
#endif
