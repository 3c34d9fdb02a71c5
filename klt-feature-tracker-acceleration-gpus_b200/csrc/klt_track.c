/* klt_track.c -- KLTTrackFeatures on the GPU.
 *
 * Host orchestration of reference src/V1/trackFeatures.c:1234-1529
 * (KLTTrackFeatures): window repair (:1258-1278), reuse of the previous frame's
 * pyramids in sequentialMode (:1285-1294) or building them from img1
 * (:1295-1308), building the pyramids of img2 (:1311-1321), the feature loop
 * (:1343-1437, one warp per feature in csrc/klt_dev.cu), and the pyramid
 * hand-over (:1503-1519).  tc->lighting_insensitive (:125-220) runs on the generic
 * warp-per-feature kernel.  The affine-consistency check (:506-1224, :1438-1497) runs on the
 * device too (csrc/klt_affine.cuh); this file keeps the per-feature templates the reference
 * attaches to the feature list (aff_img*) in step with the device's copies.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "klt_internal.h"

#define DEVCALL(s, call)                                                     \
  do {                                                                       \
    if ((call) != 0) KLTError("(KLT/B200) %s", klt_dev_error((s)->dev));      \
  } while (0)

/* KLT_B200_TIMING=1: host-side phase times of the synchronous call, printed every 64 calls */
static double now_us(void)
{
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}
static int timing_on(void)
{
  static int on = -1;
  if (on < 0) { const char *e = getenv("KLT_B200_TIMING"); on = (e && atoi(e)) ? 1 : 0; }
  return on;
}

static void fill_track_params(KLT_TrackingContext tc, const klt_tc_state *s, klt_dev_track_params *p)
{
  p->window_width = tc->window_width;
  p->window_height = tc->window_height;
  p->step_factor = tc->step_factor;
  p->max_iterations = tc->max_iterations;
  p->min_determinant = tc->min_determinant;
  p->min_displacement = tc->min_displacement;
  p->max_residue = tc->max_residue;
  p->borderx = tc->borderx;
  p->bordery = tc->bordery;
  p->exact = s->exact;
  p->lighting_insensitive = tc->lighting_insensitive ? 1 : 0;
  p->fb_max_error = s->fb_max_error > 0.0f ? s->fb_max_error : 0.0f;
  p->predict = s->predict;
  p->motion_max_error = s->motion_max_error > 0.0f ? s->motion_max_error : 0.0f;
  p->motion_hypotheses = s->motion_hypotheses;
}

/* explicit guesses (KLTB200SetGuesses or klt_dev_set_guesses: one queue, on the device) are consumed
 * by the next tracking call, which must have as many features; checked before anything is queued */
static void check_guesses(klt_dev *dev, int n, const char *who)
{
  const int g = klt_dev_guesses_pending(dev);
  if (g >= 0 && g != n)
    KLTError("(%s) %d guesses were set (KLTB200SetGuesses) for a call on %d features", who, g, n);
}

static void check_supported(KLT_TrackingContext tc, int pipelined)
{
  if (tc->affineConsistencyCheck > 2)
    KLTError("(KLTTrackFeatures) affineConsistencyCheck = %d (must be -1, 0, 1 or 2)",
             tc->affineConsistencyCheck);
  if (tc->affineConsistencyCheck >= 0 && pipelined == 1)
    KLTError("(KLT/B200) the affine consistency check keeps per-feature templates in the caller's "
             "feature list: use KLTTrackFeatures or KLTTrackFeaturesSequence, not KLTB200Resident*");
}

/* ---- affine consistency check: host side (reference trackFeatures.c:1438-1497) ---------- */
/* _KLTCreateFloatImage (klt_util.c:34-54): header and pixels in one block, freed with free() */
static _KLT_FloatImage new_float_image(int ncols, int nrows)
{
  _KLT_FloatImage im = (_KLT_FloatImage)malloc(sizeof(_KLT_FloatImageRec) +
                                               (size_t)ncols * nrows * sizeof(float));
  if (im == NULL) KLTError("(_KLTCreateFloatImage) Out of memory");
  im->ncols = ncols;
  im->nrows = nrows;
  im->data = (float *)(im + 1);
  return im;
}

static void fill_affine_params(KLT_TrackingContext tc, klt_dev_affine_params *ap)
{
  ap->check = tc->affineConsistencyCheck;
  ap->window_width = tc->affine_window_width;
  ap->window_height = tc->affine_window_height;
  ap->max_iterations = tc->affine_max_iterations;
  ap->max_residue = tc->affine_max_residue;
  ap->min_displacement = tc->affine_min_displacement;
  ap->max_displacement_differ = tc->affine_max_displacement_differ;
}

/* fill the device's per-feature state from the list; upload templates the device does not mirror */
static void affine_stage(KLT_TrackingContext tc, klt_tc_state *s, KLT_FeatureList fl,
                         klt_dev_affine_state *st)
{
  const int n = fl->nFeatures, tw = tc->affine_window_width + 2, th = tc->affine_window_height + 2;
  int i;
  if (s->aff_list != (const void *)fl || s->aff_epoch != klt_aff_epoch || s->aff_shadow_n != n) {
    free(s->aff_shadow);
    s->aff_shadow = (void **)calloc((size_t)n, sizeof(void *));
    if (s->aff_shadow == NULL) KLTError("(KLTTrackFeatures) Out of memory");
    s->aff_shadow_n = n;
    s->aff_list = fl;
    s->aff_epoch = klt_aff_epoch;
  }
  for (i = 0; i < n; i++) {
    KLT_Feature f = fl->feature[i];
    st[i].has = f->aff_img != NULL;
    st[i].aff_x = f->aff_x; st[i].aff_y = f->aff_y;
    st[i].Axx = f->aff_Axx; st[i].Ayx = f->aff_Ayx; st[i].Axy = f->aff_Axy; st[i].Ayy = f->aff_Ayy;
    st[i].flags = 0;
    if (f->aff_img != NULL && s->aff_shadow[i] != (void *)f->aff_img) {
      if (f->aff_img_gradx == NULL || f->aff_img_grady == NULL ||
          f->aff_img->ncols != tw || f->aff_img->nrows != th)
        KLTError("(KLTTrackFeatures) feature %d carries a %d by %d affine template, expected %d by %d",
                 i, f->aff_img->ncols, f->aff_img->nrows, tw, th);
      DEVCALL(s, klt_dev_affine_put_template(s->dev, i, f->aff_img->data, f->aff_img_gradx->data,
                                             f->aff_img_grady->data));
      s->aff_shadow[i] = (void *)f->aff_img;
    }
    if (f->aff_img == NULL) s->aff_shadow[i] = NULL;
  }
}

/* after the call: the aff_* members of every feature that was tracked, new templates fetched */
static void affine_collect(KLT_TrackingContext tc, klt_tc_state *s, KLT_FeatureList fl,
                           const klt_dev_affine_state *st, const unsigned char *was_live)
{
  const int n = fl->nFeatures, tw = tc->affine_window_width + 2, th = tc->affine_window_height + 2;
  const size_t tsz = (size_t)tw * th;
  float *all = NULL;
  int i, created = 0;
  for (i = 0; i < n; i++) created += was_live[i] && st[i].flags == 1;
  if (created > 8) {              /* one bulk copy instead of three small ones per feature */
    all = (float *)malloc((size_t)n * 3 * tsz * sizeof(float));
    if (all == NULL) KLTError("(KLTTrackFeatures) Out of memory");
    DEVCALL(s, klt_dev_affine_get_templates(s->dev, n, all));
  }
  for (i = 0; i < n; i++) {
    KLT_Feature f = fl->feature[i];
    if (!was_live[i]) continue;
    f->aff_x = st[i].aff_x; f->aff_y = st[i].aff_y;
    f->aff_Axx = st[i].Axx; f->aff_Ayx = st[i].Ayx; f->aff_Axy = st[i].Axy; f->aff_Ayy = st[i].Ayy;
    if (st[i].flags == 1) {       /* :1446-1457 template saved after the first successful track */
      f->aff_img = new_float_image(tw, th);
      f->aff_img_gradx = new_float_image(tw, th);
      f->aff_img_grady = new_float_image(tw, th);
      if (all != NULL) {
        memcpy(f->aff_img->data, all + (size_t)i * 3 * tsz, tsz * sizeof(float));
        memcpy(f->aff_img_gradx->data, all + (size_t)i * 3 * tsz + tsz, tsz * sizeof(float));
        memcpy(f->aff_img_grady->data, all + (size_t)i * 3 * tsz + 2 * tsz, tsz * sizeof(float));
      } else {
        DEVCALL(s, klt_dev_affine_get_template(s->dev, i, f->aff_img->data, f->aff_img_gradx->data,
                                               f->aff_img_grady->data));
      }
      s->aff_shadow[i] = (void *)f->aff_img;
    } else if (f->aff_img == NULL) {
      s->aff_shadow[i] = NULL;    /* released: freed by the caller's loop when val went negative */
    }
  }
  free(all);
}

/* after KLTTrackFeaturesSequence: the device held the per-feature state for the whole call; what it
 * ends with is what the per-call loop would have left in the list -- the aff_* members, a template for
 * every feature that holds one (cut once per feature life, so the copy is the template whenever it was
 * cut), none for the features that lost theirs */
static void affine_collect_resident(KLT_TrackingContext tc, klt_tc_state *s, KLT_FeatureList fl)
{
  const int n = fl->nFeatures, tw = tc->affine_window_width + 2, th = tc->affine_window_height + 2;
  const size_t tsz = (size_t)tw * th;
  klt_dev_affine_state *st = NULL;
  float *all;
  int i;
  DEVCALL(s, klt_dev_affine_fetch_states(s->dev, n, &st));
  all = (float *)malloc((size_t)n * 3 * tsz * sizeof(float));
  if (all == NULL) KLTError("(KLTTrackFeaturesSequence) Out of memory");
  DEVCALL(s, klt_dev_affine_get_templates(s->dev, n, all));
  for (i = 0; i < n; i++) {
    KLT_Feature f = fl->feature[i];
    if (f->val > 0) {           /* refilled after the last check: a new feature the device has not met yet */
      st[i].has = 0; st[i].aff_x = st[i].aff_y = -1.0f;
      st[i].Axx = st[i].Ayy = 1.0f; st[i].Ayx = st[i].Axy = 0.0f;
    }
    f->aff_x = st[i].aff_x; f->aff_y = st[i].aff_y;
    f->aff_Axx = st[i].Axx; f->aff_Ayx = st[i].Ayx; f->aff_Axy = st[i].Axy; f->aff_Ayy = st[i].Ayy;
    if (st[i].has) {
      if (f->aff_img == NULL) {
        f->aff_img = new_float_image(tw, th);
        f->aff_img_gradx = new_float_image(tw, th);
        f->aff_img_grady = new_float_image(tw, th);
      }
      memcpy(f->aff_img->data, all + (size_t)i * 3 * tsz, tsz * sizeof(float));
      memcpy(f->aff_img_gradx->data, all + (size_t)i * 3 * tsz + tsz, tsz * sizeof(float));
      memcpy(f->aff_img_grady->data, all + (size_t)i * 3 * tsz + 2 * tsz, tsz * sizeof(float));
      s->aff_shadow[i] = (void *)f->aff_img;
    } else {
      free(f->aff_img); free(f->aff_img_gradx); free(f->aff_img_grady);
      f->aff_img = f->aff_img_gradx = f->aff_img_grady = NULL;
      s->aff_shadow[i] = NULL;
    }
  }
  free(all);
}

/* Returns the slot holding frame 1's pyramids, building them if necessary. */
static int prepare_previous(KLT_TrackingContext tc, klt_tc_state *s, const KLT_PixelType *img1,
                            int on_device, size_t pitch, int ncols, int nrows)
{
  klt_dev *dev = klt_state_device(s);
  int gw = 0, gh = 0, gl = 0, gs = 0;

  if (tc->sequentialMode && tc->pyramid_last != NULL && s->last_slot >= 0 &&
      klt_dev_slot_valid(dev, s->last_slot)) {
    klt_dev_geometry(dev, &gw, &gh, &gl, &gs);
    if (gw != ncols || gh != nrows)
      KLTError("(KLTTrackFeatures) Size of incoming image (%d by %d) "
               "is different from size of previous image (%d by %d)\n",
               ncols, nrows, gw, gh);
    if (gl == tc->nPyramidLevels && (gl == 1 || gs == tc->subsampling))
      return s->last_slot;
    /* pyramid parameters changed between frames: fall through and rebuild */
  }
  if (img1 == NULL)
    KLTError("(KLTTrackFeatures) no previous pyramid is held and img1 is NULL");
  {
    klt_dev_build_desc q;
    klt_fill_build_desc(tc, ncols, nrows, tc->nPyramidLevels, 1, s->exact, &q);
    DEVCALL(s, klt_dev_build(dev, 0, img1, on_device, pitch, &q));
  }
  return 0;
}

static void hand_over(KLT_TrackingContext tc, klt_tc_state *s, int slot_cur)
{
  if (tc->sequentialMode) {
    s->last_slot = slot_cur;
    tc->pyramid_last = tc->pyramid_last_gradx = tc->pyramid_last_grady = (void *)s;
  } else {
    s->last_slot = -1;
    klt_dev_invalidate(s->dev, -1);
    tc->pyramid_last = tc->pyramid_last_gradx = tc->pyramid_last_grady = NULL;
  }
}

static void track_common(KLT_TrackingContext tc, const KLT_PixelType *img1,
                         const KLT_PixelType *img2, int on_device, size_t pitch,
                         int ncols, int nrows, KLT_FeatureList fl)
{
  klt_tc_state *s = klt_state_get(tc);
  klt_dev *dev;
  klt_dev_build_desc q;
  klt_dev_track_params tp;
  int slot_prev, slot_cur, n = fl->nFeatures, i, records;
  const int affine = tc->affineConsistencyCheck >= 0 && n > 0;
  klt_dev_affine_params ap;
  klt_dev_affine_state *ast = NULL;
  unsigned char *was_live = NULL;
  float *x = NULL, *y = NULL;
  int *v = NULL;

  if (KLT_verbose >= 1) {
    fprintf(stderr, "(KLT) Tracking %d features in a %d by %d image...  ",
            KLTCountRemainingFeatures(fl), ncols, nrows);
    fflush(stderr);
  }
  klt_fix_window(tc, "KLTTrackFeatures", 1);
  check_supported(tc, 0);
  dev = klt_state_device(s);
  check_guesses(dev, n, "KLTTrackFeatures");

  /* Everything below is queued on the context stream without waiting: feature upload,
   * frame upload, pyramid kernels, tracker, result download; one synchronisation at the end. */
  const int timing = timing_on();
  static __thread double acc[5]; static __thread int calls;     /* (KLT_B200_TIMING: per calling thread) */
  double t0 = timing ? now_us() : 0, t1 = 0, t2 = 0, t3 = 0;
  /* The frame upload is the long pole.  With a pinned feature list nothing has to be packed:
   * queue the one-copy mirror of the records, then queue the frame and the pyramid kernels.  An ordinary list is
   * packed into the staging area first (a few microseconds) for the same order on the copy stream. */
  slot_prev = prepare_previous(tc, s, img1, on_device, pitch, ncols, nrows);
  slot_cur = (slot_prev + 1) % KLT_DEV_SLOTS;
  /* (the global motion check rewrites the tracker's answers on the device: no record mode) */
  records = n > 0 && !affine && !(s->motion_max_error > 0.0f) && klt_list_is_pinned(fl) && fl->feature[n - 1] == fl->feature[0] + (n - 1);
  if (records) {
    DEVCALL(s, klt_dev_features_commit_records(dev, n, fl->feature[0], sizeof(KLT_FeatureRec)));
  } else {
    DEVCALL(s, klt_dev_features_staging(dev, n, &x, &y, &v));
    klt_list_to_arrays(fl, x, y, v);
    DEVCALL(s, klt_dev_features_commit(dev, n));
  }
  fill_track_params(tc, s, &tp);
  if (affine) {
    fill_affine_params(tc, &ap);
    DEVCALL(s, klt_dev_affine_begin(dev, n, &ap, &ast));
    affine_stage(tc, s, fl, ast);
    was_live = (unsigned char *)malloc((size_t)n);
    if (was_live == NULL) KLTError("(KLTTrackFeatures) Out of memory");
    for (i = 0; i < n; i++) was_live[i] = fl->feature[i]->val >= 0;
  }
  klt_fill_build_desc(tc, ncols, nrows, tc->nPyramidLevels, 1, s->exact, &q);
  DEVCALL(s, klt_dev_build(dev, slot_cur, img2, on_device, pitch, &q));
  if (timing) t1 = now_us();

  fill_track_params(tc, s, &tp);
  DEVCALL(s, klt_dev_track_resident(dev, slot_prev, slot_cur, &tp));
  if (affine) DEVCALL(s, klt_dev_affine_check(dev, slot_prev, slot_cur, &tp, &ap));
  if (timing) t2 = now_us();
  DEVCALL(s, klt_dev_features_fetch(dev, n));
  if (timing) t3 = now_us();
  /* (record mode: nothing to unpack.  A lost feature's affine templates are freed here as in the
   * reference, trackFeatures.c:1387-1392 and :1480-1489.) */
  for (i = 0; !records && i < n; i++) {
    KLT_Feature f = fl->feature[i];
    if (f->val < 0) continue;                 /* lost features are not touched (:1346) */
    f->x = x[i];
    f->y = y[i];
    f->val = v[i];
    if (v[i] < 0 && (f->aff_img || f->aff_img_gradx || f->aff_img_grady)) {
      free(f->aff_img); free(f->aff_img_gradx); free(f->aff_img_grady);   /* (:1387-1392) */
      f->aff_img = f->aff_img_gradx = f->aff_img_grady = NULL;
    }
  }

  if (affine) {
    affine_collect(tc, s, fl, ast, was_live);
    free(was_live);
  }
  hand_over(tc, s, slot_cur);
  if (timing) {
    const double t4 = now_us();
    acc[0] += t1 - t0; acc[1] += t2 - t1; acc[2] += t3 - t2; acc[3] += t4 - t3; acc[4] += t4 - t0;
    if (++calls % 64 == 0) {
      fprintf(stderr, "(KLT/B200 timing, us/call over 64 calls) build enqueue %.1f  pack+commit+track enqueue %.1f  wait %.1f  unpack %.1f  total %.1f\n",
              acc[0] / 64, acc[1] / 64, acc[2] / 64, acc[3] / 64, acc[4] / 64);
      acc[0] = acc[1] = acc[2] = acc[3] = acc[4] = 0;
    }
  }

  if (KLT_verbose >= 1) {
    fprintf(stderr, "\n\t%d features successfully tracked.\n", KLTCountRemainingFeatures(fl));
    fflush(stderr);
  }
}

void KLTTrackFeatures(KLT_TrackingContext tc, KLT_PixelType *img1, KLT_PixelType *img2,
                      int ncols, int nrows, KLT_FeatureList fl)
{
  track_common(tc, img1, img2, 0, (size_t)ncols, ncols, nrows, fl);
}

void KLTTrackFeaturesDevice(KLT_TrackingContext tc, const KLT_PixelType *d_img1,
                            const KLT_PixelType *d_img2, size_t pitch,
                            int ncols, int nrows, KLT_FeatureList fl)
{
  track_common(tc, d_img1, d_img2, 1, pitch, ncols, nrows, fl);
}

/* ---- resident-feature pipeline (no host sync per frame) ----------------------- */
void KLTB200ResidentBegin(KLT_TrackingContext tc, const KLT_PixelType *img1, int on_device,
                          size_t pitch, int ncols, int nrows, KLT_FeatureList fl)
{
  klt_tc_state *s = klt_state_get(tc);
  const int n = fl->nFeatures;
  float *x = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
  float *y = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
  int *v = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  int slot;
  if (!x || !y || !v) KLTError("(KLTB200ResidentBegin) Out of memory");
  klt_fix_window(tc, "KLTTrackFeatures", 1);
  check_supported(tc, s->in_sequence ? 2 : 1);
  if (!tc->sequentialMode)
    KLTError("(KLTB200ResidentBegin) the resident pipeline needs tc->sequentialMode = TRUE");
  {
    /* opt-in: measured on B200, the tracker and the level-0 kernel are both bound by the
     * LSU / L1 data pipe, so running them concurrently stretches both (DESIGN.md 4) */
    const char *e = getenv("KLT_B200_OVERLAP");
    DEVCALL(s, klt_dev_set_overlap(klt_state_device(s), (e != NULL && atoi(e) != 0) ? 1 : 0));
  }
  slot = prepare_previous(tc, s, img1, on_device, pitch ? pitch : (size_t)ncols, ncols, nrows);
  hand_over(tc, s, slot);
  klt_list_to_arrays(fl, x, y, v);
  DEVCALL(s, klt_dev_features_upload(s->dev, n, x, y, v));
  free(x); free(y); free(v);
}

void KLTB200ResidentStep(KLT_TrackingContext tc, const KLT_PixelType *img2, int on_device,
                         size_t pitch, int ncols, int nrows)
{
  klt_tc_state *s = klt_state_get(tc);
  klt_dev_build_desc q;
  klt_dev_track_params tp;
  int slot_prev, slot_cur;
  if (tc->pyramid_last == NULL || s->last_slot < 0)
    KLTError("(KLTB200ResidentStep) call KLTB200ResidentBegin first");
  slot_prev = s->last_slot;
  slot_cur = (slot_prev + 1) % KLT_DEV_SLOTS;      /* third slot: build(k+1) may overlap track(k) */
  klt_fill_build_desc(tc, ncols, nrows, tc->nPyramidLevels, 1, s->exact, &q);
  DEVCALL(s, klt_dev_build(s->dev, slot_cur, img2, on_device, pitch ? pitch : (size_t)ncols, &q));
  fill_track_params(tc, s, &tp);
  DEVCALL(s, klt_dev_track_resident(s->dev, slot_prev, slot_cur, &tp));
  hand_over(tc, s, slot_cur);
}

void KLTB200ResidentEnd(KLT_TrackingContext tc, KLT_FeatureList fl)
{
  klt_tc_state *s = klt_state_get(tc);
  const int n = fl->nFeatures;
  float *x = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
  float *y = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
  int *v = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  int i;
  if (!x || !y || !v) KLTError("(KLTB200ResidentEnd) Out of memory");
  DEVCALL(s, klt_dev_features_download(klt_state_device(s), n, x, y, v));
  DEVCALL(s, klt_dev_set_overlap(s->dev, 0));       /* back to the single in-order stream */
  for (i = 0; i < n; i++) {
    fl->feature[i]->x = x[i];
    fl->feature[i]->y = y[i];
    fl->feature[i]->val = v[i];
  }
  free(x); free(y); free(v);
}

/* ---- batched driver API: a whole sequence of host frames in one call ------------ */
/* Replaces the reference's serial driver loop (src/V3/example3.c:54-76: KLTTrackFeatures,
 * optional KLTReplaceLostFeatures, KLTStoreFeatureList per frame) with one pipelined call; the
 * per-frame work is the resident pipeline above, so every frame's result is bit-identical to
 * the per-call API's. */
#define SEQ_DEPTH 16          /* frames queued ahead of the one the host is storing */

/* frame k's snapshot -> table column and the affine fields of slots refilled at that frame */
static void seq_consume(klt_tc_state *s, int slot, KLT_FeatureList fl, KLT_FeatureTable ft,
                        int column, int replace)
{
  const float *x, *y;
  const int *v;
  const int n = fl->nFeatures;
  int i;
  DEVCALL(s, klt_dev_snapshot_wait(s->dev, slot, &x, &y, &v));
  if (ft != NULL && n > 0) {
    /* a table made by KLTCreateFeatureTable keeps its records in one [feature][frame] block
     * (klt.c:210-236): address them directly and prefetch ahead -- every cell of a column sits
     * on a different page, so chasing the two pointer levels per cell would be three cache
     * misses per feature */
    KLT_Feature base = ft->feature[0][0];
    const size_t stride = (size_t)ft->nFrames;
    const int regular = ft->feature[n - 1][column] == base + (size_t)(n - 1) * stride + column;
    for (i = 0; i < n; i++) {
      KLT_Feature f = regular ? base + (size_t)i * stride + column : ft->feature[i][column];
      if (regular && i + 16 < n) __builtin_prefetch(base + (size_t)(i + 16) * stride + column, 1);
      f->x = x[i]; f->y = y[i]; f->val = v[i];
    }
  }
  if (replace)                  /* a slot refilled at this frame starts a new feature (:514-541) */
    for (i = 0; i < n; i++)
      if (v[i] > 0) {
        KLT_Feature f = fl->feature[i];
        free(f->aff_img); free(f->aff_img_gradx); free(f->aff_img_grady);
        f->aff_img = f->aff_img_gradx = f->aff_img_grady = NULL;
        f->aff_x = f->aff_y = -1.0f;
        f->aff_Axx = f->aff_Ayy = 1.0f;
        f->aff_Ayx = f->aff_Axy = 0.0f;
      }
}

void KLTTrackFeaturesSequence(KLT_TrackingContext tc, KLT_PixelType *const *frames, int nframes,
                              int ncols, int nrows, KLT_FeatureList fl, KLT_FeatureTable ft,
                              int first_frame, int replace)
{
  klt_tc_state *s = klt_state_get(tc);
  const int n = fl->nFeatures;
  const int snaps = n > 0 && (ft != NULL || replace);
  klt_dev_select_params sp;
  const int affine = tc->affineConsistencyCheck >= 0 && n > 0;
  klt_dev_affine_params ap;
  klt_dev_affine_state *ast = NULL;
  klt_dev_track_params tp;
  int k, stored = 1;            /* next frame whose snapshot is to be consumed */

  if (frames == NULL || nframes < 1)
    KLTError("(KLTTrackFeaturesSequence) needs at least one frame");
  if (s->dev != NULL && klt_dev_guesses_pending(s->dev) >= 0)
    KLTError("(KLTTrackFeaturesSequence) guesses are set (KLTB200SetGuesses): the sequence call predicts "
             "by velocity only (KLTB200SetPrediction)");
  if (ft != NULL) {
    if (fl->nFeatures != ft->nFeatures)
      KLTError("(KLTTrackFeaturesSequence) FeatureList and FeatureTable must have the same number of features");
    if (first_frame < 0 || first_frame + nframes - 1 >= ft->nFrames)
      KLTError("(KLTTrackFeaturesSequence) frames %d .. %d do not fit a table of %d frames",
               first_frame, first_frame + nframes - 1, ft->nFrames);
  }
  for (k = 1; k < nframes; k++)
    if (frames[k] == NULL) KLTError("(KLTTrackFeaturesSequence) frame %d is NULL", k);
  if (KLT_verbose >= 1) {
    fprintf(stderr, "(KLT) Tracking %d features through %d frames of %d by %d...  ",
            KLTCountRemainingFeatures(fl), nframes - 1, ncols, nrows);
    fflush(stderr);
  }
  tc->sequentialMode = TRUE;
  if (replace) klt_fix_window(tc, "KLTSelectGoodFeatures", 1);
  s->in_sequence = 1;
  KLTB200ResidentBegin(tc, frames[0], 0, (size_t)ncols, ncols, nrows, fl);
  s->in_sequence = 0;
  if (replace) klt_fill_select_params(tc, 1, &sp);
  if (affine) {                 /* the per-feature state goes up once and stays on the device */
    fill_affine_params(tc, &ap);
    fill_track_params(tc, s, &tp);
    DEVCALL(s, klt_dev_affine_begin(s->dev, n, &ap, &ast));
    affine_stage(tc, s, fl, ast);
    DEVCALL(s, klt_dev_affine_upload_states(s->dev, n));
  }
  if (snaps && nframes > 1) DEVCALL(s, klt_dev_snapshot_ring(s->dev, SEQ_DEPTH));
  for (k = 1; k < nframes; k++) {
    if (snaps && k - stored >= SEQ_DEPTH) {      /* ring full: store the oldest frame while the */
      seq_consume(s, (stored - 1) % SEQ_DEPTH, fl, ft, first_frame + stored, replace);   /* GPU runs */
      stored++;
    }
    if (affine) DEVCALL(s, klt_dev_affine_keep_positions(s->dev));   /* where the templates are cut (:1446-1457) */
    KLTB200ResidentStep(tc, frames[k], 0, (size_t)ncols, ncols, nrows);
    if (affine)
      DEVCALL(s, klt_dev_affine_check_resident(s->dev, (s->last_slot + KLT_DEV_SLOTS - 1) % KLT_DEV_SLOTS,
                                               s->last_slot, &tp, &ap));
    if (replace && n > 0) {     /* REPLACING_SOME on the level-0 gradients just built (:342-348), */
      int sel_slot = s->last_slot;               /* in exact arithmetic (integer ranking keys)         */
      DEVCALL(s, klt_dev_exact_level0(s->dev, s->last_slot, &sel_slot));
      DEVCALL(s, klt_dev_select_resident(s->dev, sel_slot, &sp));
    }
    if (snaps) DEVCALL(s, klt_dev_snapshot_push(s->dev, (k - 1) % SEQ_DEPTH));
  }
  for (; snaps && stored < nframes; stored++)
    seq_consume(s, (stored - 1) % SEQ_DEPTH, fl, ft, first_frame + stored, replace);
  KLTB200ResidentEnd(tc, fl);
  if (affine) affine_collect_resident(tc, s, fl);
  if (KLT_verbose >= 1) {
    fprintf(stderr, "\n\t%d features alive after the last frame.\n", KLTCountRemainingFeatures(fl));
    fflush(stderr);
  }
}
