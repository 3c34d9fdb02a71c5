/* klt_context.c -- tracking context, feature containers, parameter derivation.
 *
 * Host C, behaviour of reference src/V1/klt.c: defaults (:20-44), constructors
 * (:90-236), KLTChangeTCPyramid (:288-343), KLTUpdateTCBorder (:362-431),
 * destructors (:441-483), KLTStopSequentialMode (:490-500),
 * KLTCountRemainingFeatures (:507-518), KLTSetVerbosity (:524-528).
 * The pyramid/border arithmetic must match the reference to the integer.
 *
 * New here: each tracking context owns a device context (stream + HBM buffers)
 * kept in a side table keyed by the tc pointer.  tc->pyramid_last* stay NULL
 * until a previous frame's pyramids are really held on the device, exactly the
 * condition the reference tests (trackFeatures.c:1285).
 */
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "klt_internal.h"

int KLT_verbose = 1;

/* ---- side table tc -> device state ---------------------------------------- */
static pthread_mutex_t g_lock = PTHREAD_MUTEX_INITIALIZER;
static klt_tc_state *g_states = NULL;

/* The hot calls look their context up once per call: a per-thread one-entry cache in front of the
 * list keeps the process-wide lock off that path (a driver thread works on one tc at a time; 64
 * contexts on 4 threads in the config-5 runner).  g_epoch moves whenever a state is dropped, which is
 * the only event that can turn a cached pointer stale. */
static unsigned long g_epoch = 1;
static __thread KLT_TrackingContext t_tc;
static __thread klt_tc_state *t_state;
static __thread unsigned long t_epoch;

klt_tc_state *klt_state_find(KLT_TrackingContext tc)
{
  klt_tc_state *s;
  if (t_state != NULL && t_tc == tc && t_epoch == __atomic_load_n(&g_epoch, __ATOMIC_ACQUIRE)) return t_state;
  pthread_mutex_lock(&g_lock);
  for (s = g_states; s != NULL && s->tc != tc; s = s->next) ;
  t_tc = tc; t_state = s; t_epoch = g_epoch;
  pthread_mutex_unlock(&g_lock);
  return s;
}

klt_tc_state *klt_state_get(KLT_TrackingContext tc)
{
  klt_tc_state *s = klt_state_find(tc);
  const char *e;
  if (s) return s;
  s = (klt_tc_state *)calloc(1, sizeof(*s));
  if (!s) KLTError("(klt_state_get) Out of memory");
  s->tc = tc;
  s->device = -1;
  s->last_slot = -1;
  e = getenv("KLT_B200_EXACT");
  s->exact = (e && atoi(e) != 0) ? 1 : 0;
  e = getenv("KLT_B200_FB_MAX_ERROR");
  s->fb_max_error = e ? strtof(e, NULL) : 0.0f;
  if (isnan(s->fb_max_error)) {
    free(s);
    KLTError("(KLT/B200) KLT_B200_FB_MAX_ERROR = %s is not a number of pixels", e);
  }
  e = getenv("KLT_B200_PREDICT");
  s->predict = KLT_B200_PREDICT_NONE;
  if (e && strcmp(e, "velocity") == 0) s->predict = KLT_B200_PREDICT_VELOCITY;
  else if (e && strcmp(e, "none") != 0) {
    free(s);
    KLTError("(KLT/B200) KLT_B200_PREDICT = %s (must be none or velocity)", e);
  }
  pthread_mutex_lock(&g_lock);
  s->next = g_states;
  g_states = s;
  t_tc = tc; t_state = s; t_epoch = g_epoch;
  pthread_mutex_unlock(&g_lock);
  return s;
}

void klt_state_drop(KLT_TrackingContext tc)
{
  klt_tc_state **pp, *s = NULL;
  pthread_mutex_lock(&g_lock);
  for (pp = &g_states; *pp; pp = &(*pp)->next)
    if ((*pp)->tc == tc) { s = *pp; *pp = s->next; break; }
  __atomic_add_fetch(&g_epoch, 1, __ATOMIC_RELEASE);     /* every thread's cached entry is void now */
  pthread_mutex_unlock(&g_lock);
  if (s) {
    if (s->dev) klt_dev_destroy(s->dev);
    free(s->aff_shadow);
    free(s);
  }
}

klt_dev *klt_state_device(klt_tc_state *s)
{
  if (!s->dev) {
    int device = s->device;
    if (device < 0) {
      const char *e = getenv("KLT_B200_DEVICE");
      if (e) device = atoi(e);
    }
    if (klt_dev_create(device, &s->dev) != 0)
      KLTError("(KLT/B200) cannot open a CUDA device: %s", klt_dev_create_error());
  }
  return s->dev;
}

void KLTB200SetDevice(KLT_TrackingContext tc, int device)
{
  klt_tc_state *s = klt_state_get(tc);
  if (s->dev && klt_dev_device(s->dev) != device)
    KLTError("(KLTB200SetDevice) context already runs on device %d", klt_dev_device(s->dev));
  s->device = device;
}

void KLTB200SetExact(KLT_TrackingContext tc, int exact)
{
  klt_tc_state *s = klt_state_get(tc);
  if (s->exact != (exact != 0)) {
    /* pyramids built in the other arithmetic mode must not be mixed in */
    if (s->dev) {
      klt_dev_invalidate(s->dev, -1);
      klt_dev_forget_host_frames(s->dev);     /* the caller may free its frame buffers now */
    }
    tc->pyramid_last = tc->pyramid_last_gradx = tc->pyramid_last_grady = NULL;
    s->last_slot = -1;
  }
  s->exact = exact != 0;
}

int KLTB200GetExact(KLT_TrackingContext tc) { return klt_state_get(tc)->exact; }

/* a setting of the tracker's launch only: the pyramids stay valid */
void KLTB200SetForwardBackward(KLT_TrackingContext tc, float max_error)
{
  if (isnan(max_error)) KLTError("(KLTB200SetForwardBackward) max_error is NaN");
  klt_state_get(tc)->fb_max_error = max_error;
}

float KLTB200GetForwardBackward(KLT_TrackingContext tc) { return klt_state_get(tc)->fb_max_error; }

void KLTB200ForwardBackwardResult(KLT_TrackingContext tc, int n, float *xb, float *yb, float *err,
                                  int *back_val)
{
  klt_tc_state *s = klt_state_find(tc);
  if (s == NULL || s->dev == NULL)
    KLTError("(KLTB200ForwardBackwardResult) no tracking call on this context ran the check");
  if (klt_dev_fb_results(s->dev, n, xb, yb, err, back_val) != 0)
    KLTError("(KLTB200ForwardBackwardResult) %s", klt_dev_error(s->dev));
}

/* a setting of the tracker's launch only, like the forward-backward check */
void KLTB200SetPrediction(KLT_TrackingContext tc, int mode)
{
  if (mode != KLT_B200_PREDICT_NONE && mode != KLT_B200_PREDICT_VELOCITY)
    KLTError("(KLTB200SetPrediction) mode %d (must be KLT_B200_PREDICT_NONE or KLT_B200_PREDICT_VELOCITY)", mode);
  klt_state_get(tc)->predict = mode;
}

int KLTB200GetPrediction(KLT_TrackingContext tc) { return klt_state_get(tc)->predict; }

void KLTB200SetGuesses(KLT_TrackingContext tc, int n, const float *gx, const float *gy, int on_device)
{
  klt_tc_state *s = klt_state_get(tc);
  if (klt_dev_set_guesses(klt_state_device(s), n, gx, gy, on_device) != 0)
    KLTError("(KLTB200SetGuesses) %s", klt_dev_error(s->dev));
}

void KLTB200PredictionResult(KLT_TrackingContext tc, int n, float *gx, float *gy, int *source)
{
  klt_tc_state *s = klt_state_find(tc);
  if (s == NULL || s->dev == NULL)
    KLTError("(KLTB200PredictionResult) no tracking call on this context ran with prediction");
  if (klt_dev_prediction_results(s->dev, n, gx, gy, source) != 0)
    KLTError("(KLTB200PredictionResult) %s", klt_dev_error(s->dev));
}
klt_dev *KLTB200Device(KLT_TrackingContext tc) { return klt_state_device(klt_state_get(tc)); }
int KLTB200LastSlot(KLT_TrackingContext tc)
{
  klt_tc_state *s = klt_state_find(tc);
  return (s && tc->pyramid_last) ? s->last_slot : -1;
}

/* ---- parameter repair shared by several entry points ---------------------- */
/* style 0: messages of klt.c ("(who) Window width must be odd. ...")
 * style 1: messages of trackFeatures.c / selectGoodFeatures.c */
void klt_fix_window(KLT_TrackingContext tc, const char *who, int style)
{
  int *dim[2];
  const char *name[2] = { "width", "height" };
  int k;
  dim[0] = &tc->window_width;
  dim[1] = &tc->window_height;
  for (k = 0; k < 2; k++)
    if (*dim[k] % 2 != 1) {
      *dim[k] += 1;
      if (style == 0)
        KLTWarning("(%s) Window %s must be odd.  Changing to %d.\n", who, name[k], *dim[k]);
      else
        KLTWarning("Tracking context's window %s must be odd.  Changing to %d.\n", name[k], *dim[k]);
    }
  for (k = 0; k < 2; k++)
    if (*dim[k] < 3) {
      *dim[k] = 3;
      if (style == 0)
        KLTWarning("(%s) Window %s must be at least three.  \nChanging to %d.\n", who, name[k], *dim[k]);
      else
        KLTWarning("Tracking context's window %s must be at least three.  \nChanging to %d.\n",
                   name[k], *dim[k]);
    }
}

float _KLTComputeSmoothSigma(KLT_TrackingContext tc)
{
  /* klt_util.c:20-24 */
  const int w = tc->window_width > tc->window_height ? tc->window_width : tc->window_height;
  return tc->smooth_sigma_fact * w;
}

/* ---- constructors ----------------------------------------------------------- */
KLT_TrackingContext KLTCreateTrackingContext(void)
{
  KLT_TrackingContext tc = (KLT_TrackingContext)malloc(sizeof(KLT_TrackingContextRec));
  if (!tc) KLTError("(KLTCreateTrackingContext) Out of memory");
  memset(tc, 0, sizeof(*tc));

  tc->mindist = 10;
  tc->window_width = tc->window_height = 7;
  tc->sequentialMode = FALSE;
  tc->smoothBeforeSelecting = TRUE;
  tc->writeInternalImages = FALSE;
  tc->lighting_insensitive = FALSE;
  tc->min_eigenvalue = 1;
  tc->min_determinant = 0.01f;
  tc->min_displacement = 0.1f;
  tc->max_iterations = 10;
  tc->max_residue = 10.0f;
  tc->grad_sigma = 1.0f;
  tc->smooth_sigma_fact = 0.1f;
  tc->pyramid_sigma_fact = 0.9f;
  tc->step_factor = 1.0f;
  tc->nSkippedPixels = 0;
  tc->affineConsistencyCheck = -1;
  tc->affine_window_width = tc->affine_window_height = 15;
  tc->affine_max_iterations = 10;
  tc->affine_max_residue = 10.0f;
  tc->affine_min_displacement = 0.02f;
  tc->affine_max_displacement_differ = 1.5f;
  tc->pyramid_last = tc->pyramid_last_gradx = tc->pyramid_last_grady = NULL;

  KLTChangeTCPyramid(tc, 15);     /* default search range */
  KLTUpdateTCBorder(tc);
  return tc;
}

static void feature_defaults(KLT_Feature f)
{
  f->aff_img = NULL;
  f->aff_img_gradx = NULL;
  f->aff_img_grady = NULL;
}

/* one block: header, pointer array, records (klt.c:148-167) */
/* Feature lists are one block (header, pointer array, records: reference klt.c:148-167).  When a
 * CUDA device is present the block is pinned host memory, so that KLTTrackFeatures can mirror the
 * records to the device in one copy and let the tracker write x | y | val of every feature straight
 * back into them (klt_dev_features_commit_records): no pack / unpack pass on the host.  Pinned
 * blocks are remembered here; anything else (no device, or a list built by hand) takes the
 * staging path. */
typedef struct pinned_block { void *p; struct pinned_block *next; } pinned_block;
static pinned_block *g_pinned = NULL;
static pthread_mutex_t g_pinned_lock = PTHREAD_MUTEX_INITIALIZER;

static void pinned_remember(void *p)
{
  pinned_block *b = (pinned_block *)malloc(sizeof(pinned_block));
  if (!b) KLTError("(KLTCreateFeatureList) Out of memory");
  pthread_mutex_lock(&g_pinned_lock);
  b->p = p; b->next = g_pinned; g_pinned = b;
  pthread_mutex_unlock(&g_pinned_lock);
}
int klt_list_is_pinned(const void *p)
{
  pinned_block *b;
  int found = 0;
  pthread_mutex_lock(&g_pinned_lock);
  for (b = g_pinned; b; b = b->next) if (b->p == p) { found = 1; break; }
  pthread_mutex_unlock(&g_pinned_lock);
  return found;
}
static int pinned_forget(void *p)
{
  pinned_block **pp, *b;
  int found = 0;
  pthread_mutex_lock(&g_pinned_lock);
  for (pp = &g_pinned; *pp; pp = &(*pp)->next)
    if ((*pp)->p == p) { b = *pp; *pp = b->next; free(b); found = 1; break; }
  pthread_mutex_unlock(&g_pinned_lock);
  return found;
}

KLT_FeatureList KLTCreateFeatureList(int nFeatures)
{
  const size_t bytes = sizeof(KLT_FeatureListRec) + (size_t)nFeatures * sizeof(KLT_Feature) +
                       (size_t)nFeatures * sizeof(KLT_FeatureRec);
  const char *env = getenv("KLT_B200_PINNED_LISTS");
  KLT_FeatureList fl = NULL;
  KLT_Feature recs;
  int i;
  if (env == NULL || atoi(env) != 0) fl = (KLT_FeatureList)klt_dev_host_alloc(bytes);
  if (fl) pinned_remember(fl);
  else fl = (KLT_FeatureList)malloc(bytes);
  if (!fl) KLTError("(KLTCreateFeatureList) Out of memory");
  fl->nFeatures = nFeatures;
  fl->feature = (KLT_Feature *)(fl + 1);
  recs = (KLT_Feature)(fl->feature + nFeatures);
  for (i = 0; i < nFeatures; i++) {
    fl->feature[i] = recs + i;
    feature_defaults(fl->feature[i]);
  }
  return fl;
}

KLT_FeatureHistory KLTCreateFeatureHistory(int nFrames)
{
  const size_t bytes = sizeof(KLT_FeatureHistoryRec) + (size_t)nFrames * sizeof(KLT_Feature) +
                       (size_t)nFrames * sizeof(KLT_FeatureRec);
  KLT_FeatureHistory fh = (KLT_FeatureHistory)malloc(bytes);
  KLT_Feature recs;
  int i;
  if (!fh) KLTError("(KLTCreateFeatureHistory) Out of memory");
  fh->nFrames = nFrames;
  fh->feature = (KLT_Feature *)(fh + 1);
  recs = (KLT_Feature)(fh->feature + nFrames);
  for (i = 0; i < nFrames; i++) fh->feature[i] = recs + i;
  return fh;
}

/* ft->feature[feat][frame]; row pointers and the pointer matrix share one block,
 * the records are a second block reachable as ft->feature[0][0] (klt.c:210-236) */
KLT_FeatureTable KLTCreateFeatureTable(int nFrames, int nFeatures)
{
  KLT_FeatureTable ft = (KLT_FeatureTable)malloc(sizeof(KLT_FeatureTableRec));
  const size_t rows = (size_t)nFeatures, cols = (size_t)nFrames;
  char *block;
  KLT_Feature recs;
  size_t i, j;
  if (!ft) KLTError("(KLTCreateFeatureTable) Out of memory");
  ft->nFrames = nFrames;
  ft->nFeatures = nFeatures;
  block = (char *)malloc(rows * sizeof(void *) + rows * cols * sizeof(KLT_Feature));
  recs = (KLT_Feature)malloc((rows > 0 && cols > 0 ? rows * cols : 1) * sizeof(KLT_FeatureRec));
  if (!block || !recs) KLTError("(KLTCreateFeatureTable) Out of memory");
  ft->feature = (KLT_Feature **)block;
  for (j = 0; j < rows; j++) {
    ft->feature[j] = (KLT_Feature *)(block + rows * sizeof(void *) + j * cols * sizeof(KLT_Feature));
    for (i = 0; i < cols; i++) ft->feature[j][i] = recs + j * cols + i;
  }
  return ft;
}

/* ---- pyramid / border parameters -------------------------------------------- */
void KLTChangeTCPyramid(KLT_TrackingContext tc, int search_range)
{
  float window_halfwidth, subsampling;
  klt_fix_window(tc, "KLTChangeTCPyramid", 0);
  window_halfwidth = (tc->window_width < tc->window_height ? tc->window_width : tc->window_height) / 2.0f;
  subsampling = ((float)search_range) / window_halfwidth;

  if (subsampling < 1.0) {
    tc->nPyramidLevels = 1;
  } else if (subsampling <= 3.0) {
    tc->nPyramidLevels = 2;
    tc->subsampling = 2;
  } else if (subsampling <= 5.0) {
    tc->nPyramidLevels = 2;
    tc->subsampling = 4;
  } else if (subsampling <= 9.0) {
    tc->nPyramidLevels = 2;
    tc->subsampling = 8;
  } else {
    /* search_range = halfwidth * (8^levels - 1) / 7, rounded up */
    const float val = (float)(log(7.0 * subsampling + 1.0) / log(8.0));
    tc->nPyramidLevels = (int)(val + 0.99);
    tc->subsampling = 8;
  }
}

void KLTUpdateTCBorder(KLT_TrackingContext tc)
{
  const int ss = tc->subsampling;
  int gauss_w, deriv_w, smooth_hw, pyramid_hw, invalid, window_hw, scale = 1, border, i;

  klt_fix_window(tc, "KLTUpdateTCBorder", 0);
  window_hw = (tc->window_width > tc->window_height ? tc->window_width : tc->window_height) / 2;

  _KLTGetKernelWidths(_KLTComputeSmoothSigma(tc), &gauss_w, &deriv_w);
  smooth_hw = gauss_w / 2;
  _KLTGetKernelWidths(tc->pyramid_sigma_fact * tc->subsampling, &gauss_w, &deriv_w);
  pyramid_hw = gauss_w / 2;

  /* pixels invalidated by the convolutions, expressed at each coarser level */
  invalid = smooth_hw;
  for (i = 1; i < tc->nPyramidLevels; i++) {
    const float val = ((float)invalid + pyramid_hw) / ss;
    invalid = (int)(val + 0.99);
  }
  for (i = 1; i < tc->nPyramidLevels; i++) scale *= ss;
  border = (invalid + window_hw) * scale;
  tc->borderx = border;
  tc->bordery = border;
}

/* ---- destructors --------------------------------------------------------------- */
void KLTFreeTrackingContext(KLT_TrackingContext tc)
{
  if (!tc) return;
  klt_state_drop(tc);          /* frees the device pyramids tc->pyramid_last* stand for */
  free(tc);
}

unsigned klt_aff_epoch = 1;

void KLTFreeFeatureList(KLT_FeatureList fl)
{
  int i;
  klt_aff_epoch++;               /* device mirrors keyed by these template addresses are stale now */
  for (i = 0; i < fl->nFeatures; i++) {
    /* the affine consistency check's templates (klt.c:453-469) */
    free(fl->feature[i]->aff_img);
    free(fl->feature[i]->aff_img_gradx);
    free(fl->feature[i]->aff_img_grady);
    feature_defaults(fl->feature[i]);
  }
  if (pinned_forget(fl)) klt_dev_host_free(fl);
  else free(fl);
}

void KLTFreeFeatureHistory(KLT_FeatureHistory fh) { free(fh); }

void KLTFreeFeatureTable(KLT_FeatureTable ft)
{
  if (ft->nFeatures > 0 && ft->nFrames > 0) free(ft->feature[0][0]);
  free(ft->feature);
  free(ft);
}

void KLTStopSequentialMode(KLT_TrackingContext tc)
{
  klt_tc_state *s = klt_state_find(tc);
  tc->sequentialMode = FALSE;
  if (s) {
    if (s->dev) {
      klt_dev_invalidate(s->dev, -1);
      klt_dev_forget_host_frames(s->dev);     /* the caller may free its frame buffers now */
    }
    s->last_slot = -1;
  }
  tc->pyramid_last = tc->pyramid_last_gradx = tc->pyramid_last_grady = NULL;
}

int KLTCountRemainingFeatures(KLT_FeatureList fl)
{
  int i, count = 0;
  for (i = 0; i < fl->nFeatures; i++)
    if (fl->feature[i]->val >= 0) count++;
  return count;
}

void KLTSetVerbosity(int verbosity) { KLT_verbose = verbosity; }

void KLTPrintTrackingContext(KLT_TrackingContext tc)
{
  FILE *o = stderr;
#define YN(b) ((b) ? "TRUE" : "FALSE")
#define PTR(p) ((p) != NULL ? "points to old image" : "NULL")
  fprintf(o, "\n\nTracking context:\n\n");
  fprintf(o, "\tmindist = %d\n", tc->mindist);
  fprintf(o, "\twindow_width = %d\n", tc->window_width);
  fprintf(o, "\twindow_height = %d\n", tc->window_height);
  fprintf(o, "\tsequentialMode = %s\n", YN(tc->sequentialMode));
  fprintf(o, "\tsmoothBeforeSelecting = %s\n", YN(tc->smoothBeforeSelecting));
  fprintf(o, "\twriteInternalImages = %s\n", YN(tc->writeInternalImages));
  fprintf(o, "\tmin_eigenvalue = %d\n", tc->min_eigenvalue);
  fprintf(o, "\tmin_determinant = %f\n", tc->min_determinant);
  fprintf(o, "\tmin_displacement = %f\n", tc->min_displacement);
  fprintf(o, "\tmax_iterations = %d\n", tc->max_iterations);
  fprintf(o, "\tmax_residue = %f\n", tc->max_residue);
  fprintf(o, "\tgrad_sigma = %f\n", tc->grad_sigma);
  fprintf(o, "\tsmooth_sigma_fact = %f\n", tc->smooth_sigma_fact);
  fprintf(o, "\tpyramid_sigma_fact = %f\n", tc->pyramid_sigma_fact);
  fprintf(o, "\tnSkippedPixels = %d\n", tc->nSkippedPixels);
  fprintf(o, "\tborderx = %d\n", tc->borderx);
  fprintf(o, "\tbordery = %d\n", tc->bordery);
  fprintf(o, "\tnPyramidLevels = %d\n", tc->nPyramidLevels);
  fprintf(o, "\tsubsampling = %d\n", tc->subsampling);
  fprintf(o, "\n\tpyramid_last = %s\n", PTR(tc->pyramid_last));
  fprintf(o, "\tpyramid_last_gradx = %s\n", PTR(tc->pyramid_last_gradx));
  fprintf(o, "\tpyramid_last_grady = %s\n", PTR(tc->pyramid_last_grady));
  fprintf(o, "\n\n");
#undef YN
#undef PTR
}

/* ---- helpers used by the hot-path wrappers ----------------------------------- */
void klt_fill_build_desc(KLT_TrackingContext tc, int ncols, int nrows, int nlevels_built,
                         int smooth, int exact, klt_dev_build_desc *q)
{
  memset(q, 0, sizeof(*q));
  q->ncols = ncols;
  q->nrows = nrows;
  q->nlevels = tc->nPyramidLevels;
  q->subsampling = tc->subsampling;
  q->nlevels_built = nlevels_built;
  q->smooth = smooth;
  q->exact = exact;
  /* taps are fetched in the order the reference would need them, so the
   * sigma cache (klt_taps.c) sees the same sequence: smooth, pyramid, gradient
   * (trackFeatures.c:1313-1321) */
  if (smooth) klt_taps_for(_KLTComputeSmoothSigma(tc), &q->smooth_taps);
  if (nlevels_built > 1) klt_taps_for(tc->subsampling * tc->pyramid_sigma_fact, &q->pyramid_taps);
  klt_taps_for(tc->grad_sigma, &q->grad_taps);
}

void klt_list_to_arrays(KLT_FeatureList fl, float *x, float *y, int *v)
{
  int i;
  for (i = 0; i < fl->nFeatures; i++) {
    x[i] = fl->feature[i]->x;
    y[i] = fl->feature[i]->y;
    v[i] = fl->feature[i]->val;
  }
}
