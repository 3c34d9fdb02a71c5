/* klt_internal.h -- private to the host C side of libklt_b200. */
#ifndef KLT_INTERNAL_H
#define KLT_INTERNAL_H

#include "klt.h"
#include "klt_b200.h"
#include "klt_cuda.h"

extern int KLT_verbose;

/* per-tracking-context device state (csrc/klt_context.c) */
typedef struct klt_tc_state {
  KLT_TrackingContext tc;
  klt_dev *dev;          /* created on first use of the hot path            */
  int device;            /* CUDA device ordinal, -1 = KLT_B200_DEVICE / current */
  int exact;             /* arithmetic mode for tracking pyramids            */
  float fb_max_error;    /* forward-backward check, > 0: on (KLTB200SetForwardBackward) */
  int predict;           /* motion prior: KLT_B200_PREDICT_* (KLTB200SetPrediction)      */
  int last_slot;         /* slot holding the previous frame's pyramids       */
  /* affine consistency check: which host template (aff_img pointer) the device's template
   * slot i mirrors; valid for list aff_list while klt_aff_epoch == aff_epoch */
  void **aff_shadow;
  int aff_shadow_n;
  int in_sequence;            /* KLTTrackFeaturesSequence is setting the resident pipeline up (affine check allowed) */
  const void *aff_list;
  unsigned aff_epoch;
  struct klt_tc_state *next;
} klt_tc_state;

klt_tc_state *klt_state_get(KLT_TrackingContext tc);          /* creates the record   */
klt_tc_state *klt_state_find(KLT_TrackingContext tc);         /* NULL if none         */
void klt_state_drop(KLT_TrackingContext tc);                  /* destroys the device  */
klt_dev *klt_state_device(klt_tc_state *s);                   /* KLTError on failure  */

/* taps with the reference's sigma cache (csrc/klt_taps.c) */
void klt_taps_for(float sigma, klt_dev_taps *out);            /* cache rule applies   */
void _KLTGetKernelWidths(float sigma, int *gauss_width, int *gaussderiv_width);

/* shared parameter repair (window odd and >= 3) */
void klt_fix_window(KLT_TrackingContext tc, const char *who, int style);

/* build descriptor from a tracking context */
void klt_fill_build_desc(KLT_TrackingContext tc, int ncols, int nrows,
                         int nlevels_built, int smooth, int exact,
                         klt_dev_build_desc *q);

/* 1 if fl is a pinned block made by KLTCreateFeatureList (record mode of the tracker) */
int klt_list_is_pinned(const void *p);

/* device selection parameters from a tracking context (csrc/klt_select.c) */
void klt_fill_select_params(KLT_TrackingContext tc, int replacing, klt_dev_select_params *sp);

/* bumped by KLTFreeFeatureList: template addresses may be reused afterwards */
extern unsigned klt_aff_epoch;

/* list <-> SoA staging */
void klt_list_to_arrays(KLT_FeatureList fl, float *x, float *y, int *v);

#endif
