// klt_dev.cu -- hand-written sm_100a CUDA kernels + the C-ABI of include/klt_cuda.h.
//
// Replaces (reference file:line):
//   _KLTToFloatImage / _convolveImageHoriz / _convolveImageVert / _convolveSeparate /
//   _KLTComputeSmoothedImage / _KLTComputeGradients      src/V1/convolve.c:37-314
//   _KLTComputePyramid                                    src/V1/pyramid.c:87-131
//   eigenvalue loop, _sortPointList, _enforceMinimumDistance
//                                                         src/V1/selectGoodFeatures.c:102-239,373-446
//   _interpolate ... _trackFeature, feature loop          src/V1/trackFeatures.c:31-486,1343-1437
//
// Numerics.  Every kernel exists in two arithmetic modes selected by a template
// flag:  EXACT = reference order of operations with separately rounded multiply
// and add (bit-identical to the CPU reference built without FMA);  !EXACT = the
// same order with fused multiply-add and shuffle-tree reductions (production,
// within 1e-4 relative of the reference).
//
// Border semantics of the separable passes (convolve.c:164-178, :216-237): the
// horizontal pass writes 0 for x < R or x >= W-R, the vertical pass consumes that
// result and writes 0 for y < R or y >= H-R.  Interior outputs only ever touch
// in-range inputs, so tiles may zero-fill reads outside the image.
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <climits>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sched.h>

#include "klt_cuda.h"

#define KLT_TRACKED         0
#define KLT_NOT_FOUND      -1
#define KLT_SMALL_DET      -2
#define KLT_MAX_ITERATIONS -3
#define KLT_OOB            -4
#define KLT_LARGE_RESIDUE  -5
#define KLT_B200_FB_INCONSISTENT -6   // include/klt_b200.h

// ---------------------------------------------------------------------------
// arithmetic helpers
// ---------------------------------------------------------------------------
template <bool EXACT>
__device__ __forceinline__ float mac(float acc, float a, float b) {
  if (EXACT) return __fadd_rn(acc, __fmul_rn(a, b));
  return fmaf(a, b, acc);
}
template <bool EXACT>
__device__ __forceinline__ float mul(float a, float b) {
  if (EXACT) return __fmul_rn(a, b);
  return a * b;
}

// taps in application order: k[m] multiplies in[x - R + m]  (the reference walks
// its array backwards, convolve.c:169-173, so k[m] = ref[w-1-m]).
struct TapsR {
  int   w;
  float k[KLT_DEV_MAX_TAPS];
};

// taps of the fused kernels (radius <= 11): plain (k) and duplicated (kk[m] = {k[m], k[m]}) so that
// a packed FFMA2 can take its multiplier pair straight from a 64-bit constant / uniform register
static constexpr int FUSED_MAX_TAPS = 24;
struct TapsF {
  int    w, pad;
  float  k[FUSED_MAX_TAPS];
  float2 kk[FUSED_MAX_TAPS];
};

static constexpr int NT = 256;   // threads per CTA of every tile kernel

#include "klt_fused.cuh"
#include "klt_march.cuh"

// ---------------------------------------------------------------------------
// generic kernels: any radius, any subsampling.  One thread per output sample.
// Used for parameter combinations the tiled kernels are not instantiated for,
// and as an independent cross-check of the tiled kernels.
// ---------------------------------------------------------------------------
template <typename SrcT, bool EXACT>
__global__ void conv_h_generic(const SrcT* __restrict__ src, int spitch, int W, int H,
                               TapsR taps, int stride, int off,
                               float* __restrict__ out, int opitch, int Wout) {
  const int xo = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (xo >= Wout || y >= H) return;
  const int R = taps.w / 2;
  const int xs = stride * xo + off;
  float acc = 0.0f;
  if (xs >= R && xs < W - R) {
    const SrcT* p = src + (size_t)y * spitch + (xs - R);
    for (int m = 0; m < taps.w; ++m) acc = mac<EXACT>(acc, (float)p[m], taps.k[m]);
  }
  out[(size_t)y * opitch + xo] = acc;
}

template <bool EXACT>
__global__ void conv_v_generic(const float* __restrict__ src, int spitch, int Wout, int Hsrc,
                               TapsR taps, int stride, int off,
                               float* __restrict__ out, int opitch, int Hout) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int yo = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= Wout || yo >= Hout) return;
  const int R = taps.w / 2;
  const int ys = stride * yo + off;
  float acc = 0.0f;
  if (ys >= R && ys < Hsrc - R) {
    const float* p = src + (size_t)(ys - R) * spitch + x;
    for (int m = 0; m < taps.w; ++m) acc = mac<EXACT>(acc, p[(size_t)m * spitch], taps.k[m]);
  }
  out[(size_t)yo * opitch + x] = acc;
}

// _KLTToFloatImage (convolve.c:37-53) for smoothBeforeSelecting == FALSE
__global__ void u8_to_f32_kernel(const unsigned char* __restrict__ src, int spitch, int W, int H,
                                 float* __restrict__ out, int opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x < W && y < H) out[(size_t)y * opitch + x] = (float)src[(size_t)y * spitch + x];
}

// ---------------------------------------------------------------------------
// tiled kernels.  A CTA owns one output tile; the source region (tile + halo)
// is staged once in shared memory, the horizontal pass runs from shared memory
// into shared memory with a register-blocked sliding window (float4 loads, PX
// outputs per thread), the vertical pass runs from shared memory to global with
// a register sliding window (PY outputs per thread, lanes along x => coalesced
// 128 B stores).  The horizontal result never goes to HBM.
// ---------------------------------------------------------------------------
template <typename SrcT>
__device__ __forceinline__ void stage_region(float* s, int sp, const SrcT* __restrict__ src,
                                             int spitch, int W, int H, int gx0, int gy0,
                                             int cols, int rows) {
  for (int i = threadIdx.x; i < rows * cols; i += NT) {
    const int r = i / cols, c = i - r * cols;
    const int gx = gx0 + c, gy = gy0 + r;
    float v = 0.0f;
    if (gx >= 0 && gx < W && gy >= 0 && gy < H) v = (float)__ldg(src + (size_t)gy * spitch + gx);
    s[r * sp + c] = v;
  }
}

// geometry of a tile kernel, all compile time.
//   SS  : subsampling between source and output (1 for plain convolution)
//   RM  : halo radius staged around the tile (max radius of the taps used)
template <int SS, int RM, int TXO, int TYO, int PX>
struct TileGeo {
  static constexpr int IW   = SS * (TXO - 1) + 2 * RM + 1;           // staged columns
  static constexpr int IH   = SS * (TYO - 1) + 2 * RM + 1;           // staged rows
  static constexpr int NWIN = SS * (PX - 1) + 2 * RM + 1;            // window of one thread
  static constexpr int NV4  = (NWIN + 3) / 4;
  static constexpr int SP0  = SS * (TXO - PX) + 4 * NV4;
  static constexpr int SP   = (SP0 > IW ? SP0 : IW) + ((4 - ((SP0 > IW ? SP0 : IW) & 3)) & 3);
  static constexpr int IN_FLOATS = IH * SP;
};

// ---- level 0: u8 frame -> smoothed float image -----------------------------
// replaces _KLTToFloatImage + _KLTComputeSmoothedImage (convolve.c:37-53,300-314)
template <int R, bool EXACT>
__global__ void __launch_bounds__(NT)
smooth_u8_tile(const unsigned char* __restrict__ src, int spitch, int W, int H, TapsR taps,
               float* __restrict__ out, int opitch) {
  constexpr int TX = 64, TY = 32, PX = 4, PY = 8;
  using G = TileGeo<1, R, TX, TY, PX>;
  extern __shared__ __align__(16) float smem[];
  float* sIn = smem;
  float* sH = smem + G::IN_FLOATS;            // [IH][TX]
  const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;

  stage_region(sIn, G::SP, src, spitch, W, H, x0 - R, y0 - R, G::IW, G::IH);
  __syncthreads();

  for (int item = threadIdx.x; item < G::IH * (TX / PX); item += NT) {
    const int r = item / (TX / PX), g = item - r * (TX / PX);
    float win[4 * G::NV4];
    const float4* p = reinterpret_cast<const float4*>(sIn + r * G::SP + g * PX);
#pragma unroll
    for (int v = 0; v < G::NV4; ++v) {
      const float4 t = p[v];
      win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
    }
    float o[PX];
#pragma unroll
    for (int q = 0; q < PX; ++q) {
      float acc = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[q + m], taps.k[m]);
      const int xg = x0 + g * PX + q;
      o[q] = (xg < R || xg >= W - R) ? 0.0f : acc;
    }
    *reinterpret_cast<float4*>(sH + r * TX + g * PX) = make_float4(o[0], o[1], o[2], o[3]);
  }
  __syncthreads();

  for (int item = threadIdx.x; item < TX * (TY / PY); item += NT) {
    const int gy = item / TX, c = item - gy * TX;
    float win[PY + 2 * R];
#pragma unroll
    for (int i = 0; i < PY + 2 * R; ++i) win[i] = sH[(gy * PY + i) * TX + c];
    const int xg = x0 + c;
#pragma unroll
    for (int q = 0; q < PY; ++q) {
      float acc = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[q + m], taps.k[m]);
      const int yg = y0 + gy * PY + q;
      if (yg < R || yg >= H - R) acc = 0.0f;
      if (xg < W && yg < H) out[(size_t)yg * opitch + xg] = acc;
    }
  }
}

// ---- gradients of one level ------------------------------------------------
// replaces _KLTComputeGradients (convolve.c:273-293): gradx = V_g(H_d(img)),
// grady = V_d(H_g(img)); both horizontal passes share one staged window.
template <int RG, int RD, bool EXACT>
__global__ void __launch_bounds__(NT)
grad_tile(const float* __restrict__ src, int spitch, int W, int H, TapsR tg, TapsR td,
          float* __restrict__ outx, float* __restrict__ outy, int opitch) {
  constexpr int RM = RG > RD ? RG : RD;
  constexpr int TX = 64, TY = 32, PX = 4, PY = 8;
  using G = TileGeo<1, RM, TX, TY, PX>;
  extern __shared__ __align__(16) float smem[];
  float* sIn = smem;
  float* sHd = smem + G::IN_FLOATS;           // [IH][TX]  horizontal derivative
  float* sHg = sHd + G::IH * TX;              // [IH][TX]  horizontal gaussian
  const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;

  stage_region(sIn, G::SP, src, spitch, W, H, x0 - RM, y0 - RM, G::IW, G::IH);
  __syncthreads();

  for (int item = threadIdx.x; item < G::IH * (TX / PX); item += NT) {
    const int r = item / (TX / PX), g = item - r * (TX / PX);
    float win[4 * G::NV4];
    const float4* p = reinterpret_cast<const float4*>(sIn + r * G::SP + g * PX);
#pragma unroll
    for (int v = 0; v < G::NV4; ++v) {
      const float4 t = p[v];
      win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
    }
    float od[PX], og[PX];
#pragma unroll
    for (int q = 0; q < PX; ++q) {
      float a = 0.0f, b = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * RD + 1; ++m) a = mac<EXACT>(a, win[q + (RM - RD) + m], td.k[m]);
#pragma unroll
      for (int m = 0; m < 2 * RG + 1; ++m) b = mac<EXACT>(b, win[q + (RM - RG) + m], tg.k[m]);
      const int xg = x0 + g * PX + q;
      od[q] = (xg < RD || xg >= W - RD) ? 0.0f : a;
      og[q] = (xg < RG || xg >= W - RG) ? 0.0f : b;
    }
    *reinterpret_cast<float4*>(sHd + r * TX + g * PX) = make_float4(od[0], od[1], od[2], od[3]);
    *reinterpret_cast<float4*>(sHg + r * TX + g * PX) = make_float4(og[0], og[1], og[2], og[3]);
  }
  __syncthreads();

  for (int item = threadIdx.x; item < TX * (TY / PY); item += NT) {
    const int gy = item / TX, c = item - gy * TX;
    float wd[PY + 2 * RM], wg[PY + 2 * RM];
#pragma unroll
    for (int i = 0; i < PY + 2 * RM; ++i) {
      wd[i] = sHd[(gy * PY + i) * TX + c];
      wg[i] = sHg[(gy * PY + i) * TX + c];
    }
    const int xg = x0 + c;
#pragma unroll
    for (int q = 0; q < PY; ++q) {
      float a = 0.0f, b = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * RG + 1; ++m) a = mac<EXACT>(a, wd[q + (RM - RG) + m], tg.k[m]);
#pragma unroll
      for (int m = 0; m < 2 * RD + 1; ++m) b = mac<EXACT>(b, wg[q + (RM - RD) + m], td.k[m]);
      const int yg = y0 + gy * PY + q;
      if (yg < RG || yg >= H - RG) a = 0.0f;
      if (yg < RD || yg >= H - RD) b = 0.0f;
      if (xg < W && yg < H) {
        outx[(size_t)yg * opitch + xg] = a;
        outy[(size_t)yg * opitch + xg] = b;
      }
    }
  }
}

// ---- one pyramid step --------------------------------------------------------
// replaces the smooth + subsample step of _KLTComputePyramid (pyramid.c:112-124):
// the Gaussian is evaluated only at the kept samples (SS*x + SS/2, SS*y + SS/2).
template <int SS, int R, int TXO, int TYO, int PY, bool EXACT>
__global__ void __launch_bounds__(NT)
pyrdown_tile(const float* __restrict__ src, int spitch, int W, int H, TapsR taps,
             float* __restrict__ out, int opitch, int Wout, int Hout) {
  constexpr int PX = 4;
  using G = TileGeo<SS, R, TXO, TYO, PX>;
  extern __shared__ __align__(16) float smem[];
  float* sIn = smem;
  float* sH = smem + G::IN_FLOATS;            // [IH][TXO]
  const int x0 = blockIdx.x * TXO, y0 = blockIdx.y * TYO;
  const int xs0 = SS * x0 + SS / 2 - R, ys0 = SS * y0 + SS / 2 - R;

  stage_region(sIn, G::SP, src, spitch, W, H, xs0, ys0, G::IW, G::IH);
  __syncthreads();

  for (int item = threadIdx.x; item < G::IH * (TXO / PX); item += NT) {
    const int r = item / (TXO / PX), g = item - r * (TXO / PX);
    float win[4 * G::NV4];
    const float4* p = reinterpret_cast<const float4*>(sIn + r * G::SP + SS * g * PX);
#pragma unroll
    for (int v = 0; v < G::NV4; ++v) {
      const float4 t = p[v];
      win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
    }
    float o[PX];
#pragma unroll
    for (int q = 0; q < PX; ++q) {
      float acc = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[SS * q + m], taps.k[m]);
      const int xs = SS * (x0 + g * PX + q) + SS / 2;
      o[q] = (xs < R || xs >= W - R) ? 0.0f : acc;
    }
    *reinterpret_cast<float4*>(sH + r * TXO + g * PX) = make_float4(o[0], o[1], o[2], o[3]);
  }
  __syncthreads();

  for (int item = threadIdx.x; item < TXO * (TYO / PY); item += NT) {
    const int gy = item / TXO, c = item - gy * TXO;
    constexpr int NW = SS * (PY - 1) + 2 * R + 1;
    float win[NW];
#pragma unroll
    for (int i = 0; i < NW; ++i) win[i] = sH[(SS * gy * PY + i) * TXO + c];
    const int xo = x0 + c;
#pragma unroll
    for (int q = 0; q < PY; ++q) {
      float acc = 0.0f;
#pragma unroll
      for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[SS * q + m], taps.k[m]);
      const int yo = y0 + gy * PY + q;
      const int ys = SS * yo + SS / 2;
      if (ys < R || ys >= H - R) acc = 0.0f;
      if (xo < Wout && yo < Hout) out[(size_t)yo * opitch + xo] = acc;
    }
  }
}

// ---------------------------------------------------------------------------
// selection kernels
// ---------------------------------------------------------------------------
// Eigenvalue map (selectGoodFeatures.c:396-423, :289-292).  One thread per
// candidate pixel; the 3 window sums run in raster order with separately
// rounded multiply/add, the eigenvalue formula in double exactly as the
// reference, then truncation to int.  Always exact: the result is an integer
// ranking key, so 1-ulp differences would reorder candidates.
// range[0] / range[1]: running maximum / minimum of the integers (both start at 0): the host
// sorts only the bits the keys actually use.  A look at the current value first keeps all but a
// handful of threads off the atomic.
__device__ __forceinline__ void note_range(int* range, int vmax, int vmin) {
  if (vmax > __ldcg(range)) atomicMax(range, vmax);
  if (vmin < 0 && vmin < __ldcg(range + 1)) atomicMin(range + 1, vmin);
}

__global__ void mineig_kernel(const float* __restrict__ gx, const float* __restrict__ gy, int pitch,
                              int bx, int by, int step, int nxc, int nyc, int hw, int hh,
                              int* __restrict__ vals, unsigned* __restrict__ idx, int* range, int clamp_neg,
                              const unsigned char* __restrict__ covered, int W) {
  const int ix = blockIdx.x * blockDim.x + threadIdx.x;
  const int iy = blockIdx.y * blockDim.y + threadIdx.y;
  if (ix >= nxc || iy >= nyc) return;
  const int x = bx + ix * step, y = by + iy * step;
  float gxx = 0.0f, gxy = 0.0f, gyy = 0.0f;
  for (int yy = y - hh; yy <= y + hh; ++yy) {
    const float* px = gx + (size_t)yy * pitch + (x - hw);
    const float* py = gy + (size_t)yy * pitch + (x - hw);
    for (int i = 0; i <= 2 * hw; ++i) {
      const float a = __ldg(px + i), b = __ldg(py + i);
      gxx = __fadd_rn(gxx, __fmul_rn(a, a));
      gxy = __fadd_rn(gxy, __fmul_rn(a, b));
      gyy = __fadd_rn(gyy, __fmul_rn(b, b));
    }
  }
  const float dif = __fsub_rn(gxx, gyy);
  const float rad = __fadd_rn(__fmul_rn(dif, dif), __fmul_rn(__fmul_rn(4.0f, gxy), gxy));
  const double ev = __ddiv_rn(__dsub_rn((double)__fadd_rn(gxx, gyy), sqrt((double)rad)), 2.0);
  const float v = (float)ev;
  const int n = iy * nxc + ix;
  int vi = (int)v;           // truncation toward zero, as the C cast
  // (rounding can leave a rank-deficient window a few units below zero; for the selection such a
  // key is as dead as 0 -- the threshold is >= 1 -- and non-negative keys let the sort skip bits)
  if (clamp_neg && vi < 0) vi = 0;
  if (covered && covered[(size_t)y * W + x]) vi = 0;       // (replacement: see run_mineig)
  vals[n] = vi;
  idx[n] = (unsigned)n;
  note_range(range, vi, vi);
}

// The same for the default 7x7 window and step 1, 8 consecutive candidates per thread: the 14
// pixels of a window row that the 8 windows cover are loaded once (4 aligned 128-bit loads per
// gradient image instead of 8 x 7 scalar ones), their products gx*gx, gx*gy, gy*gy are formed once
// and added into every window they belong to, pixel by pixel in increasing x -- for each candidate
// that is exactly the raster order and the separately rounded multiply / add of the reference, so
// the integers are identical; ~2x fewer instructions and L1 wavefronts than one thread per candidate.
__device__ __forceinline__ int mineig_value(float gxx, float gxy, float gyy) {
  const float dif = __fsub_rn(gxx, gyy);
  const float rad = __fadd_rn(__fmul_rn(dif, dif), __fmul_rn(__fmul_rn(4.0f, gxy), gxy));
  const double ev = __ddiv_rn(__dsub_rn((double)__fadd_rn(gxx, gyy), sqrt((double)rad)), 2.0);
  return (int)(float)ev;                         // truncation toward zero, as the C cast
}

__global__ void __launch_bounds__(128)
mineig7_kernel(const float* __restrict__ gx, const float* __restrict__ gy, int pitch,
               int bx, int by, int nxc, int nyc, int* __restrict__ vals, unsigned* __restrict__ idx, int* range,
               int clamp_neg, const unsigned char* __restrict__ covered, int W) {
  const int X0 = (bx & ~7) + 8 * (blockIdx.x * blockDim.x + threadIdx.x);    // absolute x of this thread's first candidate
  const int iy = blockIdx.y * blockDim.y + threadIdx.y;
  if (X0 >= bx + nxc || iy >= nyc) return;
  const int y = by + iy;
  float sxx[8], sxy[8], syy[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) { sxx[c] = 0.0f; sxy[c] = 0.0f; syy[c] = 0.0f; }
#pragma unroll 1
  for (int r = 0; r < 7; ++r) {
    const size_t row = (size_t)(y - 3 + r) * pitch + (size_t)(X0 - 4);       // 16 B aligned: pitch % 32 == 0, X0 % 8 == 0
    const float4* pa = reinterpret_cast<const float4*>(gx + row);
    const float4* pb = reinterpret_cast<const float4*>(gy + row);
    float a[16], b[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 va = __ldg(pa + q), vb = __ldg(pb + q);
      a[4 * q] = va.x; a[4 * q + 1] = va.y; a[4 * q + 2] = va.z; a[4 * q + 3] = va.w;
      b[4 * q] = vb.x; b[4 * q + 1] = vb.y; b[4 * q + 2] = vb.z; b[4 * q + 3] = vb.w;
    }
#pragma unroll
    for (int k = 1; k <= 14; ++k) {              // pixel X0 - 4 + k belongs to the windows of candidates k-7 .. k-1
      const float pxx = __fmul_rn(a[k], a[k]), pxy = __fmul_rn(a[k], b[k]), pyy = __fmul_rn(b[k], b[k]);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        if (c >= k - 7 && c <= k - 1) {
          sxx[c] = __fadd_rn(sxx[c], pxx); sxy[c] = __fadd_rn(sxy[c], pxy); syy[c] = __fadd_rn(syy[c], pyy);
        }
      }
    }
  }
  int vmax = 0, vmin = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int x = X0 + c;
    if (x >= bx && x < bx + nxc) {
      const int n = iy * nxc + (x - bx);
      int v = mineig_value(sxx[c], sxy[c], syy[c]);
      if (clamp_neg && v < 0) v = 0;
      if (covered && covered[(size_t)y * W + x]) v = 0;
      vals[n] = v;
      idx[n] = (unsigned)n;
      vmax = max(vmax, v); vmin = min(vmin, v);
    }
  }
  note_range(range, vmax, vmin);
}

// featuremap pre-stamp of the surviving features in REPLACING_SOME mode
// (selectGoodFeatures.c:160-166): one CTA per feature.
__global__ void stamp_existing_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                      const int* __restrict__ val, unsigned char* fmap,
                                      int d, int W, int H) {
  const int f = blockIdx.x;
  if (val[f] < 0 || d < 0) return;
  const int cx = (int)x[f], cy = (int)y[f];
  const int side = 2 * d + 1;
  for (int i = threadIdx.x; i < side * side; i += blockDim.x) {
    const int ix = cx - d + i % side, iy = cy - d + i / side;
    if (ix >= 0 && ix < W && iy >= 0 && iy < H) fmap[(size_t)iy * W + ix] = 1;
  }
}

// Greedy minimum-distance pass (selectGoodFeatures.c:168-235) on the sorted
// candidate list, made deterministic AND parallel: one CTA walks the list in
// batches of 1024 or GBATCH = 4096 consecutive ranks (1 or 4 per thread, see gk
// below; the next batch's keys are fetched while the current one is resolved).  Threads test the
// featuremap in parallel, survivors are compacted in rank order, and warp 0
// resolves them in rank order, 32 at a time, against the candidates already
// accepted in this batch (the only ones not yet stamped):
//  * those live in a shared-memory hash table keyed by the (d+1) x (d+1) cell they fall in --
//    two accepted candidates can never share a cell, and a conflict can only sit in the 3 x 3
//    cells around a survivor, so the test is 9 probes whatever the number accepted;
//  * conflicts inside the group of 32 are found with shuffles and settled by a fixed-point
//    iteration on ballots (the lowest undecided lane is decided in every round; a lane is
//    accepted once no earlier lane that conflicts with it is accepted or undecided).
// Accepted candidates are compacted in place at the front of the survivor arrays; records and
// stamps are then written by the whole CTA.  This reproduces the sequential result exactly
// for any batch size.  (Measured on B200 before this form: the per-accepted global load of
// open_slots[] inside the sequential loop, then the O(survivors x accepted) list test, made a
// 4K selection spend 2.4 of its 3.1 ms here.)
static constexpr int GB = 1024;
static constexpr int GK = 4;
static constexpr int GBATCH = GB * GK;

// exclusive block-wide prefix of each thread's count, in thread order; returns
// the total through *total_out (valid for all threads).  Contains two
// __syncthreads; s_wcount is scratch of GB/32 ints.
__device__ __forceinline__ int block_prefix(int cnt, int* s_wcount, int* s_total_tmp, int* total_out) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_wcount[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    const int c = s_wcount[lane];
    int winc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    s_wcount[lane] = winc - c;                   // exclusive prefix over warps
    if (lane == 31) *s_total_tmp = winc;
  }
  __syncthreads();
  *total_out = *s_total_tmp;
  return s_wcount[wid] + inc - cnt;
}

static constexpr int GTBL = 2 * GBATCH;                  // hash slots: load <= 50 % even if a whole batch is accepted
static constexpr unsigned GEMPTY = 0xffffffffu;
static constexpr size_t ENFORCE_SMEM = (size_t)GBATCH * 4 + (size_t)GTBL * 4 + (size_t)GBATCH * 4 * 2 + (size_t)GBATCH * 2;

__device__ __forceinline__ unsigned cell_hash(int cxc, int cyc) {
  return ((unsigned)cxc * 73856093u ^ (unsigned)cyc * 19349663u) & (unsigned)(GTBL - 1);
}

// The walk can be split over several launches (state[] = accepted so far, done flag, number of open
// slots; `first` starts it, `last` pads the slots that stay open), and a launch reads its candidates
// either straight from the sorted list (INDIRECT = false: ranks 0 .. npoints-1) or through a list of
// ranks (INDIRECT = true: ranks[0 .. *d_nranks-1], ascending) -- the candidates that the whole GPU
// found still uncovered on the featuremap (UncoveredOp below).  That is how the sparse part of the
// walk is kept short: with the features that survive a KLTReplaceLostFeatures call pre-stamped,
// nearly every candidate is covered from the start, and in KLTSelectGoodFeatures after the first
// ENFORCE_HEAD candidates.
static constexpr int ENFORCE_HEAD = 32768;

struct UncoveredOp {                              // for cub::DeviceSelect::If over ranks
  const int* sval; const unsigned* sidx; const unsigned char* fmap;
  int nxc, bx, by, step, W, min_eig;
  __device__ __forceinline__ bool operator()(const int& r) const {
    if (sval[r] < min_eig) return false;
    const unsigned id = sidx[r];
    const int cx = bx + (int)(id % (unsigned)nxc) * step, cy = by + (int)(id / (unsigned)nxc) * step;
    return fmap[(size_t)cy * W + cx] == 0;
  }
};

template <bool INDIRECT>
__global__ void __launch_bounds__(GB)
enforce_mindist_kernel(const int* __restrict__ sval, const unsigned* __restrict__ sidx,
                       const int* __restrict__ ranks, const int* __restrict__ d_nranks, int npoints,
                       int nxc, int bx, int by, int step, int W, int H,
                       unsigned char* fmap, int d, int min_eig, int overwrite_all,
                       int n, float* x, float* y, int* val, int* open_slots,
                       int* state, int first, int last) {
  extern __shared__ __align__(16) unsigned char enf_smem[];
  unsigned* s_xy = reinterpret_cast<unsigned*>(enf_smem);            // survivors of the batch in rank order (x | y << 16);
  unsigned* s_tbl = s_xy + GBATCH;                                   //   the accepted ones are compacted in place at the front
  unsigned* s_conf = s_tbl + GTBL;                                   // per survivor: which earlier ones of its group of 32 are within d
  unsigned* s_cell = s_conf + GBATCH;                                // per survivor: its cell of the hash grid (x | y << 16)
  unsigned short* s_r = reinterpret_cast<unsigned short*>(s_cell + GBATCH);   // rank - base of the survivors
  __shared__ int s_wcount[GB / 32];
  __shared__ int s_tmp, s_nacc, s_total, s_done;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const bool spaced = d >= 1;                    // d == 0 only excludes the pixel itself, and candidates are distinct
  const int cs = spaced ? d + 1 : 1;             // cell size of the hash grid

  if (INDIRECT) npoints = *d_nranks;
  int nopen = 0;
  bool done;
  if (first) {
    // open slots in ascending index (selectGoodFeatures.c:207-210)
    for (int b0 = 0; b0 < n; b0 += GB) {
      const int i = b0 + tid;
      const bool open = (i < n) && (overwrite_all || val[i] < 0);
      int cnt;
      const int pos = block_prefix(open ? 1 : 0, s_wcount, &s_tmp, &cnt);
      if (open) open_slots[nopen + pos] = i;
      nopen += cnt;
      __syncthreads();                           // s_wcount / s_tmp reuse
    }
    done = (nopen == 0);
    if (tid == 0) { s_total = 0; s_done = done; s_nacc = 0; }
  } else {
    nopen = state[2];
    done = (state[1] != 0);
    if (tid == 0) { s_total = state[0]; s_done = done; s_nacc = 0; }
  }
  __syncthreads();
  volatile unsigned char* vmap = fmap;

  // Batch size: gk = 1 (1024 candidates) while the map is still so empty that most candidates
  // survive it -- every survivor costs a turn of the sequential walk, and a stamp made after a small
  // batch saves the walk most of the neighbours ranked just behind the accepted one -- and gk = GK
  // (4096) once fewer than a quarter of a batch survive (then the per-batch latency dominates).
  // The size of a batch is fixed when its keys are fetched, one batch ahead.
  // keys of the first batch; thread t owns the list entries base + gk*t .. base + gk*t + gk-1
  int gk = (first && overwrite_all && !INDIRECT) ? 1 : GK;
  int nv[GK]; unsigned nid[GK];
#pragma unroll
  for (int j = 0; j < GK; ++j) {
    const int i = gk * tid + j;
    nv[j] = 0; nid[j] = 0;
    if (!done && j < gk && i < npoints) { const int r = INDIRECT ? ranks[i] : i; nv[j] = sval[r]; nid[j] = sidx[r]; }
  }
  int gk_next = gk, gk_want = gk;                // layout of the prefetched keys / size wanted for the batch after them

  for (int base = 0; base < npoints && !done; base += GB * gk, gk = gk_next) {
    const int total0 = s_total;                  // accepted before this batch (written two barriers ago,
                                                 // rewritten only after the next two)
    int cv[GK], cx[GK], cy[GK];
    bool alive[GK];
    size_t cell[GK];
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < GK; ++j) {
      cv[j] = nv[j];
      cx[j] = bx + (int)(nid[j] % (unsigned)nxc) * step;
      cy[j] = by + (int)(nid[j] / (unsigned)nxc) * step;
      cell[j] = (size_t)cy[j] * W + cx[j];
      alive[j] = (j < gk) && (base + gk * tid + j < npoints) && (cv[j] >= min_eig);
    }
    unsigned char m[GK];
#pragma unroll
    for (int j = 0; j < GK; ++j) m[j] = alive[j] ? vmap[cell[j]] : (unsigned char)1;
    // the next batch's keys do not depend on the map: fetch them behind the map reads
    gk_next = gk_want;
#pragma unroll
    for (int j = 0; j < GK; ++j) {
      const int i = base + GB * gk + gk_next * tid + j;
      nv[j] = 0; nid[j] = 0;
      if (j < gk_next && i < npoints) { const int r = INDIRECT ? ranks[i] : i; nv[j] = sval[r]; nid[j] = sidx[r]; }
    }
    if (spaced) {
#pragma unroll
      for (int k = 0; k < GTBL / GB; ++k) s_tbl[tid + k * GB] = GEMPTY;
    }
#pragma unroll
    for (int j = 0; j < GK; ++j) { alive[j] = alive[j] && (m[j] == 0); cnt += alive[j] ? 1 : 0; }
    int nsurv;
    int pos = block_prefix(cnt, s_wcount, &s_tmp, &nsurv);           // 2 barriers
#pragma unroll
    for (int j = 0; j < GK; ++j)
      if (alive[j]) { s_xy[pos] = (unsigned)cx[j] | ((unsigned)cy[j] << 16); s_r[pos] = (unsigned short)(gk * tid + j); ++pos; }
    gk_want = (nsurv * 4 > GB * gk) ? 1 : GK;     // (uniform: every thread sees the same nsurv)
    // the list is sorted descending: once the first candidate of a batch is
    // below the threshold nothing at or after it can be accepted
    if (tid == 0 && cv[0] < min_eig) s_done = 1;
    __syncthreads();
    // conflicts inside each group of 32 consecutive survivors: independent of what gets accepted,
    // so every warp prepares the groups g = wid, wid + 32, ... for the sequential walk of warp 0
    if (spaced) {
      for (int g0 = wid * 32; g0 < nsurv; g0 += GB) {
        const int s = g0 + lane;
        const unsigned pxy = s < nsurv ? s_xy[s] : 0u;
        const int px = (int)(pxy & 0xffffu), py = (int)(pxy >> 16);
        unsigned conf = 0;
#pragma unroll
        for (int i = 0; i < 31; ++i) {
          const unsigned q = __shfl_sync(0xffffffffu, pxy, i);
          const int dx = px - (int)(q & 0xffffu), dy = py - (int)(q >> 16);
          if (i < lane && dx <= d && dx >= -d && dy <= d && dy >= -d) conf |= 1u << i;
        }
        s_conf[s] = conf;
        s_cell[s] = (unsigned)(px / cs) | ((unsigned)(py / cs) << 16);
      }
      __syncthreads();
    }
    if (wid == 0) {
      const int budget = nopen - total0;
      int nacc = 0;
      for (int g0 = 0; g0 < nsurv && nacc < budget; g0 += 32) {
        const int s = g0 + lane;
        const bool valid = s < nsurv;
        const unsigned pxy = valid ? s_xy[s] : 0u;
        const unsigned short pr = valid ? s_r[s] : (unsigned short)0;
        const int px = (int)(pxy & 0xffffu), py = (int)(pxy >> 16);
        bool hit = !valid;
        unsigned conf = 0;                       // bit i: within d of lane i's survivor (i < lane)
        int pcx = 0, pcy = 0;
        if (spaced) {
          const unsigned pc = s_cell[s];
          pcx = (int)(pc & 0xffffu); pcy = (int)(pc >> 16);
          if (nacc > 0) {
            // the accepted of this batch: 3 x 3 cells around the survivor, linear probing
            unsigned h[9], e[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) { h[k] = cell_hash(pcx + k % 3 - 1, pcy + k / 3 - 1); e[k] = s_tbl[h[k]]; }
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              while (e[k] != GEMPTY) {
                const int dx = px - (int)(e[k] & 0xffffu), dy = py - (int)(e[k] >> 16);
                if (dx <= d && dx >= -d && dy <= d && dy >= -d) hit = true;
                h[k] = (h[k] + 1u) & (unsigned)(GTBL - 1);
                e[k] = s_tbl[h[k]];
              }
            }
          }
          conf = s_conf[s < GBATCH ? s : GBATCH - 1];
        }
        const unsigned cand = __ballot_sync(0xffffffffu, !hit);
        conf &= cand;
        unsigned acc = 0, und = cand;
        while (und != 0) {                       // the lowest undecided lane is decided in every round
          const bool mine = (und >> lane) & 1u;
          const bool rej = mine && (conf & acc) != 0;
          const bool ok = mine && !rej && (conf & und) == 0;
          const unsigned okm = __ballot_sync(0xffffffffu, ok), rejm = __ballot_sync(0xffffffffu, rej);
          acc |= okm;
          und &= ~(okm | rejm);
        }
        while (__popc(acc) > budget - nacc) acc &= ~(0x80000000u >> __clz(acc));   // list full: first ones in rank order
        if ((acc >> lane) & 1u) {
          const int p2 = nacc + __popc(acc & ((1u << lane) - 1u));   // p2 <= s: in-place compaction
          s_xy[p2] = pxy; s_r[p2] = pr;
          if (spaced) {
            unsigned hh = cell_hash(pcx, pcy);
            while (atomicCAS(&s_tbl[hh], GEMPTY, pxy) != GEMPTY) hh = (hh + 1u) & (unsigned)(GTBL - 1);
          }
        }
        nacc += __popc(acc);
        __syncwarp();
      }
      if (lane == 0) { s_nacc = nacc; s_total = total0 + nacc; if (total0 + nacc >= nopen) s_done = 1; }
    }
    __syncthreads();
    {
      const int nacc = s_nacc;
      for (int a = tid; a < nacc; a += GB) {     // the records of the accepted (:207-222)
        const int slot = open_slots[total0 + a];
        const unsigned q = s_xy[a];
        const int li = base + s_r[a];
        x[slot] = (float)(q & 0xffffu); y[slot] = (float)(q >> 16); val[slot] = sval[INDIRECT ? ranks[li] : li];
      }
      // stamps (:102-115).  One warp per accepted candidate; the (2d+1)^2 square is written as
      // 32-bit words -- lane = (row, word of the row), byte mask by position, red.or so that squares
      // which share a word cannot lose each other's bytes.  (Byte stores, one row per instruction,
      // made this loop 0.8 M warp instructions for 1024 accepted candidates: more than half of the
      // kernel on its single SM.)
      if (d >= 0) {
        unsigned* fmap32 = reinterpret_cast<unsigned*>(fmap);
        for (int a = wid; a < nacc; a += GB / 32) {
          const unsigned q = s_xy[a];
          const int cx0 = (int)(q & 0xffffu), cy0 = (int)(q >> 16);
          const int xa = max(cx0 - d, 0), xb = min(cx0 + d, W - 1);          // clipped column range, inclusive
          const int ya = max(cy0 - d, 0), yb = min(cy0 + d, H - 1);
          const int nw = (xb - xa + 1 + 3) / 4 + 1;                            // words a row can touch, whatever its alignment
          const int items = (yb - ya + 1) * nw;
          const float inv = 1.0f / (float)nw;
          for (int it = lane; it < items; it += 32) {
            int r = (int)(((float)it + 0.5f) * inv);                           // it / nw (exact for these sizes, checked below)
            int k = it - r * nw;
            if (k < 0) { --r; k += nw; } else if (k >= nw) { ++r; k -= nw; }
            const size_t b0 = (size_t)(ya + r) * W + xa, b1 = b0 + (size_t)(xb - xa);   // first / last byte of the row
            const size_t w = (b0 >> 2) + k;
            if (w > (b1 >> 2)) continue;
            const int lo = (w == (b0 >> 2)) ? (int)(b0 & 3) : 0, hi = (w == (b1 >> 2)) ? (int)(b1 & 3) : 3;
            const unsigned mask = (0x01010101u >> (8 * (3 - (hi - lo)))) << (8 * lo);
            atomicOr(fmap32 + w, mask);
          }
        }
      }
      done = (s_done != 0);
    }
    __syncthreads();      // stamps visible to the next batch; s_done / s_total stable while read
  }
  const int total = s_total;
  if (!last) {
    if (tid == 0) { state[0] = total; state[1] = done ? 1 : 0; state[2] = nopen; }
    return;
  }
  // out of candidates: the still-open slots become NOT_FOUND (:175-195)
  for (int k = total + tid; k < nopen; k += GB) {
    const int slot = open_slots[k];
    x[slot] = -1.0f; y[slot] = -1.0f; val[slot] = KLT_NOT_FOUND;
  }
}

// ---------------------------------------------------------------------------
// tracker: one warp per feature, coarse to fine, all levels in one launch
// ---------------------------------------------------------------------------
struct PyrView {
  const float* img[KLT_DEV_MAX_LEVELS];
  const float* gx[KLT_DEV_MAX_LEVELS];
  const float* gy[KLT_DEV_MAX_LEVELS];
  int ncols[KLT_DEV_MAX_LEVELS], nrows[KLT_DEV_MAX_LEVELS], pitch[KLT_DEV_MAX_LEVELS];
};

struct TrackArgs {
  int   nlevels;
  float ss;
  int   ww, wh;
  float step_factor;
  int   max_iterations;
  float min_determinant, min_displacement, max_residue;
  int   borderx, bordery;
  int   ncols, nrows;
  int   lighting;            // tc->lighting_insensitive: gain / bias normalised windows (track_kernel only)
  int   l2_keep;             // track7w: the new frame's footprints are loaded with an L2 evict_last policy
};

// Where a tracker kernel reads the features and where it records the results (element strides in
// 4-byte words): SoA device arrays (stride 1), the pinned SoA staging area, or -- for feature lists
// that live in pinned host memory -- a device mirror of the KLT_FeatureRec array for the input and
// the caller's own records for the output (stride = sizeof(KLT_FeatureRec) / 4, x | y | val at
// words 0 | 1 | 2), so that the synchronous API needs no pack / unpack pass on the host.
struct FeatIO {
  const float* x; const float* y; const int* val; int istride;
  float* ox; float* oy; int* oval; int ostride;
};

// Forward-backward check, one record per feature of the last tracking call (klt_dev_fb_results):
// where the backward leg from frame 2 into frame 1 ended, its distance from the start position and
// its status; (-1, -1, -1, 1) for a feature the check did not run on.
struct __align__(16) FbRec { float xb, yb, err; int back_val; };
// The check's kernel argument, the trackers' last: the records and the largest round-trip distance
// kept.  (Last, and not in TrackArgs, so that the parameter layout of the FB = false kernels is the
// one they have without the check.)
struct FbArgs { FbRec* rec; float max_error; };

// value and position the tracker records for a feature (:1383-1437): the final border test
__device__ __forceinline__ int track_outcome(const TrackArgs& a, int status, float x, float y) {
  const bool outside = (x < (float)a.borderx || x > (float)(a.ncols - 1 - a.borderx) ||
                        y < (float)a.bordery || y > (float)(a.nrows - 1 - a.bordery));
  return (status == KLT_OOB || outside) ? KLT_OOB : status;
}
__device__ __forceinline__ void record_feature(const FeatIO& io, int f, int v, float x, float y) {
  const size_t o = (size_t)f * io.ostride;
  if (v != KLT_TRACKED) { io.ox[o] = -1.0f; io.oy[o] = -1.0f; io.oval[o] = v; }
  else { io.ox[o] = x; io.oy[o] = y; io.oval[o] = KLT_TRACKED; }
}
// The decision of the check, in separately rounded float32 in both arithmetic modes: the feature is
// kept when the backward leg tracked and !(d2 > max_error^2).  Fills the feature's record.
__device__ __forceinline__ bool fb_keep(float max_error, float x0, float y0, float xb, float yb, int back_val,
                                        FbRec& r) {
  r.back_val = back_val;
  if (back_val != KLT_TRACKED) { r.xb = -1.0f; r.yb = -1.0f; r.err = -1.0f; return false; }
  const float dx = __fsub_rn(xb, x0), dy = __fsub_rn(yb, y0);
  const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
  r.xb = xb; r.yb = yb; r.err = __fsqrt_rn(d2);
  return !(d2 > __fmul_rn(max_error, max_error));
}
__device__ __forceinline__ FbRec fb_unchecked() {
  FbRec r;
  r.xb = -1.0f; r.yb = -1.0f; r.err = -1.0f; r.back_val = 1;
  return r;
}

// Motion prior: a per-feature guess g of the frame-2 position, where the descent starts instead of
// at the feature's own position.  Velocity record of a feature index, written by every tracker that
// runs with the prior: {xout, yout, xout - x0, yout - y0} for a KLT_TRACKED result (after the
// forward-backward check), px = NaN (invalid) for any other.
struct __align__(16) PredVel { float px, py, dx, dy; };
// Per feature of the last call (klt_dev_prediction_results): the guess and where it came from
// (PRED_NONE: (-1, -1)).
enum { PRED_NONE = 0, PRED_VELOCITY = 1, PRED_EXPLICIT = 2 };
struct PredRec { float gx, gy; int source; };
// The prior's kernel argument, after FbArgs (so that the PRED = false kernels keep their layout):
// explicit guesses of this call (NaN: none for that feature; gx == nullptr: none at all), the velocity
// records (read for f < vel_n; vel_n = 0 when velocity prediction is off or no record is valid) and
// the result records.
struct PredArgs { const float* gx; const float* gy; PredVel* vel; PredRec* rec; int vel_n; };

// The start of feature f's forward leg (input position (x0, y0), input status val_in) at the coarsest
// level: {x0, y0, gx, gy}, the guess g being (x0, y0) without one.  Records the guess in rec[f].  Run
// by one lane of the feature's group before the descent.  Out of line and with scalar arguments: the
// division's slow path is a call, and inlined, the values live across those calls make the PRED
// kernels spill; across this one call only what the FB kernels keep across theirs is live.
__device__ __noinline__ float4 pred_start(const float* egx, const float* egy, const PredVel* vel, PredRec* rec,
                                          int vel_n, int nlevels, float ss, int f, int val_in, float x0, float y0) {
  int src = PRED_NONE;
  float gx = x0, gy = y0;
  if (egx && isfinite(egx[f]) && isfinite(egy[f])) {
    gx = egx[f]; gy = egy[f]; src = PRED_EXPLICIT;
  } else if (val_in == KLT_TRACKED && f < vel_n) {
    const PredVel v = vel[f];
    if (x0 == v.px && y0 == v.py) { gx = __fadd_rn(x0, v.dx); gy = __fadd_rn(y0, v.dy); src = PRED_VELOCITY; }
  }
  PredRec r;
  r.gx = src ? gx : -1.0f; r.gy = src ? gy : -1.0f; r.source = src;
  rec[f] = r;
  float4 c = make_float4(x0, y0, gx, gy);
  for (int l = nlevels - 1; l >= 0; --l) {        // divided by ss once per level, as the descent divides the start
    c.x = __fdiv_rn(c.x, ss); c.y = __fdiv_rn(c.y, ss); c.z = __fdiv_rn(c.z, ss); c.w = __fdiv_rn(c.w, ss);
  }
  return c;
}
// The start of the backward leg from (xout, yout) at the coarsest level: {xout, yout, gbx, gby}, with the
// mirrored prior gb = xout - (g - x0) when the forward leg used a guess g (read back from rec[f]), else
// gb = xout.
__device__ __noinline__ float4 pred_back_start(const PredRec* rec, int nlevels, float ss, int f, float x0, float y0,
                                               float xout, float yout) {
  const PredRec r = rec[f];
  float4 c = make_float4(xout, yout, xout, yout);
  if (r.source != PRED_NONE) { c.z = __fsub_rn(xout, __fsub_rn(r.gx, x0)); c.w = __fsub_rn(yout, __fsub_rn(r.gy, y0)); }
  for (int l = nlevels - 1; l >= 0; --l) {
    c.x = __fdiv_rn(c.x, ss); c.y = __fdiv_rn(c.y, ss); c.z = __fdiv_rn(c.z, ss); c.w = __fdiv_rn(c.w, ss);
  }
  return c;
}
__device__ __forceinline__ float4 shfl4(float4 c, int width) {
  c.x = __shfl_sync(0xffffffffu, c.x, 0, width); c.y = __shfl_sync(0xffffffffu, c.y, 0, width);
  c.z = __shfl_sync(0xffffffffu, c.z, 0, width); c.w = __shfl_sync(0xffffffffu, c.w, 0, width);
  return c;
}
// Velocity record of feature f after its call, from its result v before the affine check.  (x0, y0)
// is read again from the input rather than kept in registers across the descent.
__device__ __forceinline__ void pred_velocity(const PredArgs& pr, const FeatIO& io, int f, int v,
                                              float xout, float yout) {
  PredVel w;
  if (v == KLT_TRACKED) {
    w.px = xout; w.py = yout;
    w.dx = __fsub_rn(xout, io.x[(size_t)f * io.istride]); w.dy = __fsub_rn(yout, io.y[(size_t)f * io.istride]);
  } else {
    w.px = __int_as_float(0x7fffffff); w.py = w.px; w.dx = 0.0f; w.dy = 0.0f;
  }
  pr.vel[f] = w;
}
// a feature the tracker does not run on: no guess, no velocity
__device__ __forceinline__ void pred_skip(const PredArgs& pr, int f) {
  PredRec r;
  r.gx = -1.0f; r.gy = -1.0f; r.source = PRED_NONE;
  pr.rec[f] = r;
  PredVel w;
  w.px = __int_as_float(0x7fffffff); w.py = w.px; w.dx = 0.0f; w.dy = 0.0f;
  pr.vel[f] = w;
}

// bilinear weights of _interpolate (trackFeatures.c:31-57): the four products
// (1-ax)(1-ay), ax(1-ay), (1-ax)ay, ax*ay are rounded first, then multiplied by
// the pixels and summed left to right.
struct Bilin {
  int   off;                 // yt * pitch + xt
  float w00, w01, w10, w11;
};
template <bool EXACT>
__device__ __forceinline__ Bilin bilin_setup(float x, float y, int pitch) {
  const int xt = (int)x, yt = (int)y;
  const float ax = __fsub_rn(x, (float)xt), ay = __fsub_rn(y, (float)yt);
  const float omx = __fsub_rn(1.0f, ax), omy = __fsub_rn(1.0f, ay);
  Bilin b;
  b.off = yt * pitch + xt;
  b.w00 = __fmul_rn(omx, omy);
  b.w01 = __fmul_rn(ax, omy);
  b.w10 = __fmul_rn(omx, ay);
  b.w11 = __fmul_rn(ax, ay);
  return b;
}
template <bool EXACT>
__device__ __forceinline__ float bilin_fetch(const float* __restrict__ img, int pitch, const Bilin& b) {
  const float* p = img + b.off;
  const float p00 = __ldg(p), p01 = __ldg(p + 1), p10 = __ldg(p + pitch), p11 = __ldg(p + pitch + 1);
  if (EXACT) {
    float s = __fmul_rn(b.w00, p00);
    s = __fadd_rn(s, __fmul_rn(b.w01, p01));
    s = __fadd_rn(s, __fmul_rn(b.w10, p10));
    s = __fadd_rn(s, __fmul_rn(b.w11, p11));
    return s;
  }
  return fmaf(b.w11, p11, fmaf(b.w10, p10, fmaf(b.w01, p01, b.w00 * p00)));
}

__device__ __forceinline__ bool window_oob(float x, float y, int hw, int hh, int nc, int nr) {
  // trackFeatures.c:418-425, one_plus_eps = 1.001f
  return (__fsub_rn(x, (float)hw) < 0.0f || __fsub_rn((float)nc, __fadd_rn(x, (float)hw)) < 1.001f ||
          __fsub_rn(y, (float)hh) < 0.0f || __fsub_rn((float)nr, __fadd_rn(y, (float)hh)) < 1.001f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Gain / bias of the lighting-insensitive windows (trackFeatures.c:132-167, :178-220) from the
// window samples g1 (frame 1) and g2 (frame 2):
//   alpha  = sqrt(mean(g1^2) / mean(g2^2)),  belta = mean(g1) - alpha * mean(g2)   (intensity difference)
//   alphag = sqrt(mean(g1) / mean(g2))                                             (gradient sum: the
//            reference accumulates g, not g*g, in its "sum*_squared" variables, :202 -- kept as it is)
// EXACT: the four sums run sequentially in raster order, one per lane, over the shared arrays.
struct LiGain { float alpha, belta, alphag; };
template <bool EXACT, int PPL>
__device__ __forceinline__ LiGain li_gain(const float (&g1)[PPL], const float (&g2)[PPL], int lane, int npix,
                                          float* sa, float* sb) {
  float s1 = 0.0f, s2 = 0.0f, q1 = 0.0f, q2 = 0.0f;
  if (EXACT) {
#pragma unroll
    for (int k = 0; k < PPL; ++k) {
      const int p = lane + 32 * k;
      if (p < npix) { sa[p] = g1[k]; sb[p] = g2[k]; }
    }
    __syncwarp();
    float acc = 0.0f;
    if (lane < 4) {
      const float* A = (lane & 1) ? sb : sa;
      if (lane < 2) { for (int p = 0; p < npix; ++p) acc = __fadd_rn(acc, A[p]); }
      else          { for (int p = 0; p < npix; ++p) acc = __fadd_rn(acc, __fmul_rn(A[p], A[p])); }
    }
    s1 = __shfl_sync(0xffffffffu, acc, 0); s2 = __shfl_sync(0xffffffffu, acc, 1);
    q1 = __shfl_sync(0xffffffffu, acc, 2); q2 = __shfl_sync(0xffffffffu, acc, 3);
    __syncwarp();
  } else {
#pragma unroll
    for (int k = 0; k < PPL; ++k) {
      if (lane + 32 * k < npix) { s1 += g1[k]; s2 += g2[k]; q1 = fmaf(g1[k], g1[k], q1); q2 = fmaf(g2[k], g2[k], q2); }
    }
    s1 = warp_sum(s1); s2 = warp_sum(s2); q1 = warp_sum(q1); q2 = warp_sum(q2);
  }
  const float n = (float)npix;
  LiGain g;
  g.alpha = (float)sqrt((double)__fdiv_rn(__fdiv_rn(q1, n), __fdiv_rn(q2, n)));
  const float m1 = __fdiv_rn(s1, n), m2 = __fdiv_rn(s2, n);
  g.belta = __fsub_rn(m1, __fmul_rn(g.alpha, m2));
  g.alphag = (float)sqrt((double)__fdiv_rn(m1, m2));
  return g;
}

// PPL = window pixels per lane (ceil(ww*wh / 32)); the frame-1 samples of the
// window are constant while a level iterates, so they are sampled once per
// level and kept in registers.
// The pyramid descent of one feature from (x, y) in p1's frame into p2's frame (:1343-1378): the
// status of the finest level reached and the end position (xend, yend), before the border test.
// G: (x, y) and the guess (gx, gy) the descent starts from are given at the coarsest level (pred_start);
// a guess equal to the start gives the descent without one.
template <bool EXACT, int PPL, bool G = false>
__device__ __forceinline__ int track_descent(const PyrView& p1, const PyrView& p2, const TrackArgs& a, int lane,
                                             const float (&offi)[PPL], const float (&offj)[PPL],
                                             float* swx, float* swy, float* swd,
                                             float x, float y, float& xend, float& yend,
                                             float gx = 0.0f, float gy = 0.0f) {
  const int ww = a.ww, wh = a.wh, hw = ww / 2, hh = wh / 2, npix = ww * wh;
  float xloc = x, yloc = y;
  if (!G)
    for (int r = a.nlevels - 1; r >= 0; --r) { xloc = __fdiv_rn(xloc, a.ss); yloc = __fdiv_rn(yloc, a.ss); }
  float xout = G ? gx : xloc, yout = G ? gy : yloc;
  int status = KLT_TRACKED;

  for (int r = a.nlevels - 1; r >= 0; --r) {
    xloc = __fmul_rn(xloc, a.ss); yloc = __fmul_rn(yloc, a.ss);
    xout = __fmul_rn(xout, a.ss); yout = __fmul_rn(yout, a.ss);
    const int nc = p1.ncols[r], nr = p1.nrows[r], pitch = p1.pitch[r];
    const float* __restrict__ i1 = p1.img[r];
    const float* __restrict__ gx1 = p1.gx[r];
    const float* __restrict__ gy1 = p1.gy[r];
    const float* __restrict__ i2 = p2.img[r];
    const float* __restrict__ gx2 = p2.gx[r];
    const float* __restrict__ gy2 = p2.gy[r];

    // ---- _trackFeature (trackFeatures.c:381-486) at this level -------------
    const float x1 = xloc, y1 = yloc;
    float x2 = xout, y2 = yout;
    int iteration = 0;
    float dx = 0.0f, dy = 0.0f;
    float t_i[PPL], t_gx[PPL], t_gy[PPL];
    bool have_template = false;
    const bool oob1 = window_oob(x1, y1, hw, hh, nc, nr);

    do {
      if (oob1 || window_oob(x2, y2, hw, hh, nc, nr)) { status = KLT_OOB; break; }
      if (!have_template) {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          if (lane + 32 * k < npix) {
            const Bilin b = bilin_setup<EXACT>(__fadd_rn(x1, offi[k]), __fadd_rn(y1, offj[k]), pitch);
            t_i[k] = bilin_fetch<EXACT>(i1, pitch, b);
            t_gx[k] = bilin_fetch<EXACT>(gx1, pitch, b);
            t_gy[k] = bilin_fetch<EXACT>(gy1, pitch, b);
          } else { t_i[k] = 0.0f; t_gx[k] = 0.0f; t_gy[k] = 0.0f; }
        }
        have_template = true;
      }
      float gxx = 0.0f, gxy = 0.0f, gyy = 0.0f, ex = 0.0f, ey = 0.0f;
      float s_i2[PPL], s_gx2[PPL], s_gy2[PPL];      // frame-2 samples (lighting-insensitive mode)
      LiGain lg;
      lg.alpha = 1.0f; lg.belta = 0.0f; lg.alphag = 1.0f;
      if (a.lighting) {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          s_i2[k] = 0.0f; s_gx2[k] = 0.0f; s_gy2[k] = 0.0f;
          if (lane + 32 * k < npix) {
            const Bilin b = EXACT ? bilin_setup<EXACT>(__fadd_rn(x2, offi[k]), __fadd_rn(y2, offj[k]), pitch)
                                  : bilin_setup<EXACT>(x2 + offi[k], y2 + offj[k], pitch);
            s_i2[k] = bilin_fetch<EXACT>(i2, pitch, b);
            s_gx2[k] = bilin_fetch<EXACT>(gx2, pitch, b);
            s_gy2[k] = bilin_fetch<EXACT>(gy2, pitch, b);
          }
        }
        lg = li_gain<EXACT, PPL>(t_i, s_i2, lane, npix, swx, swy);
      }
      if (EXACT) {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          const int p = lane + 32 * k;
          if (p < npix) {
            if (a.lighting) {          // g1 - g2*alpha - belta;  g1 + g2*alphag   (:165, :213-216)
              swd[p] = __fsub_rn(__fsub_rn(t_i[k], __fmul_rn(s_i2[k], lg.alpha)), lg.belta);
              swx[p] = __fadd_rn(t_gx[k], __fmul_rn(s_gx2[k], lg.alphag));
              swy[p] = __fadd_rn(t_gy[k], __fmul_rn(s_gy2[k], lg.alphag));
            } else {
              const Bilin b = bilin_setup<EXACT>(__fadd_rn(x2, offi[k]), __fadd_rn(y2, offj[k]), pitch);
              swd[p] = __fsub_rn(t_i[k], bilin_fetch<EXACT>(i2, pitch, b));
              swx[p] = __fadd_rn(t_gx[k], bilin_fetch<EXACT>(gx2, pitch, b));
              swy[p] = __fadd_rn(t_gy[k], bilin_fetch<EXACT>(gy2, pitch, b));
            }
          }
        }
        __syncwarp();
        // five sequential raster-order sums, one per lane (:227-279)
        float acc = 0.0f;
        if (lane < 5) {
          const float* A = (lane <= 1) ? swx : (lane == 2 ? swy : swd);
          const float* B = (lane == 0 || lane == 3) ? swx : swy;
          for (int p = 0; p < npix; ++p) acc = __fadd_rn(acc, __fmul_rn(A[p], B[p]));
        }
        gxx = __shfl_sync(0xffffffffu, acc, 0);
        gxy = __shfl_sync(0xffffffffu, acc, 1);
        gyy = __shfl_sync(0xffffffffu, acc, 2);
        ex = __shfl_sync(0xffffffffu, acc, 3);
        ey = __shfl_sync(0xffffffffu, acc, 4);
        __syncwarp();
      } else {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          if (lane + 32 * k < npix) {
            float df, sx, sy;
            if (a.lighting) {
              df = t_i[k] - s_i2[k] * lg.alpha - lg.belta;
              sx = fmaf(s_gx2[k], lg.alphag, t_gx[k]);
              sy = fmaf(s_gy2[k], lg.alphag, t_gy[k]);
            } else {
              const Bilin b = bilin_setup<EXACT>(x2 + offi[k], y2 + offj[k], pitch);
              df = t_i[k] - bilin_fetch<EXACT>(i2, pitch, b);
              sx = t_gx[k] + bilin_fetch<EXACT>(gx2, pitch, b);
              sy = t_gy[k] + bilin_fetch<EXACT>(gy2, pitch, b);
            }
            gxx = fmaf(sx, sx, gxx); gxy = fmaf(sx, sy, gxy); gyy = fmaf(sy, sy, gyy);
            ex = fmaf(df, sx, ex); ey = fmaf(df, sy, ey);
          }
        }
        gxx = warp_sum(gxx); gxy = warp_sum(gxy); gyy = warp_sum(gyy);
        ex = warp_sum(ex); ey = warp_sum(ey);
      }
      ex = __fmul_rn(ex, a.step_factor);
      ey = __fmul_rn(ey, a.step_factor);
      // _solveEquation (:293-307)
      const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));
      if (det < a.min_determinant) { status = KLT_SMALL_DET; break; }
      dx = __fdiv_rn(__fsub_rn(__fmul_rn(gyy, ex), __fmul_rn(gxy, ey)), det);
      dy = __fdiv_rn(__fsub_rn(__fmul_rn(gxx, ey), __fmul_rn(gxy, ex)), det);
      status = KLT_TRACKED;
      x2 = __fadd_rn(x2, dx);
      y2 = __fadd_rn(y2, dy);
      ++iteration;
    } while ((fabsf(dx) >= a.min_displacement || fabsf(dy) >= a.min_displacement) &&
             iteration < a.max_iterations);

    // :459-462
    if (window_oob(x2, y2, hw, hh, nc, nr)) status = KLT_OOB;

    // :464-474 residue of the final alignment
    if (status == KLT_TRACKED) {
      float sum = 0.0f;
      float r_i2[PPL];
      LiGain lg;
      lg.alpha = 1.0f; lg.belta = 0.0f; lg.alphag = 1.0f;
      if (a.lighting) {                 // the residue uses the normalised difference too (:466-468)
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          r_i2[k] = 0.0f;
          if (lane + 32 * k < npix) {
            const Bilin b = EXACT ? bilin_setup<EXACT>(__fadd_rn(x2, offi[k]), __fadd_rn(y2, offj[k]), pitch)
                                  : bilin_setup<EXACT>(x2 + offi[k], y2 + offj[k], pitch);
            r_i2[k] = bilin_fetch<EXACT>(i2, pitch, b);
          }
        }
        lg = li_gain<EXACT, PPL>(t_i, r_i2, lane, npix, swx, swy);
      }
      if (EXACT) {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          const int p = lane + 32 * k;
          if (p < npix) {
            if (a.lighting) {
              swd[p] = fabsf(__fsub_rn(__fsub_rn(t_i[k], __fmul_rn(r_i2[k], lg.alpha)), lg.belta));
            } else {
              const Bilin b = bilin_setup<EXACT>(__fadd_rn(x2, offi[k]), __fadd_rn(y2, offj[k]), pitch);
              swd[p] = fabsf(__fsub_rn(t_i[k], bilin_fetch<EXACT>(i2, pitch, b)));
            }
          }
        }
        __syncwarp();
        if (lane == 0)
          for (int p = 0; p < npix; ++p) sum = __fadd_rn(sum, swd[p]);
        sum = __shfl_sync(0xffffffffu, sum, 0);
        __syncwarp();
      } else {
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
          if (lane + 32 * k < npix) {
            if (a.lighting) {
              sum += fabsf(t_i[k] - r_i2[k] * lg.alpha - lg.belta);
            } else {
              const Bilin b = bilin_setup<EXACT>(x2 + offi[k], y2 + offj[k], pitch);
              sum += fabsf(t_i[k] - bilin_fetch<EXACT>(i2, pitch, b));
            }
          }
        }
        sum = warp_sum(sum);
      }
      if (__fdiv_rn(sum, (float)npix) > a.max_residue) status = KLT_LARGE_RESIDUE;
    }

    // :479-484 return value of _trackFeature
    int v;
    if (status == KLT_SMALL_DET) v = KLT_SMALL_DET;
    else if (status == KLT_OOB) v = KLT_OOB;
    else if (status == KLT_LARGE_RESIDUE) v = KLT_LARGE_RESIDUE;
    else if (iteration >= a.max_iterations) v = KLT_MAX_ITERATIONS;
    else v = KLT_TRACKED;
    status = v;
    xout = x2; yout = y2;
    if (v == KLT_SMALL_DET || v == KLT_OOB) break;      // :1378
  }
  xend = xout; yend = yout;
  return status;
}

// FB: the forward-backward check runs in the same warp after the forward leg (klt_dev_fb_results)
// PRED: the descent starts from the feature's guess (PredArgs, klt_dev_prediction_results)
template <bool EXACT, int PPL, bool FB, bool PRED = false>
__global__ void __launch_bounds__(128)
track_kernel(PyrView p1, PyrView p2, TrackArgs a, int n, FeatIO io,
             unsigned long long* __restrict__ live_total, FbArgs fb, PredArgs pr) {
  extern __shared__ float s_win[];     // EXACT only: [warps][3][npix]
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int f = blockIdx.x * (blockDim.x >> 5) + wib;
  if (f >= n) return;
  const int val_in = io.val[(size_t)f * io.istride];
  if (val_in < 0) {                                           // only features that are not lost (:1346)
    if (FB && lane == 0) fb.rec[f] = fb_unchecked();
    if (PRED && lane == 0) pred_skip(pr, f);
    return;
  }
  if (lane == 0) atomicAdd(live_total, 1ULL);

  const int ww = a.ww, wh = a.wh, hw = ww / 2, hh = wh / 2, npix = ww * wh;
  float* swx = s_win + (size_t)wib * 3 * npix;
  float* swy = swx + npix;
  float* swd = swy + npix;

  // per-lane window offsets (raster order: pixel p -> (i,j) = (p % ww - hw, p / ww - hh))
  float offi[PPL], offj[PPL];
#pragma unroll
  for (int k = 0; k < PPL; ++k) {
    const int p = lane + 32 * k;
    const int pp = p < npix ? p : 0;
    offi[k] = (float)(pp % ww - hw);
    offj[k] = (float)(pp / ww - hh);
  }

  const float x0 = io.x[(size_t)f * io.istride], y0 = io.y[(size_t)f * io.istride];
  float4 s0 = make_float4(x0, y0, 0.0f, 0.0f);              // PRED: start and guess at the coarsest level
  if (PRED) {
    if (lane == 0) s0 = pred_start(pr.gx, pr.gy, pr.vel, pr.rec, pr.vel_n, a.nlevels, a.ss, f, val_in, x0, y0);
    s0 = shfl4(s0, 32);
  }
  float xout, yout;
  int v = track_outcome(a, track_descent<EXACT, PPL, PRED>(p1, p2, a, lane, offi, offj, swx, swy, swd, s0.x, s0.y,
                                                           xout, yout, s0.z, s0.w), xout, yout);
  if (FB) {
    FbRec r = fb_unchecked();
    if (v == KLT_TRACKED) {                                   // the backward leg: frame 2 into frame 1
      float xb, yb;
      float4 sb = make_float4(xout, yout, 0.0f, 0.0f);        // PRED: from the mirrored prior
      if (PRED) {
        if (lane == 0) sb = pred_back_start(pr.rec, a.nlevels, a.ss, f, x0, y0, xout, yout);
        sb = shfl4(sb, 32);
      }
      const int vb = track_outcome(a, track_descent<EXACT, PPL, PRED>(p2, p1, a, lane, offi, offj, swx, swy, swd,
                                                                      sb.x, sb.y, xb, yb, sb.z, sb.w), xb, yb);
      if (!fb_keep(fb.max_error, x0, y0, xb, yb, vb, r)) v = KLT_B200_FB_INCONSISTENT;
    }
    if (lane == 0) fb.rec[f] = r;
  }
  if (PRED && lane == 0) pred_velocity(pr, io, f, v, xout, yout);
  if (lane == 0) record_feature(io, f, v, xout, yout);     // record (:1383-1437)
}

#include "klt_track_fast.cuh"

#include "klt_affine.cuh"

// ---------------------------------------------------------------------------
// host side of the C-ABI
// ---------------------------------------------------------------------------
// kernel classes, for launch accounting and per-kernel event timing
enum KernelId {
  KID_SMOOTH_U8 = 0, KID_GRAD, KID_PYRDOWN, KID_TRACK, KID_MINEIG, KID_SORT, KID_STAMP,
  KID_ENFORCE, KID_GENERIC_H, KID_GENERIC_V, KID_U8_TO_F32, KID_L0_FUSED, KID_LEVEL_FUSED, KID_LEVEL_FUSED_L2, KID_LEVEL_FUSED_L3, KID_TRACK_FAST, KID_TRACK7W, KID_AFFINE, KID_FILTER, KID_COPY_H2D, KID_COPY_D2H, KID_COUNT
};
static const char* const kKernelNames[KID_COUNT] = {
  "smooth_u8_tile", "grad_tile", "pyrdown_tile", "track_kernel", "mineig_kernel",
  "cub_radix_sort", "stamp_existing_kernel", "enforce_mindist_kernel",
  "conv_h_generic", "conv_v_generic", "u8_to_f32_kernel", "l0_fused_kernel", "level_fused_kernel[level 1]", "level_fused_kernel[level 2]", "level_fused_kernel[level 3+]", "track_fast_kernel", "track7w_kernel", "affine_check_kernel", "cub_select_uncovered",
  "copy_h2d", "copy_d2h"          // not kernels: timed in profiling mode, never counted as launches
};
static constexpr int PROF_POOL = 2048;     // event pairs in flight before folding
static constexpr int TRACE_CAP = 8192;     // timeline records kept per profiling session
static constexpr int KLT_BAND_EVENTS = 64; // events cycled by the banded frame upload

static constexpr int KLT_SNAP_MAX = 64;
static constexpr int KLT_HOST_REGS = 32; // pageable frame buffers remembered per context
static constexpr int KLT_TILE_QUEUES = 16;
static_assert(KLT_DEV_MAX_LEVELS <= KLT_TILE_QUEUES, "one tile queue per pyramid level");
struct Level {
  int w, h, pitch;           // pitch in floats
  float *img, *gx, *gy;
};
struct PyrSet {
  Level lv[KLT_DEV_MAX_LEVELS];
  int built_levels;          // 0 = nothing valid
  double grad_bound;         // upper bound of |gx|, |gy| at level 0 (from the taps, 8-bit input); 0 = unknown
  // what the set was built from: the device copy of the u8 frame (ours: d->frame_buf[i], or the
  // caller's device frame) and the build parameters -- klt_dev_exact_level0 rebuilds level 0 from them
  const unsigned char* src; int spitch;
  klt_dev_build_desc desc;
};

struct klt_dev {
  int device, num_sms;
  cudaStream_t stream;        // frame upload, pyramid kernels, selection
  cudaStream_t tstream;       // tracker + feature copies; == stream unless overlap is on
  cudaStream_t stream2;       // the second stream object (owned)
  int overlap;                // 1: tracker of frame k runs concurrently with the build of frame k+1
  cudaEvent_t ev_built[KLT_DEV_SLOTS];   // build of the slot finished (recorded on stream)
  cudaEvent_t ev_read[KLT_DEV_SLOTS];    // last tracker reading the slot finished (recorded on tstream)
  int read_pending[KLT_DEV_SLOTS], built_pending[KLT_DEV_SLOTS];
  cudaEvent_t ev_join;
  char err[512];
  unsigned long long launches;
  int last_path, force_generic, no_fused, last_fused, track7_off;
  // geometry
  int W, H, L, ss;
  PyrSet set[KLT_DEV_SLOTS];
  float* arena;
  size_t arena_floats;
  int guard;                 // debug: canary bands between the planes of the arena (klt_dev_set_guard)
  struct Guarded { void* user; size_t bytes; } guarded[24]; int nguarded;   // ... and around the selection / feature buffers
  float* tmp;                // generic path: horizontal-pass result, W*H floats
  unsigned char* frame;      // u8 staging of the frame being built (== frame_buf[frame_idx]), row pitch frame_pitch
  unsigned char* frame_buf[2]; int frame_idx;   // two buffers: frame k+1 goes up while level 0 of frame k is still reading
  size_t frame_cap; int frame_pitch;
  // banded upload of host frames: copy stream, one event per band, "staging consumed" event
  cudaStream_t cstream;
  cudaEvent_t ev_band[KLT_BAND_EVENTS]; int band_ev_next;
  cudaEvent_t ev_frame_free[2]; int frame_busy[2];   // per staging buffer
  int band_rows, last_bands, building_slot;
  // pageable host frames: parallel memcpy into pinned staging, chunk by chunk ahead of the DMA
  unsigned char* h_frame; size_t h_frame_cap; cudaEvent_t ev_stage_free; int stage_busy, stage_threads, last_staged;
  // pageable frame buffers the caller keeps handing in (a driver that reuses its two malloc'ed images,
  // reference src/V3/example3.c:45-46,75) are page-locked in place on second sight: the DMA then reads
  // them directly and the staging copy disappears.  Released by klt_dev_forget_host_frames / destroy.
  struct HostReg { const void* p; size_t bytes; int seen; int registered; unsigned long long stamp; } hreg[KLT_HOST_REGS];
  int reg_frames; unsigned long long reg_clock; int last_registered;
  int pdl;                     // programmatic dependent launch along the per-frame kernel chain
  // features
  float *d_x, *d_y; int* d_val; int feat_cap; int feat_n;
  float *h_x, *h_y; int* h_val;   // pinned staging
  int staging_busy;
  int no_track7w;
  int feat_out_host;            // 1: the next tracker writes its results into h_x/h_y/h_val (sync API); 2: record mode
  unsigned char* d_rec; size_t d_rec_cap; void* h_rec; int rec_stride;   // record mode (klt_dev_features_commit_records)
  cudaEvent_t ev_feat; int feat_pending;   // feature upload queued on the copy stream
  // ... or not queued yet: it goes BEHIND the bands of the frame that is built next (feat_flush)
  int feat_deferred; void* feat_def_dst; const void* feat_def_src; size_t feat_def_bytes;
  // affine consistency check (klt_dev_affine_*): per-feature state + templates, positions before tracking
  AffState* d_aff_st; AffState* h_aff_st; float* d_aff_tmpl; float* d_x0; int aff_cap, aff_tsz, aff_x0_cap;
  // ring of pinned feature snapshots (klt_dev_snapshot_*)
  unsigned char* snap_ring; size_t snap_bytes; int snap_depth, snap_events; cudaEvent_t ev_snap[KLT_SNAP_MAX];
  // selection
  int *c_val[2]; unsigned* c_idx[2]; size_t cand_cap;
  void* cub_tmp; size_t cub_bytes;
  unsigned char* fmap; size_t fmap_cap;
  int* open_slots; int open_cap;
  int* rank_list; int* sel_state;      // candidates still uncovered (ranks, ascending) / [0..2] walk state, [4] their number
  int no_filter; int replace_filter;
  int enforce_attr;            // enforce_mindist_kernel's shared-memory attribute set on this device
  // tile queues of the persistent pyramid kernels: one counter per pyramid level
  unsigned* d_tile_ctr; unsigned tile_base[KLT_TILE_QUEUES];
  // timing
  cudaEvent_t ev_a, ev_b; int ev_made;
  // per-kernel profiling (klt_dev_profile_*)
  int prof_on, prof_used;
  cudaEvent_t* prof_ev;          // 2 * PROF_POOL events
  int* prof_kid;
  double prof_ms[KID_COUNT];
  unsigned long long prof_n[KID_COUNT];
  // timeline of the profiled operations (klt_dev_trace_get): start/end in ms since profile_begin
  cudaEvent_t ev_origin;
  int trace_n; int* trace_kid; float* trace_t0; float* trace_t1;
  // features entering klt_dev_track* with val >= 0, accumulated on the device
  unsigned long long* d_live;
  // forward-backward check: one FbRec per feature of the last tracking call that ran it (fb_n >= 0)
  FbRec* d_fb; int fb_cap, fb_n; float fb_max_error;   // (fb_max_error: of the tracker being launched)
  // motion prior: per feature index a velocity record (valid for indices < vel_n) and the record of
  // the last tracking call that ran with the prior (pred_n >= 0); explicit guesses gx | gy queued for
  // the next tracking call (guess_n >= 0) in slot guess_slot of a two-slot ring (device buffers and
  // pinned staging, slot s at s * 2 * guess_cap); ev_guess[s] is recorded behind the last copy into
  // slot s and again behind the tracker that reads it, so a slot is refilled only once both are done
  PredVel* d_vel; PredRec* d_pred; int pred_cap, pred_n, vel_n;
  float* d_guess; float* h_guess; int guess_cap, guess_n, guess_slot;
  cudaEvent_t ev_guess[2]; int guess_busy[2];
  PredArgs pred;                // (of the tracker being launched)
};

// RAII around one kernel launch: counts it and, in profiling mode, brackets it
// with CUDA events on the context stream.
static void prof_fold(klt_dev* d) {
  if (d->prof_used == 0) return;
  cudaStreamSynchronize(d->stream);
  if (d->stream2) cudaStreamSynchronize(d->stream2);
  if (d->cstream) cudaStreamSynchronize(d->cstream);
  for (int i = 0; i < d->prof_used; ++i) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, d->prof_ev[2 * i], d->prof_ev[2 * i + 1]) == cudaSuccess) {
      d->prof_ms[d->prof_kid[i]] += ms;
      d->prof_n[d->prof_kid[i]] += 1;
      if (d->trace_n < TRACE_CAP) {
        float t0 = 0.0f;
        cudaEventElapsedTime(&t0, d->ev_origin, d->prof_ev[2 * i]);
        d->trace_kid[d->trace_n] = d->prof_kid[i];
        d->trace_t0[d->trace_n] = t0; d->trace_t1[d->trace_n] = t0 + ms;
        d->trace_n += 1;
      }
    }
  }
  d->prof_used = 0;
}
static int sync_all(klt_dev* d) {
  cudaError_t e = cudaStreamSynchronize(d->stream);
  if (e == cudaSuccess && d->stream2) e = cudaStreamSynchronize(d->stream2);
  if (e == cudaSuccess && d->cstream) e = cudaStreamSynchronize(d->cstream);
  d->staging_busy = 0;
  return e == cudaSuccess ? 0 : 1;
}
struct Launch {
  klt_dev* d; int slot; cudaStream_t st;
  Launch(klt_dev* d_, int kid, cudaStream_t st_ = nullptr) : d(d_), slot(-1), st(st_ ? st_ : d_->stream) {
    if (kid != KID_COPY_H2D && kid != KID_COPY_D2H) d->launches++;
    if (d->prof_on) {
      if (d->prof_used == PROF_POOL) prof_fold(d);
      slot = d->prof_used++;
      d->prof_kid[slot] = kid;
      cudaEventRecord(d->prof_ev[2 * slot], st);
    }
  }
  ~Launch() { if (slot >= 0) cudaEventRecord(d->prof_ev[2 * slot + 1], st); }
};

// kernel launch with (optionally) programmatic stream serialisation: the kernel may start before
// its predecessor in the stream has finished and synchronises itself with griddepcontrol.wait
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                            Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static char g_create_err[512] = "";

static int fail(klt_dev* d, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(d ? d->err : g_create_err, 512, fmt, ap);
  va_end(ap);
  return 1;
}
#define CU(call)                                                                       \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess)                                                             \
      return fail(d, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static TapsF to_fused(const TapsR& t) {
  TapsF f;
  memset(&f, 0, sizeof(f));
  f.w = t.w;
  for (int m = 0; m < t.w && m < FUSED_MAX_TAPS; ++m) { f.k[m] = t.k[m]; f.kk[m] = make_float2(t.k[m], t.k[m]); }
  return f;
}
static TapsR reversed(const float* k, int w) {
  TapsR t;
  memset(&t, 0, sizeof(t));
  t.w = w;
  for (int m = 0; m < w; ++m) t.k[m] = k[w - 1 - m];
  return t;
}

extern "C" int klt_dev_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
extern "C" const char* klt_dev_create_error(void) { return g_create_err; }
extern "C" const char* klt_dev_error(const klt_dev* d) { return d ? d->err : g_create_err; }
extern "C" int klt_dev_device(const klt_dev* d) { return d->device; }
extern "C" void* klt_dev_stream(const klt_dev* d) { return (void*)d->stream; }
extern "C" unsigned long long klt_dev_launch_count(const klt_dev* d) { return d->launches; }
extern "C" int klt_dev_last_build_path(const klt_dev* d) { return d->last_path; }
extern "C" void klt_dev_force_generic(klt_dev* d, int on) { d->force_generic = on; }
extern "C" void klt_dev_disable_fused(klt_dev* d, int on) { d->no_fused = on; d->track7_off = on; }
extern "C" int klt_dev_last_build_fused(const klt_dev* d) { return d->last_fused; }
extern "C" int klt_dev_last_build_bands(const klt_dev* d) { return d->last_bands; }
extern "C" int klt_dev_last_build_staged(const klt_dev* d) { return d->last_staged; }
extern "C" void klt_dev_set_stage_threads(klt_dev* d, int n) { d->stage_threads = n; }
extern "C" void klt_dev_set_band_rows(klt_dev* d, int rows) { d->band_rows = rows; }

extern "C" int klt_dev_create(int device, klt_dev** out) {
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, "no CUDA device available (%s); this library has no CPU path",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  if (device >= n) return fail(nullptr, "device %d requested but only %d present", device, n);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
  klt_dev* c = (klt_dev*)calloc(1, sizeof(klt_dev));
  if (!c) return fail(nullptr, "out of host memory");
  c->device = device;
  cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device);
  if (c->num_sms < 1) c->num_sms = 1;
  e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking);
  for (int i = 0; i < KLT_DEV_SLOTS && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&c->ev_built[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_read[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->cstream, cudaStreamNonBlocking);
  for (int i = 0; i < KLT_BAND_EVENTS && e == cudaSuccess; ++i)
    e = cudaEventCreateWithFlags(&c->ev_band[i], cudaEventDisableTiming);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&c->ev_frame_free[i], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_feat, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_stage_free, cudaEventDisableTiming);
  // default: up to 4 threads, but never more than the process was told to use (torchrun exports
  // OMP_NUM_THREADS=1 per rank so that 8 ranks do not oversubscribe the host)
  {
    int want = 4;
    if (getenv("OMP_NUM_THREADS") && atoi(getenv("OMP_NUM_THREADS")) > 0 && atoi(getenv("OMP_NUM_THREADS")) < want)
      want = atoi(getenv("OMP_NUM_THREADS"));
    if (getenv("KLT_B200_STAGE_THREADS")) want = atoi(getenv("KLT_B200_STAGE_THREADS"));
    cpu_set_t cs;
    CPU_ZERO(&cs);
    const int avail = sched_getaffinity(0, sizeof(cs), &cs) == 0 ? CPU_COUNT(&cs) : 1;
    c->stage_threads = want > avail ? avail : want;
  }
  c->band_rows = getenv("KLT_B200_BAND_ROWS") ? atoi(getenv("KLT_B200_BAND_ROWS")) : -1;
  c->reg_frames = getenv("KLT_B200_REGISTER_FRAMES") ? atoi(getenv("KLT_B200_REGISTER_FRAMES")) : 0;   // opt-in: see klt_cuda.h
  if (e != cudaSuccess) { free(c); return fail(nullptr, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
  c->tstream = c->stream;
  c->fb_n = -1;
  c->pred_n = -1; c->guess_n = -1;
  e = cudaMalloc(&c->d_live, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemsetAsync(c->d_live, 0, sizeof(unsigned long long), c->stream);
  c->pdl = getenv("KLT_B200_PDL") ? atoi(getenv("KLT_B200_PDL")) : 1;
  c->guard = getenv("KLT_B200_GUARD") ? (atoi(getenv("KLT_B200_GUARD")) != 0) : 0;
  if (getenv("KLT_B200_L2_HINTS")) {              // (per device: the symbol lives in this device's module image)
    const int hints = atoi(getenv("KLT_B200_L2_HINTS")) & 3;
    cudaMemcpyToSymbol(c_l2_hints, &hints, sizeof(int));
  }
  c->no_track7w = getenv("KLT_B200_TRACK7W") ? !atoi(getenv("KLT_B200_TRACK7W")) : 0;
  if (getenv("KLT_B200_L2_PERSIST_MB")) {       // experiment: L2 set-aside for evict_last lines (KLT_TRACK_L2_KEEP)
    int maxb = 0;
    cudaDeviceGetAttribute(&maxb, cudaDevAttrMaxPersistingL2CacheSize, c->device);
    size_t want = (size_t)atoi(getenv("KLT_B200_L2_PERSIST_MB")) << 20;
    if (want > (size_t)maxb) want = (size_t)maxb;
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
    fprintf(stderr, "(KLT/B200) persisting L2: %zu MB of max %d MB\n", want >> 20, maxb >> 20);
  }
  if (e == cudaSuccess) e = cudaMalloc(&c->d_tile_ctr, KLT_TILE_QUEUES * sizeof(unsigned));
  if (e == cudaSuccess) e = cudaMemsetAsync(c->d_tile_ctr, 0, KLT_TILE_QUEUES * sizeof(unsigned), c->stream);
  if (e != cudaSuccess) { cudaStreamDestroy(c->stream); free(c); return fail(nullptr, "cudaMalloc: %s", cudaGetErrorString(e)); }
  *out = c;
  return 0;
}

static constexpr size_t KLT_GUARD_FLOATS = 1024;      // 4 KB: keeps every plane 128-byte aligned
static constexpr int KLT_GUARD_BYTE = 0xA5;
// cudaMalloc / cudaFree with a canary band on either side in guard mode (the selection and feature buffers)
static cudaError_t guarded_malloc(klt_dev* d, void** out, size_t bytes) {
  if (!d->guard || d->nguarded >= (int)(sizeof(d->guarded) / sizeof(d->guarded[0]))) return cudaMalloc(out, bytes);
  const size_t gb = KLT_GUARD_FLOATS * sizeof(float), padded = (bytes + 255) / 256 * 256;
  unsigned char* base = nullptr;
  cudaError_t e = cudaMalloc(&base, padded + 2 * gb);
  if (e != cudaSuccess) return e;
  e = cudaMemset(base, KLT_GUARD_BYTE, padded + 2 * gb);
  if (e != cudaSuccess) { cudaFree(base); return e; }
  *out = base + gb;
  d->guarded[d->nguarded].user = base + gb; d->guarded[d->nguarded].bytes = bytes; d->nguarded += 1;
  return cudaSuccess;
}
template <typename T>
static cudaError_t guarded_malloc(klt_dev* d, T** out, size_t bytes) { return guarded_malloc(d, reinterpret_cast<void**>(out), bytes); }
static void guarded_free(klt_dev* d, void* p) {
  if (!p) return;
  for (int i = 0; i < d->nguarded; ++i)
    if (d->guarded[i].user == p) {
      cudaFree(static_cast<unsigned char*>(p) - KLT_GUARD_FLOATS * sizeof(float));
      d->guarded[i] = d->guarded[--d->nguarded];
      return;
    }
  cudaFree(p);
}
static void free_geometry(klt_dev* d) {
  cudaFree(d->arena); d->arena = nullptr;
  cudaFree(d->tmp); d->tmp = nullptr;
  memset(d->set, 0, sizeof(d->set));
  d->W = d->H = d->L = d->ss = 0;
}

extern "C" void klt_dev_destroy(klt_dev* d) {
  if (!d) return;
  cudaSetDevice(d->device);
  sync_all(d);
  klt_dev_forget_host_frames(d);
  free_geometry(d);
  cudaFree(d->frame_buf[0]); cudaFree(d->frame_buf[1]);
  guarded_free(d, d->d_x);
  guarded_free(d, d->d_fb);
  guarded_free(d, d->d_vel); guarded_free(d, d->d_pred); guarded_free(d, d->d_guess); cudaFreeHost(d->h_guess);
  for (int i = 0; i < 2; ++i) if (d->ev_guess[i]) cudaEventDestroy(d->ev_guess[i]);
  cudaFreeHost(d->h_x);
  for (int i = 0; i < 2; ++i) { guarded_free(d, d->c_val[i]); guarded_free(d, d->c_idx[i]); }
  cudaFree(d->cub_tmp); guarded_free(d, d->fmap); guarded_free(d, d->open_slots); guarded_free(d, d->rank_list); guarded_free(d, d->sel_state);
  if (d->ev_made) { cudaEventDestroy(d->ev_a); cudaEventDestroy(d->ev_b); }
  if (d->prof_ev) { for (int i = 0; i < 2 * PROF_POOL; ++i) cudaEventDestroy(d->prof_ev[i]); free(d->prof_ev); free(d->prof_kid);
    cudaEventDestroy(d->ev_origin); free(d->trace_kid); free(d->trace_t0); free(d->trace_t1); }
  cudaFree(d->d_live);
  cudaFree(d->d_tile_ctr);
  cudaFree(d->d_rec);
  for (int i = 0; i < KLT_DEV_SLOTS; ++i) { cudaEventDestroy(d->ev_built[i]); cudaEventDestroy(d->ev_read[i]); }
  cudaEventDestroy(d->ev_join);
  for (int i = 0; i < KLT_BAND_EVENTS; ++i) cudaEventDestroy(d->ev_band[i]);
  cudaEventDestroy(d->ev_frame_free[0]); cudaEventDestroy(d->ev_frame_free[1]);
  cudaEventDestroy(d->ev_feat);
  cudaEventDestroy(d->ev_stage_free);
  cudaFreeHost(d->h_frame);
  cudaFreeHost(d->snap_ring);
  cudaFree(d->d_aff_st); cudaFreeHost(d->h_aff_st); cudaFree(d->d_aff_tmpl); cudaFree(d->d_x0);
  for (int i = 0; i < d->snap_events; ++i) cudaEventDestroy(d->ev_snap[i]);
  cudaStreamDestroy(d->cstream);
  cudaStreamDestroy(d->stream);
  cudaStreamDestroy(d->stream2);
  free(d);
}

static int ensure_geometry(klt_dev* d, int W, int H, int L, int ss) {
  if (d->arena && d->W == W && d->H == H && d->L == L && d->ss == ss) return 0;
  if (W <= 0 || H <= 0) return fail(d, "bad image size %d x %d", W, H);
  if (L < 1 || L > KLT_DEV_MAX_LEVELS) return fail(d, "nPyramidLevels %d not in 1..%d", L, KLT_DEV_MAX_LEVELS);
  if (L > 1 && ss != 2 && ss != 4 && ss != 8 && ss != 16 && ss != 32)
    return fail(d, "Pyramid's subsampling must be either 2, 4, 8, 16, or 32");
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  memset(d->read_pending, 0, sizeof(d->read_pending));
  memset(d->built_pending, 0, sizeof(d->built_pending));
  free_geometry(d);
  d->vel_n = 0;                        // a velocity from frames of another size predicts nothing
  size_t per_set = 0;
  int w = W, h = H;
  int ws[KLT_DEV_MAX_LEVELS], hs[KLT_DEV_MAX_LEVELS], ps[KLT_DEV_MAX_LEVELS];
  for (int l = 0; l < L; ++l) {
    ws[l] = w; hs[l] = h; ps[l] = (w + 31) / 32 * 32;
    if (w < 1 || h < 1) return fail(d, "pyramid level %d is empty (%d x %d)", l, w, h);
    per_set += 3 * (size_t)ps[l] * h;
    if (L > 1) { w /= ss; h /= ss; }
  }
  // guard mode (debug): a canary band in front of every plane and behind the last one; the kernels
  // never write outside a plane's pitch x height, klt_dev_check_guards verifies it
  const size_t gap = d->guard ? KLT_GUARD_FLOATS : 0;
  const size_t total = KLT_DEV_SLOTS * (per_set + 3 * (size_t)L * gap) + gap;
  CU(cudaMalloc(&d->arena, total * sizeof(float) + 256));   // + slack for aligned over-reads
  d->arena_floats = total;
  if (d->guard) CU(cudaMemset(d->arena, KLT_GUARD_BYTE, total * sizeof(float) + 256));
  CU(cudaMalloc(&d->tmp, (size_t)ps[0] * H * sizeof(float)));
  float* p = d->arena;
  for (int s = 0; s < KLT_DEV_SLOTS; ++s)
    for (int l = 0; l < L; ++l) {
      Level& lv = d->set[s].lv[l];
      lv.w = ws[l]; lv.h = hs[l]; lv.pitch = ps[l];
      const size_t n = (size_t)ps[l] * hs[l];
      p += gap; lv.img = p; p += n; p += gap; lv.gx = p; p += n; p += gap; lv.gy = p; p += n;
    }
  d->W = W; d->H = H; d->L = L; d->ss = ss;
  return 0;
}

// Debug aid in place of compute-sanitizer (closed on the pool): with guard mode on, every plane of
// the pyramid arena is preceded by a 4 KB canary band (and the last one followed by one); a kernel
// that stores outside its plane lands in a band.  Returns the number of damaged canary words and the
// index (slot * 3 L + 3 level + plane; 3 L * slots = the band behind the last plane) of the first
// damaged band.  Switching the mode re-allocates the arena at the next build.
extern "C" void klt_dev_set_guard(klt_dev* d, int on) {
  if (d->guard == (on ? 1 : 0)) return;
  sync_all(d);
  free_geometry(d);
  // the selection buffers are re-created on demand (the feature arrays keep their state: they are
  // guarded when they are allocated after this call)
  for (int i = 0; i < 2; ++i) { guarded_free(d, d->c_val[i]); guarded_free(d, d->c_idx[i]); d->c_val[i] = nullptr; d->c_idx[i] = nullptr; }
  guarded_free(d, d->rank_list); guarded_free(d, d->sel_state); d->rank_list = nullptr; d->sel_state = nullptr;
  cudaFree(d->cub_tmp); d->cub_tmp = nullptr; d->cand_cap = 0;
  guarded_free(d, d->fmap); d->fmap = nullptr; d->fmap_cap = 0;
  guarded_free(d, d->open_slots); d->open_slots = nullptr; d->open_cap = 0;
  d->guard = on ? 1 : 0;
}
extern "C" int klt_dev_check_guards(klt_dev* d, long long* damaged_words, int* first_band) {
  if (damaged_words) *damaged_words = 0;
  if (first_band) *first_band = -1;
  if (!d->guard) return 0;
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  unsigned* h = (unsigned*)malloc(KLT_GUARD_FLOATS * sizeof(unsigned));
  if (!h) return fail(d, "out of memory");
  const unsigned want = 0x01010101u * (unsigned)KLT_GUARD_BYTE;
  long long bad = 0;
  int first = -1, band = 0;
  auto check = [&](const float* at) -> int {
    if (cudaMemcpy(h, at, KLT_GUARD_FLOATS * sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    for (size_t i = 0; i < KLT_GUARD_FLOATS; ++i)
      if (h[i] != want) { bad += 1; if (first < 0) first = band; }
    band += 1;
    return 0;
  };
  int rc = 0;
  for (int s = 0; d->arena && s < KLT_DEV_SLOTS && !rc; ++s)
    for (int l = 0; l < d->L && !rc; ++l) {
      const Level& lv = d->set[s].lv[l];
      rc = check(lv.img - KLT_GUARD_FLOATS) || check(lv.gx - KLT_GUARD_FLOATS) || check(lv.gy - KLT_GUARD_FLOATS);
    }
  if (!rc && d->arena) rc = check(d->arena + d->arena_floats - KLT_GUARD_FLOATS);
  // selection / feature buffers: band in front and band behind (from the first 256-byte boundary after the buffer)
  band = 1000;
  for (int i = 0; i < d->nguarded && !rc; ++i) {
    const unsigned char* u = static_cast<const unsigned char*>(d->guarded[i].user);
    rc = check(reinterpret_cast<const float*>(u - KLT_GUARD_FLOATS * sizeof(float))) ||
         check(reinterpret_cast<const float*>(u + (d->guarded[i].bytes + 255) / 256 * 256));
  }
  free(h);
  if (rc) return fail(d, "guard check: copy failed");
  if (damaged_words) *damaged_words = bad;
  if (first_band) *first_band = first;
  return 0;
}

// (for the guard test: where a plane lives, and a raw host-to-device write)
extern "C" void* klt_dev_plane_address(const klt_dev* d, int slot, int which, int level) {
  if (!d->arena || slot < 0 || slot >= KLT_DEV_SLOTS || level < 0 || level >= d->L) return nullptr;
  const Level& lv = d->set[slot].lv[level];
  return which == 0 ? (void*)lv.img : which == 1 ? (void*)lv.gx : which == 2 ? (void*)lv.gy : nullptr;
}
extern "C" int klt_dev_poke(klt_dev* d, void* device_dst, const void* host_src, size_t bytes) {
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  CU(cudaMemcpy(device_dst, host_src, bytes, cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int klt_dev_geometry(const klt_dev* d, int* W, int* H, int* L, int* ss) {
  if (W) *W = d->W; if (H) *H = d->H; if (L) *L = d->L; if (ss) *ss = d->ss;
  return d->arena != nullptr;
}
extern "C" int klt_dev_slot_valid(const klt_dev* d, int slot) {
  return d->arena && slot >= 0 && slot < KLT_DEV_SLOTS && d->set[slot].built_levels == d->L;
}
extern "C" void klt_dev_invalidate(klt_dev* d, int slot) {
  for (int s = 0; s < KLT_DEV_SLOTS; ++s) if (slot < 0 || slot == s) d->set[s].built_levels = 0;
}
extern "C" int klt_dev_level_dims(const klt_dev* d, int level, int* w, int* h) {
  if (!d->arena || level < 0 || level >= d->L) return 1;
  *w = d->set[0].lv[level].w; *h = d->set[0].lv[level].h;
  return 0;
}
extern "C" int klt_dev_sync(klt_dev* d) {
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  return 0;
}

// overlap on: the tracker and the feature copies move to a second stream, ordered against the
// pyramid builds with events, so that build(k+1) can run while track(k) is still in flight.
extern "C" int klt_dev_set_overlap(klt_dev* d, int on) {
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  memset(d->read_pending, 0, sizeof(d->read_pending));
  memset(d->built_pending, 0, sizeof(d->built_pending));
  d->overlap = on ? 1 : 0;
  d->tstream = on ? d->stream2 : d->stream;
  return 0;
}
extern "C" int klt_dev_slots(void) { return KLT_DEV_SLOTS; }

// ---- kernel dispatch ----------------------------------------------------------
template <typename K>
static int set_smem(klt_dev* d, K kernel, size_t bytes) {
  if (bytes > 48 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

template <int R, bool EXACT>
static int launch_smooth_u8(klt_dev* d, const unsigned char* src, int spitch, int W, int H,
                            const TapsR& t, float* out, int opitch) {
  using G = TileGeo<1, R, 64, 32, 4>;
  const size_t smem = (G::IN_FLOATS + G::IH * 64) * sizeof(float);
  if (set_smem(d, smooth_u8_tile<R, EXACT>, smem)) return 1;
  dim3 grid((W + 63) / 64, (H + 31) / 32);
  { Launch l(d, KID_SMOOTH_U8);
    smooth_u8_tile<R, EXACT><<<grid, NT, smem, d->stream>>>(src, spitch, W, H, t, out, opitch); }
  return 0;
}
template <bool EXACT>
static int smooth_u8_dispatch(klt_dev* d, const unsigned char* src, int spitch, int W, int H,
                              const TapsR& t, float* out, int opitch, bool* done) {
  *done = true;
  switch (t.w / 2) {
    case 1: return launch_smooth_u8<1, EXACT>(d, src, spitch, W, H, t, out, opitch);
    case 2: return launch_smooth_u8<2, EXACT>(d, src, spitch, W, H, t, out, opitch);
    case 3: return launch_smooth_u8<3, EXACT>(d, src, spitch, W, H, t, out, opitch);
    case 4: return launch_smooth_u8<4, EXACT>(d, src, spitch, W, H, t, out, opitch);
    case 5: return launch_smooth_u8<5, EXACT>(d, src, spitch, W, H, t, out, opitch);
    case 6: return launch_smooth_u8<6, EXACT>(d, src, spitch, W, H, t, out, opitch);
    default: *done = false; return 0;
  }
}

template <int RG, int RD, bool EXACT>
static int launch_grad(klt_dev* d, const float* src, int spitch, int W, int H, const TapsR& tg,
                       const TapsR& td, float* ox, float* oy, int opitch) {
  constexpr int RM = RG > RD ? RG : RD;
  using G = TileGeo<1, RM, 64, 32, 4>;
  const size_t smem = (G::IN_FLOATS + 2 * G::IH * 64) * sizeof(float);
  if (set_smem(d, grad_tile<RG, RD, EXACT>, smem)) return 1;
  dim3 grid((W + 63) / 64, (H + 31) / 32);
  { Launch l(d, KID_GRAD);
    grad_tile<RG, RD, EXACT><<<grid, NT, smem, d->stream>>>(src, spitch, W, H, tg, td, ox, oy, opitch); }
  return 0;
}
template <bool EXACT>
static int grad_dispatch(klt_dev* d, const float* src, int spitch, int W, int H, const TapsR& tg,
                         const TapsR& td, float* ox, float* oy, int opitch, bool* done) {
  *done = true;
  const int rg = tg.w / 2, rd = td.w / 2;
  if (rg == 3 && rd == 3) return launch_grad<3, 3, EXACT>(d, src, spitch, W, H, tg, td, ox, oy, opitch);
  if (rg == 2 && rd == 2) return launch_grad<2, 2, EXACT>(d, src, spitch, W, H, tg, td, ox, oy, opitch);
  if (rg == 4 && rd == 4) return launch_grad<4, 4, EXACT>(d, src, spitch, W, H, tg, td, ox, oy, opitch);
  if (rg == 4 && rd == 5) return launch_grad<4, 5, EXACT>(d, src, spitch, W, H, tg, td, ox, oy, opitch);
  if (rg == 5 && rd == 6) return launch_grad<5, 6, EXACT>(d, src, spitch, W, H, tg, td, ox, oy, opitch);
  *done = false;
  return 0;
}

template <int SS, int R, int TXO, int TYO, int PY, bool EXACT>
static int launch_pyrdown(klt_dev* d, const float* src, int spitch, int W, int H, const TapsR& t,
                          float* out, int opitch, int Wout, int Hout) {
  using G = TileGeo<SS, R, TXO, TYO, 4>;
  const size_t smem = (G::IN_FLOATS + G::IH * TXO) * sizeof(float);
  if (set_smem(d, pyrdown_tile<SS, R, TXO, TYO, PY, EXACT>, smem)) return 1;
  dim3 grid((Wout + TXO - 1) / TXO, (Hout + TYO - 1) / TYO);
  { Launch l(d, KID_PYRDOWN);
    pyrdown_tile<SS, R, TXO, TYO, PY, EXACT><<<grid, NT, smem, d->stream>>>(src, spitch, W, H, t, out,
                                                                           opitch, Wout, Hout); }
  return 0;
}
template <bool EXACT>
static int pyrdown_dispatch(klt_dev* d, int ss, const float* src, int spitch, int W, int H,
                            const TapsR& t, float* out, int opitch, int Wout, int Hout, bool* done) {
  *done = true;
  const int r = t.w / 2;
  if (ss == 2 && r == 5) return launch_pyrdown<2, 5, 32, 32, 4, EXACT>(d, src, spitch, W, H, t, out, opitch, Wout, Hout);
  if (ss == 4 && r == 10) return launch_pyrdown<4, 10, 32, 16, 2, EXACT>(d, src, spitch, W, H, t, out, opitch, Wout, Hout);
  *done = false;
  return 0;
}

// ---- TMA tensor maps -----------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn tma_encoder() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    cudaGetLastError();
  }
  return fn;
}
// 2-D row-major tensor of `elem` bytes per element; zero fill outside [0,w) x [0,h)
static bool make_tensor_map(CUtensorMap* m, const void* base, CUtensorMapDataType dt, int elem, int w, int h,
                            size_t pitch_bytes, int box_w, int box_h) {
  EncodeTiledFn enc = tma_encoder();
  if (!enc) return false;
  if (((uintptr_t)base & 15) || (pitch_bytes & 15) || ((box_w * elem) & 15) || box_w > 256 || box_h > 256)
    return false;
  cuuint64_t dims[2] = {(cuuint64_t)w, (cuuint64_t)h};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool fused_grad_taps_ok(const TapsR& tg, const TapsR& td) {
  return tg.w == 2 * FUSED_RG + 1 && td.w == 2 * FUSED_RG + 1 && td.k[FUSED_RG] == 0.0f;
}

// ---- fused kernels: plan (tensor maps, tile shapes) + launches over whole tile rows ------------
// A launch covers the tile rows [jr0, jr1) of one level, so that a frame can be built band by band
// behind its upload (klt_dev_build with a host frame) or in one go (jr0 = 0, jr1 = tiles_y).
enum LevelShape { SHAPE_NONE = 0, SHAPE_2_5_64_32, SHAPE_2_5_64_16, SHAPE_2_5_32_16, SHAPE_4_10_32_16 };
struct FusedPlan {
  bool l0_ok;                                   // level 0 runs on l0_fused_kernel
  int shape[KLT_DEV_MAX_LEVELS];                // LevelShape of level l >= 1 (SHAPE_NONE: not fused)
  CUtensorMap map[KLT_DEV_MAX_LEVELS];          // source of level l (u8 frame for l = 0, L_{l-1} else)
  int TX[KLT_DEV_MAX_LEVELS], TY[KLT_DEV_MAX_LEVELS], tiles_x[KLT_DEV_MAX_LEVELS], tiles_y[KLT_DEV_MAX_LEVELS];
  bool l0_march;                                // level 0 on l0_march_kernel (strips x segments) instead of tiles
  bool chain;                                   // level 0 on L0GeoC (also makes L1), levels >= 1 on
                                                // level_chain_kernel (map[l]: L_l itself)
  // band schedule: tile row j of level l reads rows [0, need_mul * (j + 1) + need_add) of plane src_plane[l]
  // and completes rows [0, made_mul * j) of the plane level l + 1 reads (plane 0: the u8 frame, k + 1: L_k)
  int src_plane[KLT_DEV_MAX_LEVELS], need_mul[KLT_DEV_MAX_LEVELS], need_add[KLT_DEV_MAX_LEVELS],
      made_mul[KLT_DEV_MAX_LEVELS];
};

static int level_shape_for(int ss, int r, int w, int h, int num_sms) {
  if (ss == 2 && r == 5) {
    // tile shape by level size: big levels amortise the halo with 64x32 tiles, small levels
    // need many small tiles to fill 148 SMs and to keep the per-CTA latency short.  In between
    // (4K level 2: 960x540) the wave count decides: 64x32 tiles when they all fit into ONE wave of
    // 2 CTAs per SM (255 tiles: 10.6 us), else 64x16 tiles at 3 CTAs per SM (510 tiles = 1.15
    // waves: 12.7 us; measured on the 4K step: 74.1 -> 72.8 us).
    const long px = (long)w * h;
    const long tiles_64x32 = (long)((w + 63) / 64) * ((h + 31) / 32);
    if (px >= 1500000) return SHAPE_2_5_64_32;
    if (px >= 300000) return tiles_64x32 <= 2L * num_sms ? SHAPE_2_5_64_32 : SHAPE_2_5_64_16;
    return SHAPE_2_5_32_16;
  }
  if (ss == 4 && r == 10) return SHAPE_4_10_32_16;
  return SHAPE_NONE;
}
template <int SS_, int R_, int TX_, int TY_>
struct TileShape { static constexpr int SS = SS_, R = R_, TX = TX_, TY = TY_; };
// The one place where a LevelShape (never SHAPE_NONE) becomes template arguments: f(TileShape<...>()).
template <class F>
static auto with_shape(int shape, F f) {
  switch (shape) {
    case SHAPE_2_5_64_32: return f(TileShape<2, 5, 64, 32>());
    case SHAPE_2_5_64_16: return f(TileShape<2, 5, 64, 16>());
    case SHAPE_2_5_32_16: return f(TileShape<2, 5, 32, 16>());
    default: return f(TileShape<4, 10, 32, 16>());       // SHAPE_4_10_32_16
  }
}

using L0GeoB = L0GeoT<48, 6, 6, 4>;      // 48-row tiles: 2 even passes in stages A / C, 54 KB of shared memory, 4 CTAs / SM
// Level 0 of a chained pyramid (subsampling 2, radius 5, more than one level): the tile also makes its
// 32 x 20 block of L1.  With the L1 halo and the horizontal L1 buffer a 48-row tile needs 63.6 KB, which
// leaves 3 CTAs per SM; 40-row tiles need 55.7 KB and keep 4 (32 warps).
using L0GeoC = L0GeoT<40, 7, 5, 4, true>;
// 0: 64-row tiles, 3 CTAs / SM; 1 (default): 48-row tiles, 4 CTAs / SM; 2: l0_march_kernel (klt_march.cuh: the
// barrier-free strip formulation, bit-identical, measured slower: 32.5 vs 28.7 us per 4K frame)
static int g_l0_variant = -1;
static int l0_variant() {
  if (g_l0_variant < 0) g_l0_variant = getenv("KLT_B200_L0_TILE") ? atoi(getenv("KLT_B200_L0_TILE")) : 1;
  return g_l0_variant;
}
extern "C" void klt_dev_set_l0_kernel(int variant) { g_l0_variant = variant; }
extern "C" int klt_dev_l0_kernel(void) { return l0_variant(); }
// which levels of this build can run on the fused kernels, their tensor maps and band schedule
static void fused_plan(klt_dev* d, const PyrSet& S, const unsigned char* src, int spitch,
                       const klt_dev_build_desc* q, const TapsR& ts, const TapsR& tp, const TapsR& tg,
                       const TapsR& td, FusedPlan* P) {
  memset(P, 0, sizeof(*P));
  if (d->force_generic || d->no_fused || !fused_grad_taps_ok(tg, td)) return;
  const int W = q->ncols, H = q->nrows;
  const int l0_ty = l0_variant() == 1 ? L0GeoB::TY : L0Geo::TY, l0_u8h = l0_variant() == 1 ? L0GeoB::U8_H : L0Geo::U8_H;
  if (l0_variant() == 2 && q->smooth && ts.w == 2 * MarchGeo::RS + 1 &&
      make_tensor_map(&P->map[0], src, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, W, H, (size_t)spitch, MarchGeo::IN_W, MarchGeo::PU)) {
    // strips of 120 columns x segments of rows, one task per team of the grid when the frame is big
    // enough (4K: 32 strips x 37 segments of 59 rows = 1184 tasks = 148 SMs x 2 CTAs x 4 teams)
    const int nstrips = (W + MarchGeo::SWI - 1) / MarchGeo::SWI;
    const int teams = MarchGeo::CPS * d->num_sms * MarchGeo::TEAMS;
    int nseg = teams / nstrips;
    if (nseg < 1) nseg = 1;
    int seg_rows = (H + nseg - 1) / nseg;
    if (seg_rows < 16) seg_rows = 16;
    P->l0_ok = true; P->l0_march = true;
    P->TX[0] = MarchGeo::SWI; P->TY[0] = seg_rows;
    P->tiles_x[0] = nstrips; P->tiles_y[0] = (H + seg_rows - 1) / seg_rows;
  } else if (q->smooth && ts.w == 2 * L0Geo::RS + 1 &&
      make_tensor_map(&P->map[0], src, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, W, H, (size_t)spitch, L0Geo::U8_W, l0_u8h)) {
    P->l0_ok = true;
    P->TX[0] = L0Geo::TX; P->TY[0] = l0_ty;
    P->tiles_x[0] = (W + L0Geo::TX - 1) / L0Geo::TX; P->tiles_y[0] = (H + l0_ty - 1) / l0_ty;
  }
  P->need_add[0] = L0Geo::RS + L0Geo::RG;       // u8 rows a level-0 tile row reads below its last output row
  // Chained pyramid: level 0 makes L1, level l makes L_{l+1}, so every level >= 1 reads only its own
  // plane.  The default level-0 variant with subsampling 2 / radius 5 and every level fused; builds of
  // one level keep L0GeoB.
  if (P->l0_ok && !P->l0_march && l0_variant() == 1 && q->nlevels_built > 1 && q->subsampling == 2 &&
      tp.w == 2 * NEXT_R + 1) {
    bool all = true;
    for (int l = 1; l < q->nlevels_built; ++l)
      all = all && level_shape_for(2, NEXT_R, S.lv[l].w, S.lv[l].h, d->num_sms) != SHAPE_NONE;
    CUtensorMap m0;
    if (all && make_tensor_map(&m0, src, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, W, H, (size_t)spitch, L0GeoC::U8_W,
                               L0GeoC::U8_H)) {
      P->chain = true;
      P->map[0] = m0;
      P->TY[0] = L0GeoC::TY;
      P->tiles_y[0] = (H + L0GeoC::TY - 1) / L0GeoC::TY;
      P->need_add[0] = L0GeoC::U8_H - L0GeoC::TY - (L0GeoC::RS + L0GeoC::RG + L0GeoC::XR);
    }
  }
  P->need_mul[0] = P->TY[0];
  P->made_mul[0] = P->chain ? P->TY[0] / 2 : P->TY[0];
  for (int l = 1; l < q->nlevels_built; ++l) {
    const int shape = level_shape_for(q->subsampling, tp.w / 2, S.lv[l].w, S.lv[l].h, d->num_sms);
    if (shape == SHAPE_NONE) continue;
    const Level& a = S.lv[P->chain ? l : l - 1];             // the plane the level's tiles read
    const bool ok = with_shape(shape, [&](auto s) {
      using T = decltype(s);
      P->TX[l] = T::TX; P->TY[l] = T::TY;
      if (P->chain) {                                         // L_l -> gx_l, gy_l, L_{l+1}
        using G = ChGeo<T::TX, T::TY>;
        P->src_plane[l] = l + 1;
        P->need_mul[l] = T::TY; P->need_add[l] = 1 - G::RN + G::SH - T::TY; P->made_mul[l] = T::TY / 2;
        return make_tensor_map(&P->map[l], a.img, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.w, a.h, (size_t)a.pitch * 4,
                               G::SW, G::SH);
      }
      using G = LvGeo<T::SS, T::R, T::TX, T::TY>;            // L_{l-1} -> L_l, gx_l, gy_l
      P->src_plane[l] = l;
      P->need_mul[l] = T::SS * T::TY; P->need_add[l] = G::YOFF + G::SH - T::SS * T::TY; P->made_mul[l] = T::TY;
      return make_tensor_map(&P->map[l], a.img, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.w, a.h, (size_t)a.pitch * 4,
                             G::SW, G::SH);
    });
    if (!ok) {
      if (P->chain) { memset(P, 0, sizeof(*P)); return; }   // tensor map refused: nothing runs fused
      continue;
    }
    P->shape[l] = shape;
    P->tiles_x[l] = (S.lv[l].w + P->TX[l] - 1) / P->TX[l];
    P->tiles_y[l] = (S.lv[l].h + P->TY[l] - 1) / P->TY[l];
  }
}

// One launch of a persistent pyramid kernel K: ctas is what the work can use, the grid is at most what
// the SMs hold.  K's shared-memory attribute and resident CTAs per SM are looked up once per device.
template <auto K, typename... Args>
static int launch_persistent(klt_dev* d, int kid, int nth, int smem, int ctas, int* grid, Args... args) {
  static int cps_dev[64] = {};                   // (function attributes are per device; 0: not set yet)
  int& cps = cps_dev[d->device & 63];
  if (!cps) {
    int n = 0;
    CU(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, K, nth, smem));
    cps = n < 1 ? 1 : n;
  }
  *grid = ctas < cps * d->num_sms ? ctas : cps * d->num_sms;
  Launch l(d, kid);
  CU(launch_k(K, dim3(*grid), dim3(nth), smem, d->stream, d->pdl != 0, args...));
  return 0;
}
// K over the tile rows [jr0, jr1) of pyramid level `level`, from that level's tile queue.  QUEUE marks
// where K takes its TileQueue among args.
struct QueueSlot {};
static constexpr QueueSlot QUEUE{};
template <class T> static T fill_queue(T a, const TileQueue&) { return a; }
static TileQueue fill_queue(QueueSlot, const TileQueue& q) { return q; }
template <auto K, typename... Args>
static int launch_tiles(klt_dev* d, int kid, int level, int nth, int smem, int tiles_x, int jr0, int jr1,
                        Args... args) {
  const int n = (jr1 - jr0) * tiles_x;
  const TileQueue q = {tiles_x, jr0 * tiles_x, jr1 * tiles_x, d->d_tile_ctr + level, d->tile_base[level]};
  int grid = 0;
  if (launch_persistent<K>(d, kid, nth, smem, n, &grid, fill_queue(args, q)...)) return 1;
  d->tile_base[level] += (unsigned)(n + grid);
  return 0;
}

// level 0 (u8 -> L0, gx0, gy0 (+ L1 when the plan is chained)), tile rows [jr0, jr1)
template <class G, bool EXACT>
static int l0_tiles_launch(klt_dev* d, const FusedPlan& P, int W, int H, const TapsR& ts, const TapsR& tg,
                           const TapsR& td, const TapsR& tp, const Level& lv, const Level* l1, int jr0, int jr1) {
  return launch_tiles<l0_fused_kernel<G, EXACT>>(
      d, KID_L0_FUSED, 0, 256, G::SMEM, P.tiles_x[0], jr0, jr1, P.map[0], W, H, QUEUE, to_fused(ts), to_fused(tg),
      to_fused(td), lv.img, lv.gx, lv.gy, lv.pitch, to_fused(tp), l1 ? l1->img : nullptr, l1 ? l1->pitch : 0,
      l1 ? l1->w : 0, l1 ? l1->h : 0);
}
template <bool EXACT>
static int l0_fused_launch(klt_dev* d, const FusedPlan& P, int W, int H, const TapsR& ts, const TapsR& tg,
                           const TapsR& td, const TapsR& tp, const PyrSet& S, int jr0, int jr1) {
  if (jr1 <= jr0) return 0;
  if (P.l0_march) {                              // segments [jr0, jr1) of every strip, TEAMS tasks per CTA
    using G = MarchGeo;
    const int nstrips = P.tiles_x[0], task0 = jr0 * nstrips, task1 = jr1 * nstrips;
    int grid = 0;
    return launch_persistent<l0_march_kernel<EXACT>>(
        d, KID_L0_FUSED, G::NTH, G::SMEM, (task1 - task0 + G::TEAMS - 1) / G::TEAMS, &grid, P.map[0], W, H, nstrips,
        P.TY[0], task0, task1, to_fused(ts), to_fused(tg), to_fused(td), S.lv[0].img, S.lv[0].gx, S.lv[0].gy,
        S.lv[0].pitch);
  }
  if (P.chain) return l0_tiles_launch<L0GeoC, EXACT>(d, P, W, H, ts, tg, td, tp, S.lv[0], &S.lv[1], jr0, jr1);
  if (P.TY[0] == L0GeoB::TY) return l0_tiles_launch<L0GeoB, EXACT>(d, P, W, H, ts, tg, td, tp, S.lv[0], nullptr, jr0, jr1);
  return l0_tiles_launch<L0Geo, EXACT>(d, P, W, H, ts, tg, td, tp, S.lv[0], nullptr, jr0, jr1);
}

// level l >= 1, tile rows [jr0, jr1): chained (L_l -> gx_l, gy_l (+ L_{l+1} below the coarsest level))
// or not (L_{l-1} -> L_l, gx_l, gy_l).  Accounted per pyramid level: every level runs its own
// template instantiation / tile shape.
template <bool EXACT>
static int level_launch(klt_dev* d, const FusedPlan& P, const PyrSet& S, int level, int nb, const TapsR& tp,
                        const TapsR& tg, const TapsR& td, int jr0, int jr1) {
  if (jr1 <= jr0) return 0;
  if (P.shape[level] == SHAPE_NONE) return fail(d, "level %d has no fused kernel", level);
  const Level& a = S.lv[level - 1];
  const Level& b = S.lv[level];
  const Level* nx = P.chain && level + 1 < nb ? &S.lv[level + 1] : nullptr;
  const int kid = level <= 1 ? KID_LEVEL_FUSED : level == 2 ? KID_LEVEL_FUSED_L2 : KID_LEVEL_FUSED_L3;
  const int tiles_x = P.tiles_x[level];
  return with_shape(P.shape[level], [&](auto s) {
    using T = decltype(s);
    constexpr int TX = T::TX, TY = T::TY;
    if (!P.chain)
      return launch_tiles<level_fused_kernel<T::SS, T::R, TX, TY, EXACT>>(
          d, kid, level, lv_threads<T::SS, T::R, TX, TY>(), LvGeo<T::SS, T::R, TX, TY>::SMEM, tiles_x, jr0, jr1,
          P.map[level], a.w, a.h, b.w, b.h, QUEUE, to_fused(tp), to_fused(tg), to_fused(td), b.img, b.gx, b.gy, b.pitch);
    if (nx)
      return launch_tiles<level_chain_kernel<TX, TY, true, EXACT>>(
          d, kid, level, 256, ChGeo<TX, TY>::SMEM, tiles_x, jr0, jr1, P.map[level], b.w, b.h, nx->w, nx->h, QUEUE,
          to_fused(tp), to_fused(tg), to_fused(td), b.gx, b.gy, b.pitch, nx->img, nx->pitch);
    return launch_tiles<level_chain_kernel<TX, TY, false, EXACT>>(
        d, kid, level, 256, ChGeo<TX, TY>::SMEM, tiles_x, jr0, jr1, P.map[level], b.w, b.h, 0, 0, QUEUE,
        to_fused(tp), to_fused(tg), to_fused(td), b.gx, b.gy, b.pitch, nullptr, 0);
  });
}

// generic two-kernel separable pass through d->tmp
template <typename SrcT, bool EXACT>
static int generic_separable(klt_dev* d, const SrcT* src, int spitch, int W, int H, const TapsR& kh,
                             const TapsR& kv, int stride, float* out, int opitch, int Wout, int Hout) {
  const int off = stride / 2;
  const int tp = d->set[0].lv[0].pitch;
  dim3 b(32, 8);
  dim3 g1((Wout + 31) / 32, (H + 7) / 8);
  { Launch l(d, KID_GENERIC_H);
    conv_h_generic<SrcT, EXACT><<<g1, b, 0, d->stream>>>(src, spitch, W, H, kh, stride, off, d->tmp, tp, Wout); }
  dim3 g2((Wout + 31) / 32, (Hout + 7) / 8);
  { Launch l(d, KID_GENERIC_V);
    conv_v_generic<EXACT><<<g2, b, 0, d->stream>>>(d->tmp, tp, Wout, H, kv, stride, off, out, opitch, Hout); }
  return 0;
}

// A host frame being uploaded band by band on the copy stream (klt_dev_build); the fused kernels
// are launched over the tile rows each band completes, so the upload hides the image pipeline.
// All copies are queued first (the host must never starve the copy engine), then the kernels,
// each group gated by the event of the band that completes its source rows.
static constexpr int KLT_MAX_BANDS = 48;
struct BandFeed {
  const unsigned char* host;     // tightly packed W x H
  int W, H, fp;                  // fp: row pitch of d->frame
  int nbands, next;              // bands queued / bands the compute stream has been gated on
  int enqueued;                  // bands whose copies have been queued (pageable frames: one at a time)
  bool staged;                   // pageable frame: goes through the pinned staging buffer
  int end_row[KLT_MAX_BANDS];    // band b covers rows [end_row[b-1], end_row[b])
  cudaEvent_t ev[KLT_MAX_BANDS];
};
// band schedule: mode > 0: equal bands of `mode` rows; mode == 0: one copy; mode < 0: automatic --
// frames of >= 4 MB go in two bands, 60 % / 40 % (everything behind the last band is exposed
// latency, but every extra band costs four kernel boundaries at 7-12 us each while a copy is in
// flight; measured best on B200), smaller frames in one copy
static void feed_schedule(BandFeed* f, int mode) {
  const int H = f->H;
  f->nbands = 0;
  if (mode > 0) {
    const int rows = (mode + 63) / 64 * 64;
    int r = 0;
    while (r < H && f->nbands < KLT_MAX_BANDS - 1) {
      int take = rows;
      const int left = H - r;
      if (left > rows && left < rows + rows / 2) take = left - rows / 2;   // keep the last band short
      if (take > left) take = left;
      r += take;
      f->end_row[f->nbands++] = r;
    }
    if (r < H) f->end_row[f->nbands++] = H;
  } else if (mode < 0 && (long)f->W * H >= 4L * 1000 * 1000) {
    static float frac[8] = {0.6f};
    static int nfrac = 1;
    static bool parsed = false;
    if (!parsed) {                 // tuning hook: KLT_B200_BAND_FRACS="0.3,0.6,0.85"
      parsed = true;
      const char* e = getenv("KLT_B200_BAND_FRACS");
      if (e && *e) {
        nfrac = 0;
        while (*e && nfrac < 8) {
          char* end = nullptr;
          const float v = strtof(e, &end);
          if (end == e) break;
          frac[nfrac++] = v;
          e = (*end == ',') ? end + 1 : end;
        }
      }
    }
    for (int i = 0; i < nfrac; ++i) {
      int r = (int)(frac[i] * H) / 64 * 64;
      if (r > 0 && r < H && (f->nbands == 0 || r > f->end_row[f->nbands - 1])) f->end_row[f->nbands++] = r;
    }
    f->end_row[f->nbands++] = H;
  } else {
    f->end_row[f->nbands++] = H;
  }
}
// Pageable host memory: cudaMemcpyAsync would stage it through the driver's own bounce buffers
// synchronously at ~10 GB/s (905 us per 4K frame, measured).  One host thread copies at 17 GB/s,
// four at 62 GB/s (tools/memcpy_probe.c), so the frame is copied into a pinned staging buffer by
// a few OpenMP threads in 2 MB chunks, each chunk's DMA queued as soon as it is staged
// (4K call: 867 us -> 412 us with 4 threads, 380 us with 8; pinned frames: 241 us).
static bool host_ptr_is_pageable(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return at.type == cudaMemoryTypeUnregistered;
}
// A pageable frame pointer: remember it; the second time the same buffer (address and size) comes
// in, page-lock it in place.  Returns true when the buffer is page-locked now.
static bool host_frame_register(klt_dev* d, const void* p, size_t bytes) {
  if (!d->reg_frames) return false;
  klt_dev::HostReg* slot = nullptr;
  klt_dev::HostReg* victim = &d->hreg[0];
  for (int i = 0; i < KLT_HOST_REGS; ++i) {
    klt_dev::HostReg& r = d->hreg[i];
    if (r.p == p && r.bytes == bytes) { slot = &r; break; }
    if (!r.registered && (victim->registered || r.stamp < victim->stamp)) victim = &r;
  }
  d->reg_clock += 1;
  if (!slot) {
    if (victim->registered) return false;            // table full of live registrations: keep staging
    victim->p = p; victim->bytes = bytes; victim->seen = 1; victim->stamp = d->reg_clock;
    return false;
  }
  slot->stamp = d->reg_clock;
  if (slot->seen < 0) return false;                   // registration failed before: do not retry
  slot->seen += 1;
  if (slot->seen < 2) return false;
  if (cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterDefault) != cudaSuccess) {
    cudaGetLastError();
    slot->seen = -1;
    return false;
  }
  slot->registered = 1;
  d->last_registered += 1;
  return true;
}
extern "C" int klt_dev_forget_host_frames(klt_dev* d) {
  if (!d) return 0;
  bool any = false;
  for (int i = 0; i < KLT_HOST_REGS; ++i) any = any || d->hreg[i].registered;
  if (any) {
    CU(cudaSetDevice(d->device));
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    for (int i = 0; i < KLT_HOST_REGS; ++i)
      if (d->hreg[i].registered && cudaHostUnregister(const_cast<void*>(d->hreg[i].p)) != cudaSuccess) cudaGetLastError();
  }
  memset(d->hreg, 0, sizeof(d->hreg));
  return 0;
}
extern "C" int klt_dev_registered_host_frames(const klt_dev* d) {
  int n = 0;
  for (int i = 0; i < KLT_HOST_REGS; ++i) n += d->hreg[i].registered;
  return n;
}
extern "C" void klt_dev_set_register_frames(klt_dev* d, int on) { d->reg_frames = on; }
#include "klt_stage.h"
static void parallel_memcpy(unsigned char* dst, const unsigned char* src, size_t bytes, int nthreads) {
  stage_team().copy(dst, src, bytes, nthreads);
}
static int feat_flush(klt_dev* d);
static int feed_enqueue_band(klt_dev* d, BandFeed* f, int b) {
  const int r0 = b == 0 ? 0 : f->end_row[b - 1], r1 = f->end_row[b];
  if (!f->staged) {
    const int rows = r1 - r0;
    unsigned char* dst = d->frame + (size_t)r0 * f->fp;
    const unsigned char* src = f->host + (size_t)r0 * f->W;
    Launch l(d, KID_COPY_H2D, d->cstream);
    if (f->fp == f->W)
      CU(cudaMemcpyAsync(dst, src, (size_t)rows * f->W, cudaMemcpyHostToDevice, d->cstream));
    else
      CU(cudaMemcpy2DAsync(dst, f->fp, src, f->W, f->W, rows, cudaMemcpyHostToDevice, d->cstream));
  } else {
    static unsigned chunk_kb = getenv("KLT_B200_STAGE_CHUNK_KB") ? (unsigned)atoi(getenv("KLT_B200_STAGE_CHUNK_KB")) : 1024u;
    int chunk_rows = (int)((chunk_kb << 10) / (unsigned)f->W);
    if (chunk_rows < 1) chunk_rows = 1;
    for (int y = r0; y < r1; y += chunk_rows) {
      const int rows = (y + chunk_rows < r1 ? y + chunk_rows : r1) - y;
      unsigned char* stage = d->h_frame + (size_t)y * f->W;
      parallel_memcpy(stage, f->host + (size_t)y * f->W, (size_t)rows * f->W, d->stage_threads);
      unsigned char* dst = d->frame + (size_t)y * f->fp;
      Launch l(d, KID_COPY_H2D, d->cstream);
      if (f->fp == f->W)
        CU(cudaMemcpyAsync(dst, stage, (size_t)rows * f->W, cudaMemcpyHostToDevice, d->cstream));
      else
        CU(cudaMemcpy2DAsync(dst, f->fp, stage, f->W, f->W, rows, cudaMemcpyHostToDevice, d->cstream));
    }
    if (b == f->nbands - 1) {                 // staging buffer free again once the last DMA has read it
      CU(cudaEventRecord(d->ev_stage_free, d->cstream));
      d->stage_busy = 1;
    }
  }
  f->ev[b] = d->ev_band[d->band_ev_next];
  d->band_ev_next = (d->band_ev_next + 1) % KLT_BAND_EVENTS;
  CU(cudaEventRecord(f->ev[b], d->cstream));
  f->enqueued = b + 1;
  if (b == f->nbands - 1 && feat_flush(d)) return 1;   // the committed feature upload goes behind the frame
  return 0;
}
static int feed_enqueue_copies(klt_dev* d, BandFeed* f) {
  if (d->frame_busy[d->frame_idx]) {          // the previous build's level-0 kernels may still read d->frame
    CU(cudaStreamWaitEvent(d->cstream, d->ev_frame_free[d->frame_idx], 0));
    d->frame_busy[d->frame_idx] = 0;
  }
  f->next = 0; f->enqueued = 0;
  const size_t bytes = (size_t)f->W * f->H;
  bool pageable = bytes >= (1u << 20) && host_ptr_is_pageable(f->host);
  if (pageable && host_frame_register(d, f->host, bytes)) pageable = false;
  f->staged = d->stage_threads > 0 && pageable;
  d->last_staged = f->staged ? 1 : 0;
  if (f->staged) {
    if (d->h_frame_cap < bytes) {
      if (sync_all(d)) return fail(d, "stream synchronisation failed");
      cudaFreeHost(d->h_frame); d->h_frame = nullptr; d->h_frame_cap = 0;
      CU(cudaHostAlloc(&d->h_frame, bytes, cudaHostAllocDefault));
      d->h_frame_cap = bytes;
      d->stage_busy = 0;
    }
    if (d->stage_busy) { CU(cudaEventSynchronize(d->ev_stage_free)); d->stage_busy = 0; }
    return 0;                   // bands are staged and queued one at a time, each followed by its kernels
  }
  for (int b = 0; b < f->nbands; ++b)
    if (feed_enqueue_band(d, f, b)) return 1;
  return 0;
}
// gate the compute stream on the next band (or on all of them); returns the rows then available
static int feed_wait(klt_dev* d, BandFeed* f, bool all, int* rows) {
  do {
    if (f->next >= f->enqueued && feed_enqueue_band(d, f, f->next)) return 1;
    CU(cudaStreamWaitEvent(d->stream, f->ev[f->next], 0));
    f->next += 1;
  } while (all && f->next < f->nbands);
  *rows = f->end_row[f->next - 1];
  return 0;
}

template <bool EXACT>
static int build_impl(klt_dev* d, PyrSet& S, const unsigned char* src, int spitch,
                      const klt_dev_build_desc* q, BandFeed* feed) {
  const int W = q->ncols, H = q->nrows;
  bool tiled_all = true, done = false;
  const int nb = q->nlevels_built;
  TapsR ts, tp;
  memset(&ts, 0, sizeof(ts)); memset(&tp, 0, sizeof(tp));
  if (q->smooth) ts = reversed(q->smooth_taps.gauss, q->smooth_taps.gauss_width);
  if (nb > 1) tp = reversed(q->pyramid_taps.gauss, q->pyramid_taps.gauss_width);
  const TapsR tg = reversed(q->grad_taps.gauss, q->grad_taps.gauss_width);
  const TapsR td = reversed(q->grad_taps.deriv, q->grad_taps.deriv_width);
  FusedPlan P;
  d->last_fused = 0;
  d->last_bands = 0;
  fused_plan(d, S, src, spitch, q, ts, tp, tg, td, &P);
  bool all_fused = P.l0_ok;
  for (int l = 1; l < nb; ++l) all_fused = all_fused && P.shape[l] != SHAPE_NONE;

  if (all_fused) {
    // every level runs on the fused kernels: launch whole tile rows as soon as their source rows
    // exist -- all at once for a resident frame, band by band behind the upload of a host frame
    int rows_done[KLT_DEV_MAX_LEVELS] = {0};
    int valid[KLT_DEV_MAX_LEVELS + 1] = {0};          // rows written so far of each plane of P's band schedule
    auto plane_h = [&](int p) { return p == 0 ? H : S.lv[p - 1].h; };
    valid[0] = feed ? 0 : H;
    if (feed && feed_enqueue_copies(d, feed)) return 1;
    do {
      if (feed && feed_wait(d, feed, false, &valid[0])) return 1;
      for (int l = 0; l < nb; ++l) {
        const int sp = P.src_plane[l];
        int j = rows_done[l];
        while (j < P.tiles_y[l]) {
          int need = P.need_mul[l] * (j + 1) + P.need_add[l];
          if (need > plane_h(sp)) need = plane_h(sp);
          if (need > valid[sp]) break;
          ++j;
        }
        if (l == 0 ? l0_fused_launch<EXACT>(d, P, W, H, ts, tg, td, tp, S, rows_done[0], j)
                   : level_launch<EXACT>(d, P, S, l, nb, tp, tg, td, rows_done[l], j))
          return 1;
        rows_done[l] = j;
        if (l + 1 < nb) {
          const int np = P.src_plane[l + 1];
          valid[np] = P.made_mul[l] * j < plane_h(np) ? P.made_mul[l] * j : plane_h(np);
        }
      }
    } while (valid[0] < H);
    if (feed) {
      d->last_bands = feed->nbands;
      CU(cudaEventRecord(d->ev_frame_free[d->frame_idx], d->stream));
      d->frame_busy[d->frame_idx] = 1;
    }
    for (int l = 0; l < nb; ++l)
      if (rows_done[l] != P.tiles_y[l]) return fail(d, "banded build left level %d incomplete", l);
    d->last_fused = nb;
    d->last_path = 1;
    return 0;
  }

  // ---- mixed / generic path: the whole frame must be on the device -----------------------------
  if (feed) {
    int rows = 0;
    feed->nbands = 1; feed->end_row[0] = H;
    if (feed_enqueue_copies(d, feed) || feed_wait(d, feed, true, &rows)) return 1;
    d->last_bands = 1;
  }
  int grad_from = 0;                 // first level whose gradients are still to be computed
  if (P.l0_ok) {
    if (l0_fused_launch<EXACT>(d, P, W, H, ts, tg, td, tp, S, 0, P.tiles_y[0])) return 1;
    grad_from = 1;
  }
  d->last_fused = grad_from;
  if (grad_from == 1) {
    // nothing left to do for level 0
  } else if (q->smooth) {
    done = false;
    if (!d->force_generic)
      if (smooth_u8_dispatch<EXACT>(d, src, spitch, W, H, ts, S.lv[0].img, S.lv[0].pitch, &done)) return 1;
    if (!done) {
      tiled_all = false;
      if (generic_separable<unsigned char, EXACT>(d, src, spitch, W, H, ts, ts, 1, S.lv[0].img,
                                                  S.lv[0].pitch, W, H)) return 1;
    }
  } else {
    dim3 b(32, 8), g((W + 31) / 32, (H + 7) / 8);
    Launch l(d, KID_U8_TO_F32);
    u8_to_f32_kernel<<<g, b, 0, d->stream>>>(src, spitch, W, H, S.lv[0].img, S.lv[0].pitch);
  }
  if (feed) {                        // d->frame has been consumed by the level-0 kernel(s) above
    CU(cudaEventRecord(d->ev_frame_free[d->frame_idx], d->stream));
    d->frame_busy[d->frame_idx] = 1;
  }
  // coarser levels
  bool grads_done[KLT_DEV_MAX_LEVELS] = {false};
  grads_done[0] = (grad_from == 1);
  for (int l = 1; l < nb; ++l) {
    const Level& a = S.lv[l - 1];
    const Level& b = S.lv[l];
    if (P.shape[l] != SHAPE_NONE) {
      if (level_launch<EXACT>(d, P, S, l, nb, tp, tg, td, 0, P.tiles_y[l])) return 1;
      grads_done[l] = true; d->last_fused += 1;
      continue;
    }
    done = false;
    if (!d->force_generic)
      if (pyrdown_dispatch<EXACT>(d, q->subsampling, a.img, a.pitch, a.w, a.h, tp, b.img, b.pitch,
                                  b.w, b.h, &done)) return 1;
    if (!done) {
      tiled_all = false;
      if (generic_separable<float, EXACT>(d, a.img, a.pitch, a.w, a.h, tp, tp, q->subsampling,
                                          b.img, b.pitch, b.w, b.h)) return 1;
    }
  }
  // gradients
  for (int l = 0; l < nb; ++l) {
    if (grads_done[l]) continue;
    const Level& a = S.lv[l];
    done = false;
    if (!d->force_generic)
      if (grad_dispatch<EXACT>(d, a.img, a.pitch, a.w, a.h, tg, td, a.gx, a.gy, a.pitch, &done)) return 1;
    if (!done) {
      tiled_all = false;
      if (generic_separable<float, EXACT>(d, a.img, a.pitch, a.w, a.h, td, tg, 1, a.gx, a.pitch, a.w, a.h)) return 1;
      if (generic_separable<float, EXACT>(d, a.img, a.pitch, a.w, a.h, tg, td, 1, a.gy, a.pitch, a.w, a.h)) return 1;
    }
  }
  d->last_path = tiled_all ? 1 : 0;
  return 0;
}

static int check_taps(klt_dev* d, const klt_dev_taps& t, const char* what) {
  if (t.gauss_width < 1 || t.gauss_width > KLT_DEV_MAX_TAPS || !(t.gauss_width & 1) ||
      t.deriv_width < 1 || t.deriv_width > KLT_DEV_MAX_TAPS || !(t.deriv_width & 1))
    return fail(d, "%s taps have invalid widths %d/%d", what, t.gauss_width, t.deriv_width);
  return 0;
}

extern "C" int klt_dev_build(klt_dev* d, int slot, const unsigned char* img, int img_is_device,
                             size_t img_pitch, const klt_dev_build_desc* q) {
  if (!d || !q || !img) return fail(d, "klt_dev_build: null argument");
  if (slot < 0 || slot >= KLT_DEV_SLOTS) return fail(d, "klt_dev_build: slot %d", slot);
  CU(cudaSetDevice(d->device));
  if (q->nlevels_built < 1 || q->nlevels_built > q->nlevels) return fail(d, "nlevels_built %d of %d", q->nlevels_built, q->nlevels);
  if (check_taps(d, q->grad_taps, "gradient")) return 1;
  if (q->smooth && check_taps(d, q->smooth_taps, "smoothing")) return 1;
  if (q->nlevels_built > 1 && check_taps(d, q->pyramid_taps, "pyramid")) return 1;
  if (ensure_geometry(d, q->ncols, q->nrows, q->nlevels, q->subsampling)) return 1;
  const int W = q->ncols, H = q->nrows;
  const unsigned char* src = img;
  int spitch = (int)img_pitch;
  BandFeed feed;
  memset(&feed, 0, sizeof(feed));
  if (!img_is_device) {
    const int fp = (W + 15) / 16 * 16;          // TMA needs a 16 B multiple row pitch
    const size_t bytes = (size_t)fp * H;
    if (d->frame_cap < bytes) {
      if (sync_all(d)) return fail(d, "stream synchronisation failed");
      for (int i = 0; i < 2; ++i) { cudaFree(d->frame_buf[i]); d->frame_buf[i] = nullptr; d->frame_busy[i] = 0; }
      d->frame = nullptr; d->frame_cap = 0;
      for (int i = 0; i < 2; ++i) CU(cudaMalloc(&d->frame_buf[i], bytes));
      d->frame_cap = bytes;
    }
    d->frame_idx ^= 1;                          // the other buffer may still be read by the previous build
    d->frame = d->frame_buf[d->frame_idx];
    // uploaded inside build_impl: band by band on the copy stream when every level runs fused
    feed.host = img; feed.W = W; feed.H = H; feed.fp = fp;
    feed_schedule(&feed, d->band_rows);
    d->frame_pitch = fp;
    src = d->frame;
    spitch = fp;
  } else if (spitch < W) {
    return fail(d, "device frame pitch %d < width %d", spitch, W);
  }
  PyrSet& S = d->set[slot];
  S.built_levels = 0;
  d->building_slot = slot;
  if (d->overlap && d->read_pending[slot]) {          // a tracker on the other stream may still read it
    CU(cudaStreamWaitEvent(d->stream, d->ev_read[slot], 0));
    d->read_pending[slot] = 0;
  }
  BandFeed* fp_ = img_is_device ? nullptr : &feed;
  const int rc = q->exact ? build_impl<true>(d, S, src, spitch, q, fp_) : build_impl<false>(d, S, src, spitch, q, fp_);
  if (rc) return rc;
  CU(cudaGetLastError());
  if (d->overlap) {
    CU(cudaEventRecord(d->ev_built[slot], d->stream));
    d->built_pending[slot] = 1;
  }
  S.built_levels = q->nlevels_built;
  S.src = src; S.spitch = spitch; S.desc = *q;
  {
    // |gradient| <= 255 * sum|smoothing taps|^2 * sum|derivative taps| * sum|Gaussian taps|: bounds the
    // eigenvalue keys of a selection on this slot (how many radix passes the sort needs)
    double sg = 0.0, sd = 0.0, ss = 1.0;
    for (int i = 0; i < q->grad_taps.gauss_width; ++i) sg += fabs((double)q->grad_taps.gauss[i]);
    for (int i = 0; i < q->grad_taps.deriv_width; ++i) sd += fabs((double)q->grad_taps.deriv[i]);
    if (q->smooth) { ss = 0.0; for (int i = 0; i < q->smooth_taps.gauss_width; ++i) ss += fabs((double)q->smooth_taps.gauss[i]); }
    S.grad_bound = 255.0 * ss * ss * sd * sg;
  }
  return 0;
}

extern "C" int klt_dev_read_level(klt_dev* d, int slot, int which, int level, float* out) {
  if (!d->arena || slot < 0 || slot >= KLT_DEV_SLOTS || level < 0 || level >= d->L) return fail(d, "read_level: bad slot/level");
  CU(cudaSetDevice(d->device));
  const Level& lv = d->set[slot].lv[level];
  const float* src = which == 0 ? lv.img : which == 1 ? lv.gx : lv.gy;
  CU(cudaMemcpy2DAsync(out, (size_t)lv.w * sizeof(float), src, (size_t)lv.pitch * sizeof(float),
                       (size_t)lv.w * sizeof(float), lv.h, cudaMemcpyDeviceToHost, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  return 0;
}

// ---- features --------------------------------------------------------------------
// device and pinned-host staging hold x | y | val back to back (one copy each way)
static int ensure_features(klt_dev* d, int n) {
  if (n <= d->feat_cap) return 0;
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  guarded_free(d, d->d_x);
  cudaFreeHost(d->h_x);
  d->d_x = d->d_y = nullptr; d->d_val = nullptr; d->h_x = d->h_y = nullptr; d->h_val = nullptr;
  d->feat_cap = 0;
  const int cap = (n + 1023) / 1024 * 1024;
  CU(guarded_malloc(d, &d->d_x, (size_t)cap * 12));
  CU(cudaMallocHost(&d->h_x, (size_t)cap * 12));
  d->d_y = d->d_x + cap; d->d_val = reinterpret_cast<int*>(d->d_y + cap);
  d->h_y = d->h_x + cap; d->h_val = reinterpret_cast<int*>(d->h_y + cap);
  d->feat_cap = cap;
  return 0;
}

// the pinned staging area is reused by every call: wait for copies that may still read/write it
static int staging_quiesce(klt_dev* d) {
  if (d->staging_busy) {
    CU(cudaStreamSynchronize(d->tstream));
    d->staging_busy = 0;
  }
  return 0;
}

extern "C" int klt_dev_features_upload(klt_dev* d, int n, const float* x, const float* y, const int* val) {
  CU(cudaSetDevice(d->device));
  if (n < 0) return fail(d, "negative feature count");
  if (ensure_features(d, n > 0 ? n : 1)) return 1;
  if (staging_quiesce(d)) return 1;
  d->feat_deferred = 0;                               // (a committed but never queued upload is superseded)
  memcpy(d->h_x, x, n * sizeof(float));
  memcpy(d->h_y, y, n * sizeof(float));
  memcpy(d->h_val, val, n * sizeof(int));
  CU(cudaMemcpyAsync(d->d_x, d->h_x, (size_t)d->feat_cap * 12, cudaMemcpyHostToDevice, d->tstream));
  d->staging_busy = 1;
  d->feat_out_host = 0;
  d->feat_n = n;
  return 0;
}

// staging access for the C host layer: it packs the feature list straight into pinned memory
extern "C" int klt_dev_features_staging(klt_dev* d, int n, float** x, float** y, int** val) {
  CU(cudaSetDevice(d->device));
  if (ensure_features(d, n > 0 ? n : 1)) return 1;
  if (staging_quiesce(d)) return 1;
  *x = d->h_x; *y = d->h_y; *val = d->h_val;
  return 0;
}
// queue the committed feature upload on the copy stream now (behind whatever is already there)
static int feat_flush(klt_dev* d) {
  if (!d->feat_deferred) return 0;
  d->feat_deferred = 0;
  if (d->feat_def_bytes > 0) {
    Launch l(d, KID_COPY_H2D, d->cstream);
    CU(cudaMemcpyAsync(d->feat_def_dst, d->feat_def_src, d->feat_def_bytes, cudaMemcpyHostToDevice, d->cstream));
  }
  CU(cudaEventRecord(d->ev_feat, d->cstream));
  d->feat_pending = 1;
  return 0;
}
extern "C" int klt_dev_features_commit(klt_dev* d, int n) {      // H2D of the staging area (async)
  CU(cudaSetDevice(d->device));
  if (n > d->feat_cap) return fail(d, "commit of %d features, capacity %d", n, d->feat_cap);
  // on the copy stream, BEHIND the bands of the frame the next klt_dev_build uploads (feat_flush):
  // only the tracker needs the features, and it runs after the last band's kernels anyway; ahead of
  // the frame the copy would delay every byte of it (12 us of a 235 us call at 4K / 4096 features)
  d->feat_deferred = 1; d->feat_def_dst = d->d_x; d->feat_def_src = d->h_x; d->feat_def_bytes = (size_t)d->feat_cap * 12;
  d->staging_busy = 1;
  d->feat_out_host = 1;
  d->feat_n = n;
  return 0;
}
// record mode: the feature list lives in pinned host memory (klt_dev_host_alloc).  The records are
// mirrored to the device in one copy (behind the frame bands on the copy stream), the tracker reads
// the mirror and writes x | y | val of every live feature straight into the caller's records.
extern "C" int klt_dev_features_commit_records(klt_dev* d, int n, void* first_record, size_t stride_bytes) {
  CU(cudaSetDevice(d->device));
  if (n < 0 || (stride_bytes & 3) || stride_bytes < 12) return fail(d, "commit_records: bad count / stride");
  const size_t bytes = (size_t)n * stride_bytes;
  if (d->d_rec_cap < bytes) {
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    cudaFree(d->d_rec); d->d_rec = nullptr; d->d_rec_cap = 0;
    CU(cudaMalloc(&d->d_rec, bytes ? bytes : 16));
    d->d_rec_cap = bytes ? bytes : 16;
  }
  d->feat_deferred = 1; d->feat_def_dst = d->d_rec; d->feat_def_src = first_record; d->feat_def_bytes = bytes;
  d->feat_out_host = 2;
  d->h_rec = first_record;
  d->rec_stride = (int)(stride_bytes / 4);
  d->feat_n = n;
  return 0;
}
extern "C" void* klt_dev_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (klt_dev_count() < 1) return nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
extern "C" void klt_dev_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int klt_dev_features_fetch(klt_dev* d, int n) {       // D2H into the staging area + sync
  CU(cudaSetDevice(d->device));
  if (n > d->feat_n) return fail(d, "download of %d features but %d resident", n, d->feat_n);
  if (feat_flush(d)) return 1;
  if (d->feat_out_host == 0) {
    Launch l(d, KID_COPY_D2H, d->tstream);
    CU(cudaMemcpyAsync(d->h_x, d->d_x, (size_t)d->feat_cap * 12, cudaMemcpyDeviceToHost, d->tstream));
  }                                   // else: the tracker wrote its results into the staging area
  CU(cudaStreamSynchronize(d->tstream));
  if (d->feat_pending) { CU(cudaStreamSynchronize(d->cstream)); d->feat_pending = 0; }
  if (d->overlap) CU(cudaStreamSynchronize(d->stream));
  d->staging_busy = 0;
  return 0;
}

// pipelined drivers: a ring of pinned snapshots of the resident features (x | y | val, `capacity`
// entries each).  push queues the copy of the current state into a ring slot behind the work queued
// so far and records the slot's event; wait blocks until that copy has landed.  The host thread
// consumes frame k - depth while frames k - depth + 1 .. k are still queued or running.
extern "C" int klt_dev_features_capacity(const klt_dev* d) { return d->feat_cap; }
extern "C" int klt_dev_snapshot_ring(klt_dev* d, int depth) {
  CU(cudaSetDevice(d->device));
  if (depth < 1 || depth > KLT_SNAP_MAX) return fail(d, "snapshot ring depth %d (1..%d)", depth, KLT_SNAP_MAX);
  if (d->feat_cap <= 0) return fail(d, "snapshot ring: no device-resident features");
  const size_t bytes = (size_t)depth * d->feat_cap * 12;
  if (d->snap_bytes < bytes) {
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    cudaFreeHost(d->snap_ring); d->snap_ring = nullptr; d->snap_bytes = 0;
    CU(cudaHostAlloc(&d->snap_ring, bytes, cudaHostAllocDefault));
    d->snap_bytes = bytes;
  }
  for (int i = d->snap_events; i < depth; ++i) {
    CU(cudaEventCreateWithFlags(&d->ev_snap[i], cudaEventDisableTiming));
    d->snap_events = i + 1;
  }
  d->snap_depth = depth;
  return 0;
}
extern "C" int klt_dev_snapshot_push(klt_dev* d, int slot) {
  CU(cudaSetDevice(d->device));
  if (slot < 0 || slot >= d->snap_depth || d->feat_out_host != 0) return fail(d, "snapshot_push: slot %d of %d", slot, d->snap_depth);
  { Launch l(d, KID_COPY_D2H, d->tstream);
    CU(cudaMemcpyAsync(d->snap_ring + (size_t)slot * d->feat_cap * 12, d->d_x, (size_t)d->feat_cap * 12,
                       cudaMemcpyDeviceToHost, d->tstream)); }
  CU(cudaEventRecord(d->ev_snap[slot], d->tstream));
  return 0;
}
extern "C" int klt_dev_snapshot_wait(klt_dev* d, int slot, const float** x, const float** y, const int** val) {
  if (slot < 0 || slot >= d->snap_depth) return fail(d, "snapshot_wait: slot %d of %d", slot, d->snap_depth);
  CU(cudaEventSynchronize(d->ev_snap[slot]));
  const float* base = reinterpret_cast<const float*>(d->snap_ring + (size_t)slot * d->feat_cap * 12);
  *x = base; *y = base + d->feat_cap; *val = reinterpret_cast<const int*>(base + 2 * (size_t)d->feat_cap);
  return 0;
}

extern "C" int klt_dev_features_download(klt_dev* d, int n, float* x, float* y, int* val) {
  if (klt_dev_features_fetch(d, n)) return 1;
  memcpy(x, d->h_x, n * sizeof(float));
  memcpy(y, d->h_y, n * sizeof(float));
  memcpy(val, d->h_val, n * sizeof(int));
  return 0;
}

static void make_view(const PyrSet& S, int L, PyrView* v) {
  memset(v, 0, sizeof(*v));
  for (int l = 0; l < L; ++l) {
    v->img[l] = S.lv[l].img; v->gx[l] = S.lv[l].gx; v->gy[l] = S.lv[l].gy;
    v->ncols[l] = S.lv[l].w; v->nrows[l] = S.lv[l].h; v->pitch[l] = S.lv[l].pitch;
  }
}

// where the tracker records its results: the device arrays (resident pipelines) or, for the
// synchronous API, straight into the pinned host staging area (posted writes over PCIe, no D2H copy)
static FeatIO feat_io(klt_dev* d) {
  FeatIO io;
  if (d->feat_out_host == 2) {              // record mode: device mirror in, the caller's pinned records out
    const float* in = reinterpret_cast<const float*>(d->d_rec);
    float* out = reinterpret_cast<float*>(d->h_rec);
    io.x = in; io.y = in + 1; io.val = reinterpret_cast<const int*>(in + 2); io.istride = d->rec_stride;
    io.ox = out; io.oy = out + 1; io.oval = reinterpret_cast<int*>(out + 2); io.ostride = d->rec_stride;
  } else {
    io.x = d->d_x; io.y = d->d_y; io.val = d->d_val; io.istride = 1;
    io.ox = d->feat_out_host ? d->h_x : d->d_x;
    io.oy = d->feat_out_host ? d->h_y : d->d_y;
    io.oval = d->feat_out_host ? d->h_val : d->d_val;
    io.ostride = 1;
  }
  return io;
}

static FbArgs fb_args(const klt_dev* d) {
  FbArgs f;
  f.rec = d->d_fb; f.max_error = d->fb_max_error;
  return f;
}

template <bool EXACT, int PPL, bool FB, bool PRED>
static int launch_track(klt_dev* d, const PyrView& v1, const PyrView& v2, const TrackArgs& a, int n) {
  const int warps = 4;
  const size_t smem = EXACT ? (size_t)warps * 3 * a.ww * a.wh * sizeof(float) : 0;
  if (set_smem(d, track_kernel<EXACT, PPL, FB, PRED>, smem)) return 1;
  { Launch l(d, KID_TRACK, d->tstream);
    track_kernel<EXACT, PPL, FB, PRED><<<(n + warps - 1) / warps, warps * 32, smem, d->tstream>>>(
        v1, v2, a, n, feat_io(d), d->d_live, fb_args(d), d->pred); }
  return 0;
}
template <bool EXACT, int PPL>
static int launch_track(klt_dev* d, const PyrView& v1, const PyrView& v2, const TrackArgs& a, int n, bool fb, bool pred) {
  if (pred) return fb ? launch_track<EXACT, PPL, true, true>(d, v1, v2, a, n) : launch_track<EXACT, PPL, false, true>(d, v1, v2, a, n);
  return fb ? launch_track<EXACT, PPL, true, false>(d, v1, v2, a, n) : launch_track<EXACT, PPL, false, false>(d, v1, v2, a, n);
}

template <int WW, int RPL, bool FB, bool PRED>
static void launch_track_fast_t(klt_dev* d, const PyrView& v1, const PyrView& v2, const TrackArgs& a, int n) {
  track_fast_kernel<WW, RPL, FB, PRED><<<(8 * n + 127) / 128, 128, 0, d->tstream>>>(
      v1, v2, a, n, feat_io(d), d->d_live, fb_args(d), d->pred);
}
template <int WW, int RPL>
static void launch_track_fast_t(klt_dev* d, const PyrView& v1, const PyrView& v2, const TrackArgs& a, int n, bool fb, bool pred) {
  Launch l(d, KID_TRACK_FAST, d->tstream);
  if (pred) fb ? launch_track_fast_t<WW, RPL, true, true>(d, v1, v2, a, n) : launch_track_fast_t<WW, RPL, false, true>(d, v1, v2, a, n);
  else fb ? launch_track_fast_t<WW, RPL, true, false>(d, v1, v2, a, n) : launch_track_fast_t<WW, RPL, false, false>(d, v1, v2, a, n);
}
// square odd windows up to 15x15; returns false if this window has no instantiation
static bool launch_track_fast(klt_dev* d, const PyrView& v1, const PyrView& v2, const TrackArgs& a, int n, bool fb, bool pred) {
  switch (a.ww) {
    case 3: launch_track_fast_t<3, 1>(d, v1, v2, a, n, fb, pred); return true;
    case 5: launch_track_fast_t<5, 1>(d, v1, v2, a, n, fb, pred); return true;
    case 7:
      if (d->track7_off) { launch_track_fast_t<7, 1>(d, v1, v2, a, n, fb, pred); return true; }
      if (!d->no_track7w) {                                  // one warp per feature, scalar loads
        Launch l(d, KID_TRACK7W, d->tstream);
        launch_k(pred ? (fb ? track7w_kernel<true, true> : track7w_kernel<false, true>)
                      : (fb ? track7w_kernel<true, false> : track7w_kernel<false, false>),
                 dim3((n + 3) / 4), dim3(128), 0, d->tstream,
                 d->pdl != 0 && !d->overlap, v1, v2, a, n, feat_io(d), d->d_live, fb_args(d), d->pred);
        return true;
      }
      launch_track_fast_t<7, 1>(d, v1, v2, a, n, fb, pred);
      return true;
    case 9: launch_track_fast_t<9, 2>(d, v1, v2, a, n, fb, pred); return true;
    case 11: launch_track_fast_t<11, 2>(d, v1, v2, a, n, fb, pred); return true;
    case 13: launch_track_fast_t<13, 2>(d, v1, v2, a, n, fb, pred); return true;
    case 15: launch_track_fast_t<15, 2>(d, v1, v2, a, n, fb, pred); return true;
    default: return false;
  }
}

static void fill_track_args(const klt_dev* d, const klt_dev_track_params* p, TrackArgs* a) {
  memset(a, 0, sizeof(*a));
  a->nlevels = d->L; a->ss = (float)d->ss; a->ww = p->window_width; a->wh = p->window_height;
  a->step_factor = p->step_factor; a->max_iterations = p->max_iterations;
  a->min_determinant = p->min_determinant; a->min_displacement = p->min_displacement;
  a->max_residue = p->max_residue; a->borderx = p->borderx; a->bordery = p->bordery;
  a->ncols = d->W; a->nrows = d->H;
  a->lighting = p->lighting_insensitive ? 1 : 0;
  { static int keep = getenv("KLT_TRACK_L2_KEEP") ? atoi(getenv("KLT_TRACK_L2_KEEP")) : 1; a->l2_keep = keep; }
}
extern "C" void klt_dev_disable_track7w(klt_dev* d, int on) { d->no_track7w = on; }
extern "C" int klt_dev_track_resident(klt_dev* d, int slot_prev, int slot_cur,
                                      const klt_dev_track_params* p) {
  CU(cudaSetDevice(d->device));
  if (!klt_dev_slot_valid(d, slot_prev) || !klt_dev_slot_valid(d, slot_cur))
    return fail(d, "klt_dev_track: pyramid slot %d or %d not built", slot_prev, slot_cur);
  if (p->window_width < 3 || p->window_height < 3 || !(p->window_width & 1) || !(p->window_height & 1))
    return fail(d, "tracking window %d x %d must be odd and >= 3", p->window_width, p->window_height);
  const int n = d->feat_n;
  const bool fb = p->fb_max_error > 0.0f;
  d->fb_n = fb ? n : -1;
  d->fb_max_error = p->fb_max_error;
  const int guess_n = d->guess_n;                    // explicit guesses are consumed by this call
  d->guess_n = -1;
  if (p->predict < 0 || p->predict > 1) return fail(d, "klt_dev_track: predict = %d (0: none, 1: velocity)", p->predict);
  if (guess_n >= 0 && guess_n != n)
    return fail(d, "klt_dev_track: %d guesses queued for a call on %d features", guess_n, n);
  const bool pred = p->predict != 0 || guess_n >= 0;
  d->pred_n = pred ? n : -1;
  if (!pred) d->vel_n = 0;                           // this call leaves the velocity records behind
  if (n == 0) return 0;
  if (fb && d->fb_cap < n) {                         // the check's result records (klt_dev_fb_results)
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    guarded_free(d, d->d_fb); d->d_fb = nullptr; d->fb_cap = 0;
    const int cap = (n + 1023) / 1024 * 1024;
    CU(guarded_malloc(d, &d->d_fb, (size_t)cap * sizeof(FbRec)));
    d->fb_cap = cap;
  }
  if (pred && d->pred_cap < n) {                     // the prior's records: new ones hold no velocity
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    guarded_free(d, d->d_vel); guarded_free(d, d->d_pred); d->d_vel = nullptr; d->d_pred = nullptr;
    d->pred_cap = 0; d->vel_n = 0;
    const int cap = (n + 1023) / 1024 * 1024;
    CU(guarded_malloc(d, &d->d_vel, (size_t)cap * sizeof(PredVel)));
    CU(guarded_malloc(d, &d->d_pred, (size_t)cap * sizeof(PredRec)));
    d->pred_cap = cap;
  }
  float* const guesses = d->d_guess + (size_t)d->guess_slot * 2 * d->guess_cap;
  d->pred.gx = guess_n >= 0 ? guesses : nullptr;
  d->pred.gy = guess_n >= 0 ? guesses + d->guess_cap : nullptr;
  d->pred.vel = d->d_vel; d->pred.rec = d->d_pred;
  d->pred.vel_n = p->predict == 1 ? d->vel_n : 0;
  if (pred) d->vel_n = n;                            // the tracker writes the records of features 0 .. n-1
  if (feat_flush(d)) return 1;
  if (d->feat_pending) {                             // features uploaded on the copy stream
    CU(cudaStreamWaitEvent(d->tstream, d->ev_feat, 0));
    d->feat_pending = 0;
  }
  if (d->overlap) {                                  // the pyramids are produced on the other stream
    const int sl[2] = {slot_prev, slot_cur};
    for (int k = 0; k < 2; ++k)
      if (d->built_pending[sl[k]]) {                  // once waited for, stream order covers later trackers
        CU(cudaStreamWaitEvent(d->tstream, d->ev_built[sl[k]], 0));
        d->built_pending[sl[k]] = 0;
      }
  }
  PyrView v1, v2;
  make_view(d->set[slot_prev], d->L, &v1);
  make_view(d->set[slot_cur], d->L, &v2);
  TrackArgs a;
  fill_track_args(d, p, &a);
  const int npix = a.ww * a.wh;
  const int ppl = (npix + 31) / 32;
  int rc;
  if (p->exact) {
    if (ppl <= 2) rc = launch_track<true, 2>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 4) rc = launch_track<true, 4>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 8) rc = launch_track<true, 8>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 16) rc = launch_track<true, 16>(d, v1, v2, a, n, fb, pred);
    else return fail(d, "tracking window %d x %d too large (max 512 pixels)", a.ww, a.wh);
  } else if (!d->force_generic && !a.lighting && a.ww == a.wh && a.ww <= 15 && launch_track_fast(d, v1, v2, a, n, fb, pred)) {
    rc = 0;
  } else {
    if (ppl <= 2) rc = launch_track<false, 2>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 4) rc = launch_track<false, 4>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 8) rc = launch_track<false, 8>(d, v1, v2, a, n, fb, pred);
    else if (ppl <= 16) rc = launch_track<false, 16>(d, v1, v2, a, n, fb, pred);
    else return fail(d, "tracking window %d x %d too large (max 512 pixels)", a.ww, a.wh);
  }
  if (rc) return rc;
  CU(cudaGetLastError());
  if (guess_n >= 0) CU(cudaEventRecord(d->ev_guess[d->guess_slot], d->tstream));   // the slot's last reader
  if (d->overlap) {
    CU(cudaEventRecord(d->ev_read[slot_prev], d->tstream));
    CU(cudaEventRecord(d->ev_read[slot_cur], d->tstream));
    d->read_pending[slot_prev] = d->read_pending[slot_cur] = 1;
  }
  return 0;
}

extern "C" int klt_dev_fb_results(klt_dev* d, int n, float* xb, float* yb, float* err, int* back_val) {
  CU(cudaSetDevice(d->device));
  if (d->fb_n < 0) return fail(d, "fb_results: the last tracking call did not run the forward-backward check");
  if (n != d->fb_n) return fail(d, "fb_results: %d features requested, the last tracking call had %d", n, d->fb_n);
  if (n == 0) return 0;
  FbRec* h = (FbRec*)malloc((size_t)n * sizeof(FbRec));
  if (!h) return fail(d, "out of host memory");
  cudaError_t e = cudaMemcpyAsync(h, d->d_fb, (size_t)n * sizeof(FbRec), cudaMemcpyDeviceToHost, d->tstream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(d->tstream);
  if (e != cudaSuccess) { free(h); return fail(d, "fb_results: %s", cudaGetErrorString(e)); }
  for (int i = 0; i < n; ++i) {
    if (xb) xb[i] = h[i].xb;
    if (yb) yb[i] = h[i].yb;
    if (err) err[i] = h[i].err;
    if (back_val) back_val[i] = h[i].back_val;
  }
  free(h);
  return 0;
}

// Pipelined drivers queue the guesses of step k + 1 while step k's tracker may not have run yet: the
// guesses go into the other slot of the ring, and a slot is refilled only after the tracker that
// read it (and the copy that filled it) has finished -- the host waits for that, so it runs at most
// two tracking calls with explicit guesses ahead of the device.
extern "C" int klt_dev_set_guesses(klt_dev* d, int n, const float* gx, const float* gy, int on_device) {
  CU(cudaSetDevice(d->device));
  if (n < 0 || (n > 0 && (!gx || !gy))) return fail(d, "set_guesses: bad count or NULL array");
  if (!d->ev_guess[0])
    for (int i = 0; i < 2; ++i) CU(cudaEventCreateWithFlags(&d->ev_guess[i], cudaEventDisableTiming));
  if (d->guess_cap < n) {
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    guarded_free(d, d->d_guess); cudaFreeHost(d->h_guess);
    d->d_guess = nullptr; d->h_guess = nullptr; d->guess_cap = 0; d->guess_busy[0] = d->guess_busy[1] = 0;
    const int cap = (n + 1023) / 1024 * 1024;
    CU(guarded_malloc(d, &d->d_guess, (size_t)cap * 4 * sizeof(float)));
    CU(cudaMallocHost(&d->h_guess, (size_t)cap * 4 * sizeof(float)));
    d->guess_cap = cap;
  }
  const int s = d->guess_slot ^ 1;
  if (d->guess_busy[s]) { CU(cudaEventSynchronize(d->ev_guess[s])); d->guess_busy[s] = 0; }
  float* dst = d->d_guess + (size_t)s * 2 * d->guess_cap;
  if (n > 0) {                 // on the copy stream like the feature upload: the tracker waits for ev_feat
    const float *sx = gx, *sy = gy;
    cudaMemcpyKind kind = cudaMemcpyDeviceToDevice;
    if (!on_device) {          // through pinned staging: the copy is asynchronous, the caller's arrays free
      float* h = d->h_guess + (size_t)s * 2 * d->guess_cap;
      memcpy(h, gx, (size_t)n * sizeof(float));
      memcpy(h + d->guess_cap, gy, (size_t)n * sizeof(float));
      sx = h; sy = h + d->guess_cap; kind = cudaMemcpyHostToDevice;
    }
    CU(cudaMemcpyAsync(dst, sx, (size_t)n * sizeof(float), kind, d->cstream));
    CU(cudaMemcpyAsync(dst + d->guess_cap, sy, (size_t)n * sizeof(float), kind, d->cstream));
    CU(cudaEventRecord(d->ev_guess[s], d->cstream));
    d->guess_busy[s] = 1;
    CU(cudaEventRecord(d->ev_feat, d->cstream));
    d->feat_pending = 1;
  }
  d->guess_n = n;
  d->guess_slot = s;
  return 0;
}

extern "C" int klt_dev_guesses_pending(const klt_dev* d) { return d->guess_n; }

extern "C" int klt_dev_prediction_results(klt_dev* d, int n, float* gx, float* gy, int* source) {
  CU(cudaSetDevice(d->device));
  if (d->pred_n < 0) return fail(d, "prediction_results: the last tracking call ran without prediction");
  if (n != d->pred_n) return fail(d, "prediction_results: %d features requested, the last tracking call had %d", n, d->pred_n);
  if (n == 0) return 0;
  PredRec* h = (PredRec*)malloc((size_t)n * sizeof(PredRec));
  if (!h) return fail(d, "out of host memory");
  cudaError_t e = cudaMemcpyAsync(h, d->d_pred, (size_t)n * sizeof(PredRec), cudaMemcpyDeviceToHost, d->tstream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(d->tstream);
  if (e != cudaSuccess) { free(h); return fail(d, "prediction_results: %s", cudaGetErrorString(e)); }
  for (int i = 0; i < n; ++i) {
    if (gx) gx[i] = h[i].gx;
    if (gy) gy[i] = h[i].gy;
    if (source) source[i] = h[i].source;
  }
  free(h);
  return 0;
}

extern "C" int klt_dev_track(klt_dev* d, int slot_prev, int slot_cur, const klt_dev_track_params* p,
                             int n, float* x, float* y, int* val) {
  if (klt_dev_features_upload(d, n, x, y, val)) return 1;
  if (klt_dev_track_resident(d, slot_prev, slot_cur, p)) return 1;
  return klt_dev_features_download(d, n, x, y, val);
}

// ---- affine consistency check (reference trackFeatures.c:1438-1497) ---------------------------
// Protocol of one KLTTrackFeatures call with tc->affineConsistencyCheck >= 0:
//   features committed (staging mode) -> klt_dev_affine_begin (returns the pinned per-feature state
//   array for the host to fill; keeps the tracker's output on the device and saves the positions
//   before tracking) -> [klt_dev_affine_put_template for templates the device does not mirror]
//   -> klt_dev_track_resident -> klt_dev_affine_check -> klt_dev_features_fetch (synchronises)
//   -> the host reads the state array (flags: 1 template created, 2 released) and fetches created
//   templates with klt_dev_affine_get_template(s).
static_assert(sizeof(AffState) == sizeof(klt_dev_affine_state), "affine state layout");
extern "C" int klt_dev_affine_begin(klt_dev* d, int n, const klt_dev_affine_params* ap, klt_dev_affine_state** staging) {
  CU(cudaSetDevice(d->device));
  if (!ap || n <= 0 || n != d->feat_n) return fail(d, "affine_begin: %d features but %d committed", n, d->feat_n);
  if (ap->window_width < 3 || ap->window_height < 3 || !(ap->window_width & 1) || !(ap->window_height & 1) ||
      ap->window_width * ap->window_height > 2048)
    return fail(d, "affine window %d x %d must be odd, >= 3 and at most 2048 pixels", ap->window_width, ap->window_height);
  const int tsz = (ap->window_width + 2) * (ap->window_height + 2);
  if (d->aff_cap < n || d->aff_tsz != tsz) {
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    cudaFree(d->d_aff_st); cudaFreeHost(d->h_aff_st); cudaFree(d->d_aff_tmpl);
    d->d_aff_st = nullptr; d->h_aff_st = nullptr; d->d_aff_tmpl = nullptr; d->aff_cap = 0;
    const int cap = (n + 1023) / 1024 * 1024;
    CU(cudaMalloc(&d->d_aff_st, (size_t)cap * sizeof(AffState)));
    CU(cudaMallocHost(&d->h_aff_st, (size_t)cap * sizeof(AffState)));
    CU(cudaMalloc(&d->d_aff_tmpl, (size_t)cap * 3 * tsz * sizeof(float)));
    d->aff_cap = cap; d->aff_tsz = tsz;
  }
  if (d->aff_x0_cap < d->feat_cap) {
    if (sync_all(d)) return fail(d, "stream synchronisation failed");
    cudaFree(d->d_x0); d->d_x0 = nullptr; d->aff_x0_cap = 0;
    CU(cudaMalloc(&d->d_x0, (size_t)d->feat_cap * 12));
    d->aff_x0_cap = d->feat_cap;
  }
  if (d->feat_out_host == 2) return fail(d, "affine_begin: record-mode features (use the staging area)");
  d->feat_out_host = 0;                              // the check needs the tracker's answers on the device
  if (feat_flush(d)) return 1;
  if (d->feat_pending) {
    CU(cudaStreamWaitEvent(d->tstream, d->ev_feat, 0));
    d->feat_pending = 0;
  }
  CU(cudaMemcpyAsync(d->d_x0, d->d_x, (size_t)d->feat_cap * 12, cudaMemcpyDeviceToDevice, d->tstream));
  *staging = reinterpret_cast<klt_dev_affine_state*>(d->h_aff_st);
  return 0;
}
extern "C" int klt_dev_affine_put_template(klt_dev* d, int i, const float* img, const float* gx, const float* gy) {
  CU(cudaSetDevice(d->device));
  if (i < 0 || i >= d->aff_cap || !img || !gx || !gy) return fail(d, "affine_put_template: feature %d", i);
  const size_t tb = (size_t)d->aff_tsz * sizeof(float);
  float* dst = d->d_aff_tmpl + (size_t)i * 3 * d->aff_tsz;
  CU(cudaMemcpyAsync(dst, img, tb, cudaMemcpyHostToDevice, d->tstream));
  CU(cudaMemcpyAsync(dst + d->aff_tsz, gx, tb, cudaMemcpyHostToDevice, d->tstream));
  CU(cudaMemcpyAsync(dst + 2 * d->aff_tsz, gy, tb, cudaMemcpyHostToDevice, d->tstream));
  return 0;
}
static int affine_check_core(klt_dev* d, int slot_prev, int slot_cur, const klt_dev_track_params* tp,
                             const klt_dev_affine_params* ap, bool resident);
extern "C" int klt_dev_affine_check(klt_dev* d, int slot_prev, int slot_cur, const klt_dev_track_params* tp,
                                    const klt_dev_affine_params* ap) {
  return affine_check_core(d, slot_prev, slot_cur, tp, ap, false);
}
// ---- the check inside the resident / sequence pipeline: the per-feature state stays on the device ----
// klt_dev_affine_begin + the staging array + klt_dev_affine_put_template set it up as for the per-call
// API; klt_dev_affine_upload_states sends the state up ONCE; then, per frame,
// klt_dev_affine_keep_positions (before the tracker: the positions the templates are cut at),
// klt_dev_track_resident, klt_dev_affine_check_resident; klt_dev_affine_fetch_states at the end.  The
// kernel keeps `has` itself (a lost feature releases its template, a first successful track cuts one),
// which is all the host does between the calls of the per-call API.
extern "C" int klt_dev_affine_upload_states(klt_dev* d, int n) {
  CU(cudaSetDevice(d->device));
  if (n <= 0 || d->aff_cap < n) return fail(d, "affine_upload_states without affine_begin");
  Launch l(d, KID_COPY_H2D, d->tstream);
  CU(cudaMemcpyAsync(d->d_aff_st, d->h_aff_st, (size_t)n * sizeof(AffState), cudaMemcpyHostToDevice, d->tstream));
  return 0;
}
extern "C" int klt_dev_affine_keep_positions(klt_dev* d) {
  CU(cudaSetDevice(d->device));
  if (!d->d_x0 || d->aff_x0_cap < d->feat_cap) return fail(d, "affine_keep_positions without affine_begin");
  CU(cudaMemcpyAsync(d->d_x0, d->d_x, (size_t)d->feat_cap * 12, cudaMemcpyDeviceToDevice, d->tstream));
  return 0;
}
extern "C" int klt_dev_affine_check_resident(klt_dev* d, int slot_prev, int slot_cur, const klt_dev_track_params* tp,
                                             const klt_dev_affine_params* ap) {
  return affine_check_core(d, slot_prev, slot_cur, tp, ap, true);
}
extern "C" int klt_dev_affine_fetch_states(klt_dev* d, int n, klt_dev_affine_state** staging) {
  CU(cudaSetDevice(d->device));
  if (n <= 0 || d->aff_cap < n || !staging) return fail(d, "affine_fetch_states without affine_begin");
  { Launch l(d, KID_COPY_D2H, d->tstream);
    CU(cudaMemcpyAsync(d->h_aff_st, d->d_aff_st, (size_t)n * sizeof(AffState), cudaMemcpyDeviceToHost, d->tstream)); }
  CU(cudaStreamSynchronize(d->tstream));
  *staging = reinterpret_cast<klt_dev_affine_state*>(d->h_aff_st);
  return 0;
}
static int affine_check_core(klt_dev* d, int slot_prev, int slot_cur, const klt_dev_track_params* tp,
                             const klt_dev_affine_params* ap, bool resident) {
  CU(cudaSetDevice(d->device));
  if (!klt_dev_slot_valid(d, slot_prev) || !klt_dev_slot_valid(d, slot_cur))
    return fail(d, "affine_check: pyramid slot %d or %d not built", slot_prev, slot_cur);
  const int n = d->feat_n;
  if (n <= 0 || d->aff_cap < n || !d->d_x0) return fail(d, "affine_check without affine_begin");
  AffArgs a;
  memset(&a, 0, sizeof(a));
  a.check = ap->check; a.aw = ap->window_width; a.ah = ap->window_height; a.max_iterations = ap->max_iterations;
  a.max_residue = ap->max_residue; a.th_aff = ap->min_displacement; a.mdd = ap->max_displacement_differ;
  a.step_factor = tp->step_factor; a.small = tp->min_determinant; a.th = tp->min_displacement;
  a.nlevels = d->L; a.ss = (float)d->ss;
  a.resident = resident ? 1 : 0;
  a.lighting = tp->lighting_insensitive ? 1 : 0;
  const Level& l1 = d->set[slot_prev].lv[0];
  const Level& l2 = d->set[slot_cur].lv[0];
  a.ncols = l2.w; a.nrows = l2.h; a.pitch = l2.pitch;
  if (l1.pitch != l2.pitch) return fail(d, "affine_check: level-0 pitches differ");
  a.i1 = l1.img; a.gx1 = l1.gx; a.gy1 = l1.gy;
  a.i2 = l2.img; a.gx2 = l2.gx; a.gy2 = l2.gy;
  const int warps = 4;
  const size_t smem = (size_t)warps * (3 * a.aw * a.ah + 48) * sizeof(float);
  if (set_smem(d, affine_check_kernel, smem)) return 1;
  if (!resident) {
    Launch l(d, KID_COPY_H2D, d->tstream);
    CU(cudaMemcpyAsync(d->d_aff_st, d->h_aff_st, (size_t)n * sizeof(AffState), cudaMemcpyHostToDevice, d->tstream));
  }
  { Launch l(d, KID_AFFINE, d->tstream);
    const float* x0 = d->d_x0;
    affine_check_kernel<<<(n + warps - 1) / warps, warps * 32, smem, d->tstream>>>(
        a, n, x0, x0 + d->feat_cap, reinterpret_cast<const int*>(x0 + 2 * (size_t)d->feat_cap),
        d->d_x, d->d_y, d->d_val, d->d_aff_st, d->d_aff_tmpl); }
  CU(cudaGetLastError());
  if (!resident) {
    Launch l(d, KID_COPY_D2H, d->tstream);
    CU(cudaMemcpyAsync(d->h_aff_st, d->d_aff_st, (size_t)n * sizeof(AffState), cudaMemcpyDeviceToHost, d->tstream));
  }
  return 0;
}
// after the call's synchronisation: template i (image, gradx, grady: (w+2)(h+2) floats each)
extern "C" int klt_dev_affine_get_template(klt_dev* d, int i, float* img, float* gx, float* gy) {
  CU(cudaSetDevice(d->device));
  if (i < 0 || i >= d->aff_cap) return fail(d, "affine_get_template: feature %d", i);
  const size_t tb = (size_t)d->aff_tsz * sizeof(float);
  const float* src = d->d_aff_tmpl + (size_t)i * 3 * d->aff_tsz;
  CU(cudaMemcpyAsync(img, src, tb, cudaMemcpyDeviceToHost, d->tstream));
  CU(cudaMemcpyAsync(gx, src + d->aff_tsz, tb, cudaMemcpyDeviceToHost, d->tstream));
  CU(cudaMemcpyAsync(gy, src + 2 * d->aff_tsz, tb, cudaMemcpyDeviceToHost, d->tstream));
  CU(cudaStreamSynchronize(d->tstream));
  return 0;
}
// all templates of features [0, n) in one copy: n x 3 x (w+2)(h+2) floats
extern "C" int klt_dev_affine_get_templates(klt_dev* d, int n, float* all) {
  CU(cudaSetDevice(d->device));
  if (n < 0 || n > d->aff_cap || !all) return fail(d, "affine_get_templates: %d features", n);
  CU(cudaMemcpyAsync(all, d->d_aff_tmpl, (size_t)n * 3 * d->aff_tsz * sizeof(float), cudaMemcpyDeviceToHost, d->tstream));
  CU(cudaStreamSynchronize(d->tstream));
  return 0;
}

// ---- selection --------------------------------------------------------------------
struct CandGeo { int bx, by, step, nxc, nyc; long npoints; };

static CandGeo cand_geometry(const klt_dev* d, const klt_dev_select_params* p) {
  CandGeo g;
  g.bx = p->borderx; g.by = p->bordery;
  if (g.bx < p->window_width / 2) g.bx = p->window_width / 2;
  if (g.by < p->window_height / 2) g.by = p->window_height / 2;
  g.step = p->nSkippedPixels + 1;
  const int spanx = d->W - 2 * g.bx, spany = d->H - 2 * g.by;
  g.nxc = spanx > 0 ? (spanx + g.step - 1) / g.step : 0;
  g.nyc = spany > 0 ? (spany + g.step - 1) / g.step : 0;
  g.npoints = (long)g.nxc * g.nyc;
  return g;
}

static int ensure_candidates(klt_dev* d, size_t n) {
  if (n <= d->cand_cap) return 0;
  CU(cudaStreamSynchronize(d->stream));
  for (int i = 0; i < 2; ++i) { guarded_free(d, d->c_val[i]); guarded_free(d, d->c_idx[i]); d->c_val[i] = nullptr; d->c_idx[i] = nullptr; }
  cudaFree(d->cub_tmp); d->cub_tmp = nullptr; d->cand_cap = 0;
  for (int i = 0; i < 2; ++i) {
    CU(guarded_malloc(d, &d->c_val[i], n * sizeof(int)));
    CU(guarded_malloc(d, &d->c_idx[i], n * sizeof(unsigned)));
  }
  guarded_free(d, d->rank_list); guarded_free(d, d->sel_state); d->rank_list = nullptr; d->sel_state = nullptr;
  CU(guarded_malloc(d, &d->rank_list, n * sizeof(int)));
  CU(guarded_malloc(d, &d->sel_state, 8 * sizeof(int)));
  size_t bytes = 0, bytes2 = 0;
  CU(cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, d->c_val[0], d->c_val[1], d->c_idx[0],
                                               d->c_idx[1], (int)n, 0, 32, d->stream));
  CU(cub::DeviceSelect::If(nullptr, bytes2, thrust::counting_iterator<int>(0), d->rank_list, d->sel_state + 4,
                           (int)n, UncoveredOp{}, d->stream));
  if (bytes2 > bytes) bytes = bytes2;
  CU(cudaMalloc(&d->cub_tmp, bytes ? bytes : 16));
  d->cub_bytes = bytes;
  d->cand_cap = n;
  return 0;
}

// covered (replacement only): the minimum-distance map with the surviving features already stamped.
// A candidate under a stamp can never be accepted, whatever its key (selectGoodFeatures.c:176-177), so
// its key is written as 0 -- below every threshold: the sort moves all of them behind the live
// candidates and the walk stops in front of them, without a separate filter pass over the sorted list
// (80 us per 4K call, 21 us at 640x480).
static int run_mineig(klt_dev* d, int slot, const klt_dev_select_params* p, const CandGeo& g, int clamp_neg,
                      const unsigned char* covered = nullptr) {
  const Level& lv = d->set[slot].lv[0];
  CU(cudaMemsetAsync(d->sel_state + 5, 0, 2 * sizeof(int), d->stream));        // key range: max, min
  dim3 b(32, 8), grid((g.nxc + 31) / 32, (g.nyc + 7) / 8);
  if (p->window_width / 2 == 3 && p->window_height / 2 == 3 && g.step == 1 && g.bx >= 8 && g.by >= 3 &&
      (lv.pitch & 31) == 0 && ((g.bx + g.nxc - 1) & ~7) + 12 <= lv.pitch &&      // the 16-column row loads stay inside the pitch
      !getenv("KLT_B200_MINEIG_SCALAR")) {
    const int span = g.bx + g.nxc - (g.bx & ~7);                               // columns from the first 8-aligned block on
    dim3 b7(32, 4), g7((span + 255) / 256, (g.nyc + 3) / 4);
    Launch l(d, KID_MINEIG);
    mineig7_kernel<<<g7, b7, 0, d->stream>>>(lv.gx, lv.gy, lv.pitch, g.bx, g.by, g.nxc, g.nyc, d->c_val[0], d->c_idx[0],
                                             d->sel_state + 5, clamp_neg, covered, d->W);
    return 0;
  }
  { Launch l(d, KID_MINEIG);
    mineig_kernel<<<grid, b, 0, d->stream>>>(lv.gx, lv.gy, lv.pitch, g.bx, g.by, g.step, g.nxc, g.nyc,
                                             p->window_width / 2, p->window_height / 2, d->c_val[0], d->c_idx[0],
                                             d->sel_state + 5, clamp_neg, covered, d->W); }
  return 0;
}

extern "C" int klt_dev_eigen_map(klt_dev* d, int slot, const klt_dev_select_params* p, int* out, int* npoints) {
  CU(cudaSetDevice(d->device));
  if (!d->arena || slot < 0 || slot >= KLT_DEV_SLOTS || d->set[slot].built_levels < 1) return fail(d, "eigen_map: slot %d has no level 0", slot);
  const CandGeo g = cand_geometry(d, p);
  if (npoints) *npoints = (int)g.npoints;
  if (!out || g.npoints == 0) return 0;
  if (ensure_candidates(d, (size_t)g.npoints)) return 1;
  if (run_mineig(d, slot, p, g, 0)) return 1;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, d->c_val[0], g.npoints * sizeof(int), cudaMemcpyDeviceToHost, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  return 0;
}

// selection over the features resident on the device (d_x | d_y | d_val): eigenvalue map, ranking,
// minimum-distance pass; host == nullptr leaves the result on the device (no synchronisation)
static int select_core(klt_dev* d, int slot, const klt_dev_select_params* p, int n,
                       float* x, float* y, int* val, bool host) {
  CU(cudaSetDevice(d->device));
  if (!d->arena || slot < 0 || slot >= KLT_DEV_SLOTS || d->set[slot].built_levels < 1) return fail(d, "select: slot %d has no level 0", slot);
  if (n <= 0) return 0;
  if (d->W > 65535 || d->H > 65535) return fail(d, "select: images larger than 65535 pixels a side are not supported");
  if (!d->enforce_attr) {
    CU(cudaFuncSetAttribute(enforce_mindist_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENFORCE_SMEM));
    CU(cudaFuncSetAttribute(enforce_mindist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENFORCE_SMEM));
    const char* nf = getenv("KLT_B200_NO_FILTER");   // A/B: walk the whole sorted list in one launch
    d->no_filter = (nf && nf[0] == '1') ? 1 : 0;
    { const char* rf = getenv("KLT_B200_REPLACE_FILTER"); d->replace_filter = (rf && rf[0] == '1') ? 1 : 0; }
    d->enforce_attr = 1;
  }
  cudaStream_t saved_t = d->tstream;
  if (d->overlap) { if (sync_all(d)) return fail(d, "stream synchronisation failed"); d->tstream = d->stream; }
  struct Restore { klt_dev* d; cudaStream_t t; ~Restore() { d->tstream = t; } } restore{d, saved_t};
  const CandGeo g = cand_geometry(d, p);
  int mindist = p->mindist < 0 ? 0 : p->mindist;
  const int dist = mindist - 1;                    // the reference works with mindist-1 (:157)
  const int min_eig = p->min_eigenvalue < 1 ? 1 : p->min_eigenvalue;   // (:148)
  if (host && klt_dev_features_upload(d, n, x, y, val)) return 1;
  if (!host && (n != d->feat_n || d->feat_out_host != 0)) return fail(d, "select_resident: %d features are not resident on the device", n);
  const size_t npx = (size_t)d->W * d->H;
  if (d->fmap_cap < npx) {
    CU(cudaStreamSynchronize(d->stream));
    guarded_free(d, d->fmap); d->fmap = nullptr; d->fmap_cap = 0;
    CU(guarded_malloc(d, &d->fmap, npx + 4));        // (+4: the stamps are written as 32-bit words)
    d->fmap_cap = npx;
  }
  if (d->open_cap < n) {
    CU(cudaStreamSynchronize(d->stream));
    guarded_free(d, d->open_slots); d->open_slots = nullptr; d->open_cap = 0;
    CU(guarded_malloc(d, &d->open_slots, (size_t)n * sizeof(int)));
    d->open_cap = n;
  }
  CU(cudaMemsetAsync(d->fmap, 0, npx, d->stream));
  const bool prestamp = !p->overwrite_all && !d->no_filter && !d->replace_filter;
  if (!p->overwrite_all && prestamp) {
    Launch l(d, KID_STAMP);
    stamp_existing_kernel<<<n, 128, 0, d->stream>>>(d->d_x, d->d_y, d->d_val, d->fmap, dist, d->W, d->H);
  }
  const int* sval = nullptr; const unsigned* sidx = nullptr;
  if (g.npoints > 0) {
    if (ensure_candidates(d, (size_t)g.npoints)) return 1;
    if (run_mineig(d, slot, p, g, 1, prestamp ? d->fmap : nullptr)) return 1;
    size_t bytes = d->cub_bytes;
    int end_bit = 32;
    {
      // keys <= (gxx + gyy) / 2 <= window pixels * bound^2 (with 1 % slack for the float roundings)
      const double gb = d->set[slot].grad_bound;
      const double kb = 1.01 * (double)p->window_width * (double)p->window_height * gb * gb + 2.0;
      if (gb > 0.0 && kb < 2147483647.0) { end_bit = 1; while (end_bit < 31 && ((long long)kb >> end_bit) != 0) ++end_bit; }
    }
    if (host) {
      // the synchronous API can afford one look at the key range: eigenvalues of 8-bit frames use
      // 15-21 bits, i.e. 2-3 radix passes instead of 4
      int range[2] = {0, 0};
      CU(cudaMemcpyAsync(range, d->sel_state + 5, sizeof(range), cudaMemcpyDeviceToHost, d->stream));
      CU(cudaStreamSynchronize(d->stream));
      if (range[1] >= 0) { end_bit = 1; while (end_bit < 31 && (range[0] >> end_bit) != 0) ++end_bit; }
      else end_bit = 32;
    }
    { Launch l(d, KID_SORT);   // several cub kernels, timed and counted as one
      CU(cub::DeviceRadixSort::SortPairsDescending(d->cub_tmp, bytes, d->c_val[0], d->c_val[1], d->c_idx[0],
                                                   d->c_idx[1], (int)g.npoints, 0, end_bit, d->stream)); }
    sval = d->c_val[1]; sidx = d->c_idx[1];
  }
  if (!p->overwrite_all && !prestamp) {
    Launch l(d, KID_STAMP);
    stamp_existing_kernel<<<n, 128, 0, d->stream>>>(d->d_x, d->d_y, d->d_val, d->fmap, dist, d->W, d->H);
  }
  {
    const int np = (int)g.npoints, nxc = g.nxc > 0 ? g.nxc : 1;
    // the candidates the featuremap does not cover yet, from list position `from` on, as ranks
    auto uncovered = [&](int from) -> int {
      Launch l(d, KID_FILTER);
      size_t bytes = d->cub_bytes;
      CU(cub::DeviceSelect::If(d->cub_tmp, bytes, thrust::counting_iterator<int>(from), d->rank_list, d->sel_state + 4,
                               np - from, UncoveredOp{sval, sidx, d->fmap, nxc, g.bx, g.by, g.step, d->W, min_eig},
                               d->stream));
      return 0;
    };
    auto walk = [&](bool indirect, int first, int last, int npts) {
      Launch l(d, KID_ENFORCE);
      if (indirect)
        enforce_mindist_kernel<true><<<1, GB, ENFORCE_SMEM, d->stream>>>(
            sval, sidx, d->rank_list, d->sel_state + 4, 0, nxc, g.bx, g.by, g.step, d->W, d->H, d->fmap, dist, min_eig,
            p->overwrite_all, n, d->d_x, d->d_y, d->d_val, d->open_slots, d->sel_state, first, last);
      else
        enforce_mindist_kernel<false><<<1, GB, ENFORCE_SMEM, d->stream>>>(
            sval, sidx, nullptr, nullptr, npts, nxc, g.bx, g.by, g.step, d->W, d->H, d->fmap, dist, min_eig,
            p->overwrite_all, n, d->d_x, d->d_y, d->d_val, d->open_slots, d->sel_state, first, last);
    };
    const int head = ENFORCE_HEAD;
    if (np > 0 && prestamp) {
      // replacement: the candidates under the surviving features' stamps carry key 0 (run_mineig) and
      // sit behind the live ones; the walk reads the sorted arrays directly and ends at the first dead key
      walk(false, 1, 1, np);
    } else if (np > 0 && !p->overwrite_all && !d->no_filter) {
      // (KLT_B200_REPLACE_FILTER=1, the round-1 path: filter the sorted list for uncovered candidates)
      if (uncovered(0)) return 1;
      walk(true, 1, 1, 0);
    } else if (np > 2 * head && !d->no_filter) {
      // selection: dense head of the list straight from the sorted arrays, the rest through the filter
      walk(false, 1, 0, head);
      int walk_done = 0;
      if (host) {
        // the synchronous API synchronises anyway: one look at the walk's state saves the filter
        // (81 us over the 7.5 M candidates of a 4K frame) whenever the list filled inside the head
        CU(cudaMemcpyAsync(&walk_done, d->sel_state + 1, sizeof(int), cudaMemcpyDeviceToHost, d->stream));
        CU(cudaStreamSynchronize(d->stream));
      }
      if (!walk_done && uncovered(head)) return 1;
      walk(true, 0, 1, 0);                       // (done: no candidates are read, only the open slots are padded)
    } else {
      walk(false, 1, 1, np);
    }
  }
  CU(cudaGetLastError());
  if (d->overlap) {
    // the selection ran on the build stream; the feature copies that follow (snapshot, fetch) are
    // queued on the tracker stream and must see its result
    CU(cudaEventRecord(d->ev_join, d->stream));
    CU(cudaStreamWaitEvent(saved_t, d->ev_join, 0));
  }
  return host ? klt_dev_features_download(d, n, x, y, val) : 0;
}
extern "C" int klt_dev_select(klt_dev* d, int slot, const klt_dev_select_params* p, int n,
                              float* x, float* y, int* val) {
  return select_core(d, slot, p, n, x, y, val, true);
}
// KLTReplaceLostFeatures / KLTSelectGoodFeatures on the device-resident feature arrays (pipelined
// drivers, klt_dev_features_upload ... klt_dev_features_download); nothing is synchronised
extern "C" int klt_dev_select_resident(klt_dev* d, int slot, const klt_dev_select_params* p) {
  return select_core(d, slot, p, d->feat_n, nullptr, nullptr, nullptr, false);
}

// KLTReplaceLostFeatures ranks candidates by the truncated-integer eigenvalues of the LAST TRACKED
// frame's level-0 gradients (reference selectGoodFeatures.c:342-348).  Tracking pyramids are built
// in fma arithmetic by default, and a 1-ulp gradient difference can move a key across an integer
// boundary, which re-orders the greedy minimum-distance pass.  So a replacement on a slot that was
// not built in exact arithmetic first rebuilds level 0 (image + gradients, same taps) in exact
// arithmetic from the u8 frame, which is still on the device, into the slot the next frame will
// overwrite anyway; *slot_out is the slot to select on.  76 us at 4K, 4 us at 640x480.
extern "C" int klt_dev_exact_level0(klt_dev* d, int slot, int* slot_out) {
  if (!d || !slot_out) return fail(d, "klt_dev_exact_level0: null argument");
  if (!d->arena || slot < 0 || slot >= KLT_DEV_SLOTS || d->set[slot].built_levels < 1)
    return fail(d, "exact_level0: slot %d has no level 0", slot);
  const PyrSet& S = d->set[slot];
  if (S.desc.exact) { *slot_out = slot; return 0; }
  if (!S.src) return fail(d, "exact_level0: the frame slot %d was built from is not known", slot);
  const int dst = (slot + 1) % KLT_DEV_SLOTS;
  klt_dev_build_desc q = S.desc;
  q.exact = 1; q.nlevels_built = 1;
  const unsigned char* src = S.src;
  if (klt_dev_build(d, dst, src, 1, (size_t)S.spitch, &q)) return 1;
  for (int i = 0; i < 2; ++i)                  // our own staging buffer: the next upload into it must wait
    if (src == d->frame_buf[i]) {
      CU(cudaEventRecord(d->ev_frame_free[i], d->stream));
      d->frame_busy[i] = 1;
    }
  *slot_out = dst;
  return 0;
}

// ---- device timing on the context stream (benches) ------------------------------
// CUDA events recorded on the stream the kernels are launched on; torch's own
// events would only see torch's current stream.
extern "C" int klt_dev_timer_start(klt_dev* d) {
  CU(cudaSetDevice(d->device));
  if (!d->ev_made) { CU(cudaEventCreate(&d->ev_a)); CU(cudaEventCreate(&d->ev_b)); d->ev_made = 1; }
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  CU(cudaEventRecord(d->ev_a, d->tstream));
  return 0;
}
extern "C" int klt_dev_timer_stop(klt_dev* d, float* ms) {
  CU(cudaSetDevice(d->device));
  if (!d->ev_made) return fail(d, "timer_stop without timer_start");
  if (d->overlap) {                 // everything queued on the build stream must be inside the interval
    CU(cudaEventRecord(d->ev_join, d->stream));
    CU(cudaStreamWaitEvent(d->tstream, d->ev_join, 0));
  }
  CU(cudaEventRecord(d->ev_b, d->tstream));
  CU(cudaEventSynchronize(d->ev_b));
  CU(cudaEventElapsedTime(ms, d->ev_a, d->ev_b));
  return 0;
}

// ---- per-kernel profiling -----------------------------------------------------------
extern "C" int klt_dev_profile_begin(klt_dev* d) {
  CU(cudaSetDevice(d->device));
  if (!d->prof_ev) {
    d->prof_ev = (cudaEvent_t*)calloc(2 * PROF_POOL, sizeof(cudaEvent_t));
    d->prof_kid = (int*)calloc(PROF_POOL, sizeof(int));
    if (!d->prof_ev || !d->prof_kid) return fail(d, "out of host memory");
    for (int i = 0; i < 2 * PROF_POOL; ++i) CU(cudaEventCreate(&d->prof_ev[i]));
    CU(cudaEventCreate(&d->ev_origin));
    d->trace_kid = (int*)calloc(TRACE_CAP, sizeof(int));
    d->trace_t0 = (float*)calloc(TRACE_CAP, sizeof(float));
    d->trace_t1 = (float*)calloc(TRACE_CAP, sizeof(float));
    if (!d->trace_kid || !d->trace_t0 || !d->trace_t1) return fail(d, "out of host memory");
  }
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  memset(d->prof_ms, 0, sizeof(d->prof_ms));
  memset(d->prof_n, 0, sizeof(d->prof_n));
  d->prof_used = 0;
  d->trace_n = 0;
  CU(cudaEventRecord(d->ev_origin, d->stream));
  d->prof_on = 1;
  return 0;
}
extern "C" int klt_dev_profile_end(klt_dev* d) {
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  prof_fold(d);
  d->prof_on = 0;
  return 0;
}
extern "C" int klt_dev_profile_kernels(void) { return KID_COUNT; }
extern "C" int klt_dev_trace_count(const klt_dev* d) { return d->trace_n; }
extern "C" const char* klt_dev_trace_get(const klt_dev* d, int i, float* t0_ms, float* t1_ms) {
  if (i < 0 || i >= d->trace_n) return nullptr;
  if (t0_ms) *t0_ms = d->trace_t0[i];
  if (t1_ms) *t1_ms = d->trace_t1[i];
  return kKernelNames[d->trace_kid[i]];
}
extern "C" const char* klt_dev_profile_get(const klt_dev* d, int kid, unsigned long long* launches, double* total_ms) {
  if (kid < 0 || kid >= KID_COUNT) return nullptr;
  if (launches) *launches = d->prof_n[kid];
  if (total_ms) *total_ms = d->prof_ms[kid];
  return kKernelNames[kid];
}
extern "C" int klt_dev_live_total(klt_dev* d, unsigned long long* out, int reset) {
  CU(cudaSetDevice(d->device));
  if (sync_all(d)) return fail(d, "stream synchronisation failed");
  CU(cudaMemcpyAsync(out, d->d_live, sizeof(*out), cudaMemcpyDeviceToHost, d->tstream));
  if (reset) CU(cudaMemsetAsync(d->d_live, 0, sizeof(*out), d->tstream));
  CU(cudaStreamSynchronize(d->tstream));
  return 0;
}
