// klt_motion.cuh -- global motion check: a RANSAC homography over the correspondences of one
// tracking call, with the features that disagree with it dropped on the device (DESIGN.md 4,
// "Global motion check").  Included by klt_dev.cu after the tracker kernels; the tracker itself is
// not touched.  Three launches on the tracker stream, right behind the tracker:
//   motion_prep_kernel   (one CTA)   correspondences {x0, y0, x1, y1} in feature-index order, m,
//                                    hypothesis counts zeroed, per-feature err = -1
//   motion_score_kernel  (grid)      hypothesis blocks x correspondence chunks: each thread solves one
//                                    hypothesis and counts its inliers in the CTA's chunk
//   motion_refine_kernel (one CTA)   winner, least-squares refinement over its inliers, classification,
//                                    outliers written into x | y | val, the frame's model record
// The arithmetic is the spec (tests/motion_oracle.py restates it): fp64 with separately rounded
// operations for the solves, separately rounded fp32 for the scores; it does not depend on the
// tracker's arithmetic mode.
#include <cub/block/block_scan.cuh>

#define KLT_B200_MOTION_OUTLIER -7   // include/klt_b200.h

constexpr int MOTION_PREP_THREADS = 1024;
constexpr int MOTION_SCORE_THREADS = 128;    // hypotheses per score CTA, one per thread
constexpr int MOTION_CHUNK = 128;            // correspondences per score CTA (profiles/r6_motion_chunk_sweep.json)
constexpr int MOTION_REFINE_THREADS = 256;
constexpr int MOTION_DRAWS = 16;             // draws per hypothesis for its 4 distinct indices
constexpr int MOTION_MIN_KEEP = 8;           // a model is applied when it keeps at least this many
constexpr double MOTION_COLLINEAR = 1e-6;    // |cross| of 3 normalised sample points below: degenerate
constexpr double MOTION_PIVOT = 1e-10;       // |pivot| below: singular system
constexpr int MOTION_SUMS = 23;              // distinct sums of the refinement's normal equations

// normalisation of pixel coordinates: (p - (cx, cy)) * s, cx = W/2, cy = H/2, s = 2 / max(W, H)
struct MotionGeo { double cx, cy, s; };
// the frame's model record (klt_dev_motion_model)
struct MotionModelRec { float H[9]; int valid, tracked, inliers, hypothesis; };

// lowbias32 (Chris Wellons' integer hash): the sampler's mixer
__device__ __forceinline__ unsigned motion_mix32(unsigned x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}

// Hypothesis h's sample: draws r = mix32(h * 16 + j), index (r * m) >> 32, the first 4 distinct
// indices in draw order; false when 16 draws give fewer.
__device__ __forceinline__ bool motion_sample(int h, int m, int (&s)[4]) {
  s[0] = s[1] = s[2] = s[3] = -1;
  int k = 0;
#pragma unroll
  for (int j = 0; j < MOTION_DRAWS; ++j) {
    const unsigned r = motion_mix32((unsigned)h * 16u + (unsigned)j);
    const int i = (int)(((unsigned long long)r * (unsigned)m) >> 32);
    if (k < 4 && i != s[0] && i != s[1] && i != s[2] && i != s[3]) {
      if (k == 0) s[0] = i; else if (k == 1) s[1] = i; else if (k == 2) s[2] = i; else s[3] = i;
      ++k;
    }
  }
  return k == 4;
}

__device__ __forceinline__ double motion_norm(float p, double c, double s) {
  return __dmul_rn(__dadd_rn((double)p, -c), s);
}
__device__ __forceinline__ double motion_cross(const double (&x)[4], const double (&y)[4], int a, int b, int c) {
  return __dadd_rn(__dmul_rn(__dadd_rn(x[b], -x[a]), __dadd_rn(y[c], -y[a])),
                   -__dmul_rn(__dadd_rn(y[b], -y[a]), __dadd_rn(x[c], -x[a])));
}
// true when any 3 of the 4 points are nearly collinear
__device__ __forceinline__ bool motion_degenerate(const double (&x)[4], const double (&y)[4]) {
  return fabs(motion_cross(x, y, 0, 1, 2)) < MOTION_COLLINEAR || fabs(motion_cross(x, y, 0, 1, 3)) < MOTION_COLLINEAR ||
         fabs(motion_cross(x, y, 0, 2, 3)) < MOTION_COLLINEAR || fabs(motion_cross(x, y, 1, 2, 3)) < MOTION_COLLINEAR;
}

// Gaussian elimination with partial pivoting of the augmented 8 x 9 system A (pivot: the largest |a|,
// the first on ties); false when a pivot is below MOTION_PIVOT.  Every index is a compile-time
// constant and the row swap is a conditional exchange with each candidate row.  A lives in the stack
// frame (576 bytes of L1-resident local memory): the division's slow path is a call, and no set of
// registers survives it that could hold 72 doubles.
__device__ __forceinline__ bool motion_solve8(double (&A)[8][9], double (&h)[8]) {
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    int p = k;
    double best = fabs(A[k][k]);
#pragma unroll
    for (int i = k + 1; i < 8; ++i) {
      const double a = fabs(A[i][k]);
      if (a > best) { best = a; p = i; }
    }
    ok = ok && best >= MOTION_PIVOT;
#pragma unroll
    for (int i = k + 1; i < 8; ++i)
      if (p == i) {
#pragma unroll
        for (int j = k; j < 9; ++j) { const double t = A[k][j]; A[k][j] = A[i][j]; A[i][j] = t; }
      }
#pragma unroll
    for (int i = k + 1; i < 8; ++i) {
      const double f = __ddiv_rn(A[i][k], A[k][k]);
#pragma unroll
      for (int j = k + 1; j < 9; ++j) A[i][j] = __dadd_rn(A[i][j], -__dmul_rn(f, A[k][j]));
    }
  }
#pragma unroll
  for (int i = 7; i >= 0; --i) {
    double s = A[i][8];
#pragma unroll
    for (int j = i + 1; j < 8; ++j) s = __dadd_rn(s, -__dmul_rn(A[i][j], h[j]));
    h[i] = __ddiv_rn(s, A[i][i]);
  }
  return ok;
}

// The normalised model n (n[8] = 1) in pixel coordinates, T^-1 n T with T the normalisation, scaled
// to H[8] = 1 and rounded to float; false when the scale is not finite and nonzero or an entry is
// not finite.
__device__ __forceinline__ bool motion_denorm(const double (&n)[8], const MotionGeo& g, float (&H)[8]) {
  const double ox = __dmul_rn(g.s, g.cx), oy = __dmul_rn(g.s, g.cy);
  double M[9];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double a = n[3 * r], b = n[3 * r + 1], c = r == 2 ? 1.0 : n[3 * r + 2];
    M[3 * r] = __dmul_rn(a, g.s);
    M[3 * r + 1] = __dmul_rn(b, g.s);
    M[3 * r + 2] = __dadd_rn(c, -__dadd_rn(__dmul_rn(a, ox), __dmul_rn(b, oy)));
  }
  double D[9];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    D[j] = __dadd_rn(__ddiv_rn(M[j], g.s), __dmul_rn(g.cx, M[6 + j]));
    D[3 + j] = __dadd_rn(__ddiv_rn(M[3 + j], g.s), __dmul_rn(g.cy, M[6 + j]));
    D[6 + j] = M[6 + j];
  }
  const double w = D[8];
  if (!(isfinite(w) && w != 0.0)) return false;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    H[k] = __double2float_rn(__ddiv_rn(D[k], w));
    ok = ok && isfinite(H[k]);
  }
  return ok;
}

// rows 2k, 2k + 1 of the DLT system (h22 = 1) for normalised (x, y) -> (u, v)
__device__ __forceinline__ void motion_rows(double (&A)[8][9], int k, double x, double y, double u, double v) {
#pragma unroll
  for (int j = 0; j < 9; ++j) { A[2 * k][j] = 0.0; A[2 * k + 1][j] = 0.0; }
  A[2 * k][0] = x; A[2 * k][1] = y; A[2 * k][2] = 1.0;
  A[2 * k][6] = -__dmul_rn(u, x); A[2 * k][7] = -__dmul_rn(u, y); A[2 * k][8] = u;
  A[2 * k + 1][3] = x; A[2 * k + 1][4] = y; A[2 * k + 1][5] = 1.0;
  A[2 * k + 1][6] = -__dmul_rn(v, x); A[2 * k + 1][7] = -__dmul_rn(v, y); A[2 * k + 1][8] = v;
}

// hypothesis h over the m correspondences: sample, degeneracy test, minimal solve, pixel model
// (out of line: inlined, the score kernel spills the values it keeps across the solve)
__device__ __noinline__ bool motion_hypothesis(int h, const float4* __restrict__ corr, int m, const MotionGeo& g,
                                               float (&H)[8]) {
  int s[4];
  if (!motion_sample(h, m, s)) return false;
  double px[4], py[4], qx[4], qy[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 c = corr[s[k]];
    px[k] = motion_norm(c.x, g.cx, g.s); py[k] = motion_norm(c.y, g.cy, g.s);
    qx[k] = motion_norm(c.z, g.cx, g.s); qy[k] = motion_norm(c.w, g.cy, g.s);
  }
  if (motion_degenerate(px, py) || motion_degenerate(qx, qy)) return false;
  double A[8][9];
#pragma unroll
  for (int k = 0; k < 4; ++k) motion_rows(A, k, px[k], py[k], qx[k], qy[k]);
  double n[8];
  if (!motion_solve8(A, n)) return false;
  return motion_denorm(n, g, H);
}

// squared reprojection distance of correspondence c under H, separately rounded float32; front: w > 0
__device__ __forceinline__ float motion_d2(const float (&H)[8], float4 c, bool& front) {
  const float u = __fadd_rn(__fadd_rn(__fmul_rn(H[0], c.x), __fmul_rn(H[1], c.y)), H[2]);
  const float v = __fadd_rn(__fadd_rn(__fmul_rn(H[3], c.x), __fmul_rn(H[4], c.y)), H[5]);
  const float w = __fadd_rn(__fadd_rn(__fmul_rn(H[6], c.x), __fmul_rn(H[7], c.y)), 1.0f);
  const float dx = __fsub_rn(__fdiv_rn(u, w), c.z), dy = __fsub_rn(__fdiv_rn(v, w), c.w);
  front = w > 0.0f;
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ bool motion_inlier(const float (&H)[8], float4 c, float e2) {
  bool front;
  const float d2 = motion_d2(H, c, front);
  return front && !(d2 > e2);
}

// The hypothesis state: hyp[0] = m, hyp[1 + h] the inlier count of hypothesis h, hyp[1 + cap + h] its
// validity (written by the score kernel), float model at hyp + 1 + 2 * cap + 8 h.
struct MotionHyp {
  int* base; int cap;
  __device__ int& m() const { return base[0]; }
  __device__ int& count(int h) const { return base[1 + h]; }
  __device__ int& valid(int h) const { return base[1 + cap + h]; }
  __device__ float* model(int h) const { return reinterpret_cast<float*>(base + 1 + 2 * cap) + 8 * (size_t)h; }
};

// x0 | y0 | val0 (the positions before the tracker, stride cap) and the tracker's x | y | val
__global__ void __launch_bounds__(MOTION_PREP_THREADS)
motion_prep_kernel(int n, int cap, const float* __restrict__ start, const float* __restrict__ x,
                   const float* __restrict__ y, const int* __restrict__ val, float4* __restrict__ corr,
                   int* __restrict__ cidx, float* __restrict__ err, MotionHyp hyp, int nhyp) {
  using Scan = cub::BlockScan<int, MOTION_PREP_THREADS>;
  __shared__ typename Scan::TempStorage tmp;
  const int* val0 = reinterpret_cast<const int*>(start + 2 * (size_t)cap);
  int m = 0;
  for (int base = 0; base < n; base += MOTION_PREP_THREADS) {
    const int f = base + threadIdx.x;
    const int take = f < n && val0[f] >= 0 && val[f] == KLT_TRACKED;
    int pos, total;
    Scan(tmp).ExclusiveSum(take, pos, total);
    if (take) {
      corr[m + pos] = make_float4(start[f], start[cap + f], x[f], y[f]);
      cidx[m + pos] = f;
    }
    if (f < n) err[f] = -1.0f;
    m += total;
    __syncthreads();                     // tmp is reused by the next tile's scan
  }
  if (threadIdx.x == 0) hyp.m() = m;
  for (int h = threadIdx.x; h < nhyp; h += MOTION_PREP_THREADS) hyp.count(h) = 0;
}

// blockIdx.x: hypotheses blockIdx.x * 128 + threadIdx.x; blockIdx.y: correspondences from
// blockIdx.y * MOTION_CHUNK.  The CTAs of chunk 0 also record each hypothesis' model and validity;
// the other chunks exit when they lie beyond m.  Every CTA solves its own hypotheses: one fp64 8 x 8
// solve per thread costs less than a score chunk and spreads over all SMs.
__global__ void __launch_bounds__(MOTION_SCORE_THREADS)
motion_score_kernel(const float4* __restrict__ corr, MotionHyp hyp, int nhyp, float e2, MotionGeo g) {
  __shared__ float4 s_c[MOTION_CHUNK];
  const int m = hyp.m();
  const int c0 = blockIdx.y * MOTION_CHUNK;
  const bool writer = blockIdx.y == 0;
  if (!writer && c0 >= m) return;
  const int h = blockIdx.x * MOTION_SCORE_THREADS + threadIdx.x;
  float H[8];
  bool valid = h < nhyp && motion_hypothesis(h, corr, m, g, H);
  if (writer && h < nhyp) {
    hyp.valid(h) = valid;
    if (valid) {
      float* o = hyp.model(h);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = H[k];
    }
  }
  const int cn = min(MOTION_CHUNK, m - c0);
  for (int i = threadIdx.x; i < cn; i += MOTION_SCORE_THREADS) s_c[i] = corr[c0 + i];
  __syncthreads();
  if (!valid) return;
  int cnt = 0;
#pragma unroll 4
  for (int i = 0; i < cn; ++i) cnt += motion_inlier(H, s_c[i], e2);
  if (cnt) atomicAdd(&hyp.count(h), cnt);
}

template <typename T>
__device__ __forceinline__ T motion_warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// One CTA.  The winner is the valid hypothesis with the most inliers, the lowest index on ties
// (invalid hypotheses are reported with count -1).  The refinement is one least-squares DLT over the
// winner's inliers: the normal equations' 23 distinct sums are accumulated per thread over a strided
// slice, reduced across each warp and then over the warps in order, and solved as the minimal
// system is; a singular system keeps the minimal model.  Every correspondence gets err = sqrt(d2)
// under the final model (+inf behind it, w <= 0); with >= MOTION_MIN_KEEP inliers the outliers become
// (-1, -1, KLT_B200_MOTION_OUTLIER).
__global__ void __launch_bounds__(MOTION_REFINE_THREADS)
motion_refine_kernel(const float4* __restrict__ corr, const int* __restrict__ cidx, MotionHyp hyp, int nhyp,
                     float e2, MotionGeo g, float* __restrict__ x, float* __restrict__ y, int* __restrict__ val,
                     float* __restrict__ err, MotionModelRec* __restrict__ rec) {
  constexpr int WARPS = MOTION_REFINE_THREADS / 32;
  __shared__ int s_bc[WARPS], s_bh[WARPS];
  __shared__ double s_sum[WARPS][MOTION_SUMS];
  __shared__ float s_H[8];
  __shared__ int s_win, s_keep;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int m = hyp.m();

  int bc = -1, bh = 0x7fffffff;                 // this thread's best, h ascending: first wins ties
  for (int h = tid; h < nhyp; h += MOTION_REFINE_THREADS) {
    int c = hyp.count(h);
    if (!hyp.valid(h)) { c = -1; hyp.count(h) = -1; }
    if (c > bc) { bc = c; bh = h; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const int oc = __shfl_down_sync(0xffffffffu, bc, o), oh = __shfl_down_sync(0xffffffffu, bh, o);
    if (oc > bc || (oc == bc && oh < bh)) { bc = oc; bh = oh; }
  }
  if (lane == 0) { s_bc[wid] = bc; s_bh[wid] = bh; }
  if (tid == 0) s_keep = 0;
  __syncthreads();
  if (tid == 0) {
    int c = s_bc[0], w = s_bh[0];
    for (int i = 1; i < WARPS; ++i)
      if (s_bc[i] > c || (s_bc[i] == c && s_bh[i] < w)) { c = s_bc[i]; w = s_bh[i]; }
    s_win = c >= 0 ? w : -1;
  }
  __syncthreads();
  const int win = s_win;
  if (win < 0) {                                 // no valid hypothesis: nothing is dropped, err stays -1
    if (tid == 0) {
      MotionModelRec r;
      for (int k = 0; k < 9; ++k) r.H[k] = __int_as_float(0x7fffffff);
      r.valid = 0; r.tracked = m; r.inliers = 0; r.hypothesis = -1;
      *rec = r;
    }
    return;
  }
  float H[8];
  {
    const float* w = hyp.model(win);
#pragma unroll
    for (int k = 0; k < 8; ++k) H[k] = w[k];
  }

  // refinement: the normal equations over the winner's inliers, in normalised coordinates
  double S[MOTION_SUMS];
#pragma unroll
  for (int k = 0; k < MOTION_SUMS; ++k) S[k] = 0.0;
  for (int i = tid; i < m; i += MOTION_REFINE_THREADS) {
    const float4 c = corr[i];
    if (!motion_inlier(H, c, e2)) continue;
    const double px = motion_norm(c.x, g.cx, g.s), py = motion_norm(c.y, g.cy, g.s);
    const double u = motion_norm(c.z, g.cx, g.s), v = motion_norm(c.w, g.cy, g.s);
    const double q = __dadd_rn(__dmul_rn(u, u), __dmul_rn(v, v));
    const double ux = __dmul_rn(u, px), uy = __dmul_rn(u, py), vx = __dmul_rn(v, px), vy = __dmul_rn(v, py);
    const double qx = __dmul_rn(q, px), qy = __dmul_rn(q, py);
    const double t[MOTION_SUMS] = {
        __dmul_rn(px, px), __dmul_rn(px, py), px, __dmul_rn(py, py), py, 1.0,
        __dmul_rn(ux, px), __dmul_rn(ux, py), __dmul_rn(uy, py), ux, uy,
        __dmul_rn(vx, px), __dmul_rn(vx, py), __dmul_rn(vy, py), vx, vy,
        __dmul_rn(qx, px), __dmul_rn(qx, py), __dmul_rn(qy, py), qx, qy, u, v};
#pragma unroll
    for (int k = 0; k < MOTION_SUMS; ++k) S[k] = __dadd_rn(S[k], t[k]);
  }
#pragma unroll
  for (int k = 0; k < MOTION_SUMS; ++k) {
    const double w = motion_warp_sum(S[k]);
    if (lane == 0) s_sum[wid][k] = w;
  }
  __syncthreads();
  if (tid == 0) {
    double T[MOTION_SUMS];
#pragma unroll
    for (int k = 0; k < MOTION_SUMS; ++k) {
      double a = s_sum[0][k];
      for (int i = 1; i < WARPS; ++i) a = __dadd_rn(a, s_sum[i][k]);
      T[k] = a;
    }
    enum { XX, XY, X, YY, Y, ONE, UXX, UXY, UYY, UX, UY, VXX, VXY, VYY, VX, VY, QXX, QXY, QYY, QX, QY, U, V };
    double A[8][9] = {
        {T[XX], T[XY], T[X], 0, 0, 0, -T[UXX], -T[UXY], T[UX]},
        {T[XY], T[YY], T[Y], 0, 0, 0, -T[UXY], -T[UYY], T[UY]},
        {T[X], T[Y], T[ONE], 0, 0, 0, -T[UX], -T[UY], T[U]},
        {0, 0, 0, T[XX], T[XY], T[X], -T[VXX], -T[VXY], T[VX]},
        {0, 0, 0, T[XY], T[YY], T[Y], -T[VXY], -T[VYY], T[VY]},
        {0, 0, 0, T[X], T[Y], T[ONE], -T[VX], -T[VY], T[V]},
        {-T[UXX], -T[UXY], -T[UX], -T[VXX], -T[VXY], -T[VX], T[QXX], T[QXY], -T[QX]},
        {-T[UXY], -T[UYY], -T[UY], -T[VXY], -T[VYY], -T[VY], T[QXY], T[QYY], -T[QY]}};
    double n[8];
    float R[8];
    const bool refined = motion_solve8(A, n) && motion_denorm(n, g, R);
#pragma unroll
    for (int k = 0; k < 8; ++k) s_H[k] = refined ? R[k] : H[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 8; ++k) H[k] = s_H[k];

  // classification under the final model
  int keep = 0;
  for (int i = tid; i < m; i += MOTION_REFINE_THREADS) {
    bool front;
    const float d2 = motion_d2(H, corr[i], front);
    keep += front && !(d2 > e2);
    err[cidx[i]] = front ? __fsqrt_rn(d2) : __int_as_float(0x7f800000);
  }
  keep = motion_warp_sum(keep);
  if (lane == 0) atomicAdd(&s_keep, keep);
  __syncthreads();
  const int kept = s_keep;
  const bool applied = kept >= MOTION_MIN_KEEP;
  if (applied)
    for (int i = tid; i < m; i += MOTION_REFINE_THREADS)
      if (!motion_inlier(H, corr[i], e2)) {
        const int f = cidx[i];
        x[f] = -1.0f; y[f] = -1.0f; val[f] = KLT_B200_MOTION_OUTLIER;
      }
  if (tid == 0) {
    MotionModelRec r;
#pragma unroll
    for (int k = 0; k < 8; ++k) r.H[k] = applied ? H[k] : __int_as_float(0x7fffffff);
    r.H[8] = applied ? 1.0f : __int_as_float(0x7fffffff);
    r.valid = applied; r.tracked = m; r.inliers = kept; r.hypothesis = win;
    *rec = r;
  }
}
