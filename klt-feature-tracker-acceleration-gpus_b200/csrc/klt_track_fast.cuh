// klt_track_fast.cuh -- production (FMA-mode) tracker kernel, included by klt_dev.cu.
//
// Same algorithm as track_kernel (reference src/V1/trackFeatures.c:381-486 per level and
// :1343-1437 across levels) re-mapped for latency: the warp-per-feature kernel is bound by a
// long dependent instruction chain (ncu: 2.6 k warp instructions per feature, 25 % issue
// utilisation, every first touch of a level a DRAM miss).  Here
//   * 8 lanes own one feature, 4 features share a warp: lane r of a group handles window row
//     r - WH/2 (WW pixels, all independent => deep memory-level parallelism);
//   * the bilinear weights are computed once per window position instead of once per pixel
//     (the fractional offsets of x+i and x are equal up to float rounding);
//   * the five window sums are reduced with 3 xor-shuffles over the 8 lanes, every lane ends
//     up with the totals and solves the 2x2 system redundantly (no broadcast);
//   * the footprint of the next finer level is prefetched into L2 while the current level
//     iterates.
// Windows up to 15 x 8*RPL rows are supported through the WW / RPL template parameters; the
// bit-exact mode and larger windows stay on track_kernel.
#pragma once

__device__ __forceinline__ void prefetch_l2(const void* p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

__device__ __forceinline__ float group_sum8(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

// one window row of bilinear samples: out[i] = interp(img, xt+i+ax, yrow+ay), i = 0..WW-1
template <int WW>
__device__ __forceinline__ void sample_row(const float* __restrict__ img, int pitch, int xt, int yrow,
                                           float ax, float ay, float* out) {
  const float* p0 = img + (size_t)yrow * pitch + xt;
  const float* p1 = p0 + pitch;
  float a[WW + 1], b[WW + 1];
#pragma unroll
  for (int i = 0; i <= WW; ++i) { a[i] = __ldg(p0 + i); b[i] = __ldg(p1 + i); }
  const float w00 = (1.0f - ax) * (1.0f - ay), w01 = ax * (1.0f - ay), w10 = (1.0f - ax) * ay, w11 = ax * ay;
#pragma unroll
  for (int i = 0; i < WW; ++i)
    out[i] = fmaf(w11, b[i + 1], fmaf(w10, b[i], fmaf(w01, a[i + 1], w00 * a[i])));
}

// The pyramid descent of the feature of this lane's group from (x, y) in p1's frame into p2's frame:
// the status of the finest level reached and the end position, before the border test.  Called by
// all lanes of the warp; groups with alive == false only take part in the shuffles.
// WW: window width (odd, <= 15); RPL: window rows per lane (window height <= 8 * RPL)
// G: (x, y) and the guess (gx, gy) the descent starts from are given at the coarsest level (pred_start).
template <int WW, int RPL, bool G = false>
__device__ __forceinline__ int track_fast_descent(const PyrView& p1, const PyrView& p2, const TrackArgs& a,
                                                  int r8, bool alive, float x, float y, float& xend, float& yend,
                                                  float gx = 0.0f, float gy = 0.0f) {
  const int wh = a.wh, hw = WW / 2, hh = wh / 2;
  float xloc = x, yloc = y;
  if (!G)
    for (int r = a.nlevels - 1; r >= 0; --r) { xloc = xloc / a.ss; yloc = yloc / a.ss; }
  float xout = G ? gx : xloc, yout = G ? gy : yloc;
  int status = KLT_TRACKED;
  bool running = alive;                                      // false once a level returned SMALL_DET / OOB

  // rows of the window this lane owns: j = r8 + 8*k - hh  (valid if r8 + 8*k < wh)
  for (int r = a.nlevels - 1; r >= 0; --r) {
    if (running) { xloc *= a.ss; yloc *= a.ss; xout *= a.ss; yout *= a.ss; }
    const int nc = p1.ncols[r], nr = p1.nrows[r], pitch = p1.pitch[r];
    const float* __restrict__ i1 = p1.img[r];
    const float* __restrict__ gx1 = p1.gx[r];
    const float* __restrict__ gy1 = p1.gy[r];
    const float* __restrict__ i2 = p2.img[r];
    const float* __restrict__ gx2 = p2.gx[r];
    const float* __restrict__ gy2 = p2.gy[r];

    // prefetch the footprint of the next finer level around the predicted positions
    if (running && r > 0) {
      const int pn = p1.pitch[r - 1], ncn = p1.ncols[r - 1], nrn = p1.nrows[r - 1];
      const int px1 = (int)(xloc * a.ss) - hw, py1 = (int)(yloc * a.ss) - hh + r8;
      const int px2 = (int)(xout * a.ss) - hw, py2 = (int)(yout * a.ss) - hh + r8;
      if (px1 >= 0 && py1 >= 0 && px1 + WW < ncn && py1 < nrn) {
        const size_t o = (size_t)py1 * pn + px1;
        prefetch_l2(p1.img[r - 1] + o); prefetch_l2(p1.img[r - 1] + o + WW);
        prefetch_l2(p1.gx[r - 1] + o);  prefetch_l2(p1.gx[r - 1] + o + WW);
        prefetch_l2(p1.gy[r - 1] + o);  prefetch_l2(p1.gy[r - 1] + o + WW);
      }
      if (px2 >= 0 && py2 >= 0 && px2 + WW < ncn && py2 < nrn) {
        const size_t o = (size_t)py2 * pn + px2;
        prefetch_l2(p2.img[r - 1] + o); prefetch_l2(p2.img[r - 1] + o + WW);
        prefetch_l2(p2.gx[r - 1] + o);  prefetch_l2(p2.gx[r - 1] + o + WW);
        prefetch_l2(p2.gy[r - 1] + o);  prefetch_l2(p2.gy[r - 1] + o + WW);
      }
    }

    // ---- _trackFeature at this level ----------------------------------------------------
    const float x1 = xloc, y1 = yloc;
    float x2 = xout, y2 = yout;
    int iteration = 0;
    float dx = 0.0f, dy = 0.0f;
    float t_i[RPL][WW], t_gx[RPL][WW], t_gy[RPL][WW];
    bool iterating = running;                                // this group still inside the do-while
    int lvl_status = KLT_TRACKED;

    if (iterating && window_oob(x1, y1, hw, hh, nc, nr)) { lvl_status = KLT_OOB; iterating = false; }
    if (iterating && window_oob(x2, y2, hw, hh, nc, nr)) { lvl_status = KLT_OOB; iterating = false; }
    if (iterating) {
      const int xt = (int)x1, yt = (int)y1;
      const float ax = x1 - (float)xt, ay = y1 - (float)yt;
#pragma unroll
      for (int k = 0; k < RPL; ++k) {
        const int row = r8 + 8 * k;
        if (row < wh) {
          sample_row<WW>(i1, pitch, xt - hw, yt - hh + row, ax, ay, t_i[k]);
          sample_row<WW>(gx1, pitch, xt - hw, yt - hh + row, ax, ay, t_gx[k]);
          sample_row<WW>(gy1, pitch, xt - hw, yt - hh + row, ax, ay, t_gy[k]);
        }
      }
    }

    while (__any_sync(0xffffffffu, iterating)) {
      float gxx = 0.0f, gxy = 0.0f, gyy = 0.0f, ex = 0.0f, ey = 0.0f;
      if (iterating) {
        const int xt = (int)x2, yt = (int)y2;
        const float ax = x2 - (float)xt, ay = y2 - (float)yt;
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
          const int row = r8 + 8 * k;
          if (row < wh) {
            float s_i[WW], s_gx[WW], s_gy[WW];
            sample_row<WW>(i2, pitch, xt - hw, yt - hh + row, ax, ay, s_i);
            sample_row<WW>(gx2, pitch, xt - hw, yt - hh + row, ax, ay, s_gx);
            sample_row<WW>(gy2, pitch, xt - hw, yt - hh + row, ax, ay, s_gy);
#pragma unroll
            for (int i = 0; i < WW; ++i) {
              const float df = t_i[k][i] - s_i[i];
              const float sx = t_gx[k][i] + s_gx[i];
              const float sy = t_gy[k][i] + s_gy[i];
              gxx = fmaf(sx, sx, gxx); gxy = fmaf(sx, sy, gxy); gyy = fmaf(sy, sy, gyy);
              ex = fmaf(df, sx, ex); ey = fmaf(df, sy, ey);
            }
          }
        }
      }
      gxx = group_sum8(gxx); gxy = group_sum8(gxy); gyy = group_sum8(gyy);
      ex = group_sum8(ex); ey = group_sum8(ey);
      if (iterating) {
        ex *= a.step_factor; ey *= a.step_factor;
        const float det = gxx * gyy - gxy * gxy;
        if (det < a.min_determinant) {
          lvl_status = KLT_SMALL_DET; iterating = false;
        } else {
          dx = (gyy * ex - gxy * ey) / det;
          dy = (gxx * ey - gxy * ex) / det;
          x2 += dx; y2 += dy;
          ++iteration;
          const bool again = (fabsf(dx) >= a.min_displacement || fabsf(dy) >= a.min_displacement) &&
                             iteration < a.max_iterations;
          if (!again) iterating = false;
          else if (window_oob(x2, y2, hw, hh, nc, nr)) { lvl_status = KLT_OOB; iterating = false; }
        }
      }
    }

    // after the loop (:459-474): bounds of the final position, then the residue
    bool need_res = false;
    if (running) {
      if (window_oob(x2, y2, hw, hh, nc, nr)) lvl_status = KLT_OOB;
      need_res = (lvl_status == KLT_TRACKED);
    }
    if (__any_sync(0xffffffffu, need_res)) {
      float sum = 0.0f;
      if (need_res) {
        const int xt = (int)x2, yt = (int)y2;
        const float ax = x2 - (float)xt, ay = y2 - (float)yt;
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
          const int row = r8 + 8 * k;
          if (row < wh) {
            float s_i[WW];
            sample_row<WW>(i2, pitch, xt - hw, yt - hh + row, ax, ay, s_i);
#pragma unroll
            for (int i = 0; i < WW; ++i) sum += fabsf(t_i[k][i] - s_i[i]);
          }
        }
      }
      sum = group_sum8(sum);
      if (need_res && sum / (float)(WW * wh) > a.max_residue) lvl_status = KLT_LARGE_RESIDUE;
    }
    if (running) {
      int v;                                               // return value of _trackFeature (:479-484)
      if (lvl_status == KLT_SMALL_DET) v = KLT_SMALL_DET;
      else if (lvl_status == KLT_OOB) v = KLT_OOB;
      else if (lvl_status == KLT_LARGE_RESIDUE) v = KLT_LARGE_RESIDUE;
      else if (iteration >= a.max_iterations) v = KLT_MAX_ITERATIONS;
      else v = KLT_TRACKED;
      status = v;
      xout = x2; yout = y2;
      if (v == KLT_SMALL_DET || v == KLT_OOB) running = false;       // :1378
    }
    if (!__any_sync(0xffffffffu, running)) break;
  }

  xend = xout; yend = yout;
  return status;
}

// FB: the forward-backward check runs in the same group after the forward leg (klt_dev_fb_results)
// PRED: the descent starts from the feature's guess (PredArgs, klt_dev_prediction_results)
template <int WW, int RPL, bool FB, bool PRED = false>
__global__ void __launch_bounds__(128)
track_fast_kernel(PyrView p1, PyrView p2, TrackArgs a, int n, FeatIO io,
                  unsigned long long* __restrict__ live_total, FbArgs fb, PredArgs pr) {
  const int lane = threadIdx.x & 31;
  const int r8 = lane & 7;                                   // lane within the feature group
  const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;   // feature of this group

  bool alive = false;                                        // feature still being tracked
  float x0 = 0.0f, y0 = 0.0f;
  int v0 = -1;
  if (f < n) {
    v0 = io.val[(size_t)f * io.istride];
    alive = v0 >= 0;                                         // only features that are not lost (:1346)
    if (alive) { x0 = io.x[(size_t)f * io.istride]; y0 = io.y[(size_t)f * io.istride]; }
  }
  {
    const unsigned bal = __ballot_sync(0xffffffffu, alive && r8 == 0);
    if (lane == 0 && bal) atomicAdd(live_total, (unsigned long long)__popc(bal));
  }
  if (!__any_sync(0xffffffffu, alive)) {
    if (FB && f < n && r8 == 0) fb.rec[f] = fb_unchecked();
    if (PRED && f < n && r8 == 0) pred_skip(pr, f);
    return;
  }

  float4 s0 = make_float4(x0, y0, 0.0f, 0.0f);              // PRED: start and guess at the coarsest level
  if (PRED) {
    if (r8 == 0) {
      if (alive) s0 = pred_start(pr.gx, pr.gy, pr.vel, pr.rec, pr.vel_n, a.nlevels, a.ss, f, v0, x0, y0);
      else if (f < n) pred_skip(pr, f);
    }
    s0 = shfl4(s0, 8);
  }
  float xout, yout;
  int v = track_fast_descent<WW, RPL, PRED>(p1, p2, a, r8, alive, s0.x, s0.y, xout, yout, s0.z, s0.w);
  if (alive) v = track_outcome(a, v, xout, yout);
  if (FB) {
    FbRec r = fb_unchecked();
    const bool back = alive && v == KLT_TRACKED;             // the backward leg: frame 2 into frame 1
    if (__any_sync(0xffffffffu, back)) {
      float xb, yb;
      float4 sb = make_float4(xout, yout, 0.0f, 0.0f);        // PRED: from the mirrored prior
      if (PRED) {
        if (back && r8 == 0) sb = pred_back_start(pr.rec, a.nlevels, a.ss, f, x0, y0, xout, yout);
        sb = shfl4(sb, 8);
      }
      int vb = track_fast_descent<WW, RPL, PRED>(p2, p1, a, r8, back, sb.x, sb.y, xb, yb, sb.z, sb.w);
      if (back) {
        vb = track_outcome(a, vb, xb, yb);
        if (!fb_keep(fb.max_error, x0, y0, xb, yb, vb, r)) v = KLT_B200_FB_INCONSISTENT;
      }
    }
    if (f < n && r8 == 0) fb.rec[f] = r;
  }
  if (PRED && alive && r8 == 0) pred_velocity(pr, io, f, v, xout, yout);
  if (alive && r8 == 0) record_feature(io, f, v, xout, yout);   // record (:1383-1437)
}

// ---------------------------------------------------------------------------------------------
// 7x7 window, one WARP per feature (track7w_kernel): the latency-optimised tracker.
//
// track7_kernel (8 lanes per feature) issues ~350 dependent-ish instructions per Newton iteration
// from each warp at 1.7 warps per scheduler: measured, a pass over half of the features takes as
// long as a pass over all of them (27 us) -- the kernel is a latency chain, not a throughput
// problem, and the GPU is idle otherwise.  Here the 8x8 pixel footprint is spread over all 32
// lanes (lane = 4 * row + column pair): each lane holds the three pixels it needs per image,
// interpolates two window columns (10 instructions per image instead of ~53), the five sums are
// reduced with 5 xor-shuffles, every lane solves the 2x2 system.  ~135 instructions per iteration
// and 4x as many warps in flight.  Same per-sample arithmetic as track7_kernel; the sums are
// added in a different (tree) order.
// ---------------------------------------------------------------------------------------------
struct Pix3 { float a, b, c; };
__device__ __forceinline__ Pix3 pix3_load(const float* __restrict__ img, int off) {
  const float* p = img + off;
  Pix3 r;
  r.a = __ldg(p); r.b = __ldg(p + 1); r.c = __ldg(p + 2);
  return r;
}
// L2 eviction policies for the gathers.  The footprints read from the NEW frame's pyramids are
// (up to the integer cell the feature ends in) the footprints the next frame's call reads from its
// PREVIOUS pyramids; marked evict_last they survive the ~140 MB the next pyramid build streams
// through the 126 MB L2, so half of the next call's gathers hit L2 instead of DRAM.  The previous
// frame's footprints are dead after this call: evict_first.
__device__ __forceinline__ unsigned long long l2_policy(int kind) {   // 0 normal, 1 evict_last, 2 evict_first
  unsigned long long p;
  if (kind == 1) asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2) asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float ldg_policy(const float* p, unsigned long long pol) {
  float v;
  asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
// two loads per lane; the third pixel (column 2c + 2) is the first pixel of the lane to the right.
// Lane c = 3 receives the next row's first pixel instead, which it never uses (its second window
// column does not exist).  A third of the load instructions (and of their L1 wavefronts: every load
// instruction of the warp touches 8 rows = 8+ cache lines) for one shuffle.  Warp-uniform callers only.
__device__ __forceinline__ Pix3 pix3_load(const float* __restrict__ img, int off, unsigned long long pol) {
  const float* p = img + off;
  Pix3 r;
  if ((off & 1) == 0) {        // footprint starts at an even column (warp uniform: row pitches are even): one 64-bit load
    asm("ld.global.nc.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;" : "=f"(r.a), "=f"(r.b) : "l"(p), "l"(pol));
  } else {
    r.a = ldg_policy(p, pol); r.b = ldg_policy(p + 1, pol);
  }
  r.c = __shfl_down_sync(0xffffffffu, r.a, 1);
  return r;
}
// bilinear samples of this lane's two window columns in its window row; the row below comes from
// lane + 4 (lanes 28..31 hold footprint row 7 and only feed the shuffle)
__device__ __forceinline__ void pix3_interp(const Pix3& p, float ax, float ay, float& o0, float& o1) {
  const float h0 = fmaf(ax, p.b - p.a, p.a), h1 = fmaf(ax, p.c - p.b, p.b);
  const float b0 = __shfl_down_sync(0xffffffffu, h0, 4), b1 = __shfl_down_sync(0xffffffffu, h1, 4);
  o0 = fmaf(ay, b0 - h0, h0);
  o1 = fmaf(ay, b1 - h1, h1);
}
__device__ __forceinline__ float warp_sum32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// totals of four per-lane values in every lane with a splitting butterfly: the xor-16 exchange
// halves the values a lane carries from four to two, the xor-8 exchange to one, three plain steps
// finish it and four broadcasts hand every total to every lane: 10 shuffles, 6 adds, 6 selects
// instead of 20 shuffles and 20 adds.
__device__ __forceinline__ void warp_sum4x(float& g0, float& g1, float& g2, float& g3, int lane) {
  const bool hi16 = (lane & 16) != 0, hi8 = (lane & 8) != 0;
  const float r0 = __shfl_xor_sync(0xffffffffu, hi16 ? g0 : g2, 16);
  const float r1 = __shfl_xor_sync(0xffffffffu, hi16 ? g1 : g3, 16);
  const float k0 = (hi16 ? g2 : g0) + r0, k1 = (hi16 ? g3 : g1) + r1;    // lower half: g0, g1; upper half: g2, g3
  float k = (hi8 ? k1 : k0) + __shfl_xor_sync(0xffffffffu, hi8 ? k0 : k1, 8);
  k += __shfl_xor_sync(0xffffffffu, k, 4);
  k += __shfl_xor_sync(0xffffffffu, k, 2);
  k += __shfl_xor_sync(0xffffffffu, k, 1);           // lanes 0-7: g0, 8-15: g1, 16-23: g2, 24-31: g3
  g0 = __shfl_sync(0xffffffffu, k, 0); g1 = __shfl_sync(0xffffffffu, k, 8);
  g2 = __shfl_sync(0xffffffffu, k, 16); g3 = __shfl_sync(0xffffffffu, k, 24);
}

// The pyramid descent of the warp's feature from (x, y) in p1's frame (gathers with L2 policy pol1)
// into p2's frame (pol2): the status of the finest level reached and the end position, before the
// border test.
// G: (x, y) and the guess (gx, gy) the descent starts from are given at the coarsest level (pred_start).
template <bool G = false>
__device__ __forceinline__ int track7w_descent(const PyrView& p1, const PyrView& p2, const TrackArgs& a, int lane,
                                               unsigned long long pol1, unsigned long long pol2,
                                               float x, float y, float& xend, float& yend,
                                               float gx = 0.0f, float gy = 0.0f) {
  constexpr int hw = 3, hh = 3;
  const int r = lane >> 2, c = lane & 3;                     // footprint row, column pair
  const bool v0 = r < 7, v1 = r < 7 && c < 3;                // window samples (2c, r) and (2c + 1, r)
  float xloc = x, yloc = y;
  if (!G)
    for (int l = a.nlevels - 1; l >= 0; --l) { xloc = xloc / a.ss; yloc = yloc / a.ss; }
  float xout = G ? gx : xloc, yout = G ? gy : yloc;
  int status = KLT_TRACKED;

  for (int l = a.nlevels - 1; l >= 0; --l) {
    xloc *= a.ss; yloc *= a.ss; xout *= a.ss; yout *= a.ss;
    const int nc = p1.ncols[l], nr = p1.nrows[l], pitch = p1.pitch[l];
    const float* __restrict__ i2 = p2.img[l];
    const float* __restrict__ gx2 = p2.gx[l];
    const float* __restrict__ gy2 = p2.gy[l];
    const float x1 = xloc, y1 = yloc;
    float x2 = xout, y2 = yout;
    int iteration = 0, lvl_status = KLT_TRACKED;
    bool iterating = true;
    if (window_oob(x1, y1, hw, hh, nc, nr) || window_oob(x2, y2, hw, hh, nc, nr)) { lvl_status = KLT_OOB; iterating = false; }

    float t_i0 = 0.f, t_i1 = 0.f, t_gx0 = 0.f, t_gx1 = 0.f, t_gy0 = 0.f, t_gy1 = 0.f;
    Pix3 c_i, c_gx, c_gy;
    c_i.a = c_i.b = c_i.c = 0.f; c_gx = c_i; c_gy = c_i;
    int c_xt = -1000000, c_yt = -1000000;
    if (iterating) {
      // all 18 loads of the level are issued before the first use
      const int xt1 = (int)x1, yt1 = (int)y1, xt2 = (int)x2, yt2 = (int)y2;
      const int o1 = (yt1 - 3 + r) * pitch + (xt1 - 3 + 2 * c), o2 = (yt2 - 3 + r) * pitch + (xt2 - 3 + 2 * c);
      const Pix3 r_i = pix3_load(p1.img[l], o1, pol1), r_gx = pix3_load(p1.gx[l], o1, pol1), r_gy = pix3_load(p1.gy[l], o1, pol1);
      c_i = pix3_load(i2, o2, pol2); c_gx = pix3_load(gx2, o2, pol2); c_gy = pix3_load(gy2, o2, pol2);
      c_xt = xt2; c_yt = yt2;
      const float ax = x1 - (float)xt1, ay = y1 - (float)yt1;
      pix3_interp(r_i, ax, ay, t_i0, t_i1);
      pix3_interp(r_gx, ax, ay, t_gx0, t_gx1);
      pix3_interp(r_gy, ax, ay, t_gy0, t_gy1);
    }

    float dx = 0.0f, dy = 0.0f;
    while (iterating) {                                       // warp uniform
      const int xt = (int)x2, yt = (int)y2;
      if (xt != c_xt || yt != c_yt) {                         // the integer footprint moved: re-read it
        const int o2 = (yt - 3 + r) * pitch + (xt - 3 + 2 * c);
        c_i = pix3_load(i2, o2, pol2); c_gx = pix3_load(gx2, o2, pol2); c_gy = pix3_load(gy2, o2, pol2);
        c_xt = xt; c_yt = yt;
      }
      const float ax = x2 - (float)xt, ay = y2 - (float)yt;
      float s_i0, s_i1, s_gx0, s_gx1, s_gy0, s_gy1;
      pix3_interp(c_i, ax, ay, s_i0, s_i1);
      pix3_interp(c_gx, ax, ay, s_gx0, s_gx1);
      pix3_interp(c_gy, ax, ay, s_gy0, s_gy1);
      float gxx = 0.0f, gxy = 0.0f, gyy = 0.0f, ex = 0.0f, ey = 0.0f;
      {
        const float df = v0 ? t_i0 - s_i0 : 0.0f, sx = v0 ? t_gx0 + s_gx0 : 0.0f, sy = v0 ? t_gy0 + s_gy0 : 0.0f;
        gxx = sx * sx; gxy = sx * sy; gyy = sy * sy; ex = df * sx; ey = df * sy;
      }
      {
        const float df = v1 ? t_i1 - s_i1 : 0.0f, sx = v1 ? t_gx1 + s_gx1 : 0.0f, sy = v1 ? t_gy1 + s_gy1 : 0.0f;
        gxx = fmaf(sx, sx, gxx); gxy = fmaf(sx, sy, gxy); gyy = fmaf(sy, sy, gyy);
        ex = fmaf(df, sx, ex); ey = fmaf(df, sy, ey);
      }
      warp_sum4x(gxx, gxy, gyy, ex, lane);
      ey = warp_sum32(ey);
      ex *= a.step_factor; ey *= a.step_factor;
      const float det = gxx * gyy - gxy * gxy;
      if (det < a.min_determinant) { lvl_status = KLT_SMALL_DET; break; }
      const float inv = __frcp_rn(det);
      dx = (gyy * ex - gxy * ey) * inv;
      dy = (gxx * ey - gxy * ex) * inv;
      x2 += dx; y2 += dy;
      ++iteration;
      const bool again = (fabsf(dx) >= a.min_displacement || fabsf(dy) >= a.min_displacement) &&
                         iteration < a.max_iterations;
      if (!again) break;
      if (window_oob(x2, y2, hw, hh, nc, nr)) { lvl_status = KLT_OOB; break; }
    }

    // after the loop (:459-474): bounds of the final position, then the residue
    if (lvl_status == KLT_TRACKED && window_oob(x2, y2, hw, hh, nc, nr)) lvl_status = KLT_OOB;
    if (lvl_status == KLT_TRACKED) {
      const int xt = (int)x2, yt = (int)y2;
      if (xt != c_xt || yt != c_yt) c_i = pix3_load(i2, (yt - 3 + r) * pitch + (xt - 3 + 2 * c), pol2);
      float s_i0, s_i1;
      pix3_interp(c_i, x2 - (float)xt, y2 - (float)yt, s_i0, s_i1);
      float sum = (v0 ? fabsf(t_i0 - s_i0) : 0.0f) + (v1 ? fabsf(t_i1 - s_i1) : 0.0f);
      sum = warp_sum32(sum);
      if (sum * (1.0f / 49.0f) > a.max_residue) lvl_status = KLT_LARGE_RESIDUE;
    }
    int v;                                                   // return value of _trackFeature (:479-484)
    if (lvl_status == KLT_SMALL_DET) v = KLT_SMALL_DET;
    else if (lvl_status == KLT_OOB) v = KLT_OOB;
    else if (lvl_status == KLT_LARGE_RESIDUE) v = KLT_LARGE_RESIDUE;
    else if (iteration >= a.max_iterations) v = KLT_MAX_ITERATIONS;
    else v = KLT_TRACKED;
    status = v;
    xout = x2; yout = y2;
    if (v == KLT_SMALL_DET || v == KLT_OOB) break;           // :1378
  }

  xend = xout; yend = yout;
  return status;
}

// FB: the forward-backward check runs in the same warp after the forward leg (klt_dev_fb_results).
// Its backward leg reads the new frame with the new frame's policy (evict_last) and the old frame
// with the old frame's (evict_first), as the forward leg does.
// PRED: the descent starts from the feature's guess (PredArgs, klt_dev_prediction_results); lane 0
// reads and writes the velocity record after pdl_wait, like the features.
template <bool FB, bool PRED = false>
__global__ void __launch_bounds__(128)
track7w_kernel(PyrView p1, PyrView p2, TrackArgs a, int n, FeatIO io,
               unsigned long long* __restrict__ live_total, FbArgs fb, PredArgs pr) {
  const int lane = threadIdx.x & 31;
  const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned long long pol1 = l2_policy(a.l2_keep ? 2 : 0), pol2 = l2_policy(a.l2_keep ? 1 : 0);
  pdl_wait();                                                 // pyramids and features come from earlier kernels
  // the whole grid is resident at once (a warp per feature, no shared memory): whatever follows in
  // the stream -- the next frame's level-0 kernel -- may move into the SMs as these warps retire
  pdl_launch_dependents();
  if (f >= n) return;
  const int val_in = io.val[(size_t)f * io.istride];
  if (val_in < 0) {                                           // only features that are not lost (:1346)
    if (FB && lane == 0) fb.rec[f] = fb_unchecked();
    if (PRED && lane == 0) pred_skip(pr, f);
    return;
  }
  if (lane == 0) atomicAdd(live_total, 1ULL);
  const float x0 = io.x[(size_t)f * io.istride], y0 = io.y[(size_t)f * io.istride];
  float4 s0 = make_float4(x0, y0, 0.0f, 0.0f);              // PRED: start and guess at the coarsest level
  if (PRED) {
    if (lane == 0) s0 = pred_start(pr.gx, pr.gy, pr.vel, pr.rec, pr.vel_n, a.nlevels, a.ss, f, val_in, x0, y0);
    s0 = shfl4(s0, 32);
  }
  float xout, yout;
  int v = track_outcome(a, track7w_descent<PRED>(p1, p2, a, lane, pol1, pol2, s0.x, s0.y, xout, yout, s0.z, s0.w),
                        xout, yout);
  if (FB) {
    FbRec r = fb_unchecked();
    if (v == KLT_TRACKED) {                                   // the backward leg: frame 2 into frame 1
      float xb, yb;
      float4 sb = make_float4(xout, yout, 0.0f, 0.0f);        // PRED: from the mirrored prior
      if (PRED) {
        if (lane == 0) sb = pred_back_start(pr.rec, a.nlevels, a.ss, f, x0, y0, xout, yout);
        sb = shfl4(sb, 32);
      }
      const int vb = track_outcome(a, track7w_descent<PRED>(p2, p1, a, lane, pol2, pol1, sb.x, sb.y, xb, yb, sb.z, sb.w),
                                   xb, yb);
      if (!fb_keep(fb.max_error, x0, y0, xb, yb, vb, r)) v = KLT_B200_FB_INCONSISTENT;
    }
    if (lane == 0) fb.rec[f] = r;
  }
  if (PRED && lane == 0) pred_velocity(pr, io, f, v, xout, yout);
  if (lane == 0) record_feature(io, f, v, xout, yout);     // record (:1383-1437)
}

