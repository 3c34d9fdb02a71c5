// klt_fused.cuh -- TMA-staged, fused frame kernels (included by klt_dev.cu).
//
// l0_fused_kernel   : u8 frame          -> L0, gx0, gy0      (1 B read + 12 B written per pixel)
//                     (+ L1 with the NX geometry: the pyramid step from the L0 tile already on chip)
// level_chain_kernel: L_l (float)       -> gx_l, gy_l (+ L_{l+1})
// level_fused_kernel: L_{l-1} (float)   -> L_l, gx_l, gy_l   (one pyramid step + its gradients;
//                     subsampling 4, other radii and the non-chained level-0 variants)
//
// Replaces, per level, _KLTToFloatImage + _KLTComputeSmoothedImage (+ the smooth/subsample
// step of _KLTComputePyramid) + _KLTComputeGradients (reference src/V1/convolve.c:37-53,
// 273-314, src/V1/pyramid.c:112-124 as sequenced by trackFeatures.c:1311-1321) without any
// float input image, horizontal-pass temporary or smoothed-before-subsample image touching HBM.
//
// Both kernels are persistent (grid = resident CTAs, tiles claimed from an atomic counter): the
// TMA load of the next tile's source box is issued as soon as the current one has been
// consumed, so its latency hides behind the remaining stages.  All stages of a tile run in
// shared memory:
//   L0   : TMA u8 box -> A: horizontal Gaussian -> B: vertical Gaussian (+ L0 stores)
//   level: TMA f32 box -> P1: horizontal Gaussian at the kept columns -> P2: vertical Gaussian
//          at the kept rows (+ L_l stores)
//   both : C: horizontal DoG and Gaussian of the level tile -> D: vertical Gaussian / DoG,
//          float4 stores of gx, gy
// Every buffer has its column origin at x0-4 (16 B aligned) and a row pitch that is an odd
// number of 16 B chunks, so that the quarter-warp lane mappings used below make every 128-bit
// shared access conflict free.  128-bit shared loads are issued through inline PTX: left to
// the compiler, windows with unused edge elements get narrowed into conflicting 32/64-bit loads.
//
// Zero bands of the separable passes (convolve.c:164-178, :216-237) are applied only by tiles
// that touch the image border (BORDER flag, CTA uniform).  The derivative kernel's centre tap
// is exactly 0 (convolve.c:79: -i * gauss with i = 0) and is skipped; the host checks that.
#pragma once

#include <cuda.h>          // CUtensorMap (types only; the encoder is fetched at run time)

// ---- TMA / mbarrier primitives (sm_90+ PTX) ------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned phase) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "KLT_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra KLT_DONE;\n\t"
      "bra KLT_WAIT;\n\t"
      "KLT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(phase)
      : "memory");
}
// The innermost start coordinate must be a multiple of 16 bytes (measured on B200: a u8
// box starting at x0-8 raises "illegal instruction"; x0-16 and negative / out-of-range
// coordinates are fine and zero-filled).
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int cx, int cy,
                                            unsigned long long* bar) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<unsigned long long>(map)), "r"(cx), "r"(cy), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds128(const float* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(smem_u32(p)));
  return v;
}

// u8 -> f32 without the conversion pipe: 0x4B0000bb is the float 2^23 + bb.
#ifndef KLT_U8_I2F
#define KLT_U8_I2F 0
#endif
__device__ __forceinline__ float u8_to_float(unsigned word, unsigned byte_sel) {
#if KLT_U8_I2F
  return (float)((word >> (8 * byte_sel)) & 0xffu);       // one I2F.U8 with a byte selector (conversion pipe)
#else
  return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7440u + byte_sel)) - 8388608.0f;
#endif
}

// packed FP32 FMA (Blackwell FFMA2): (ax, ay) += (vx, vy) * (kk.x, kk.y), each half an ordinary
// IEEE fma -- bit-identical to two fmaf, half the issue slots.  The packs are register renames.
__device__ __forceinline__ void ffma2(float& ax, float& ay, float vx, float vy, float2 kk) {
  unsigned long long a, v, k;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(ax), "f"(ay));
  asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(vx), "f"(vy));
  asm("mov.b64 %0, {%1, %2};" : "=l"(k) : "f"(kk.x), "f"(kk.y));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(v), "l"(k));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(ax), "=f"(ay) : "l"(a));
}
// a += v * t.k[m] on four columns: the vertical passes (scatter form)
__device__ __forceinline__ void fma4(float4& a, const float4& v, const TapsF& t, int m, bool exact) {
  if (exact) {
    const float k = t.k[m];
    a.x = __fadd_rn(a.x, __fmul_rn(v.x, k)); a.y = __fadd_rn(a.y, __fmul_rn(v.y, k));
    a.z = __fadd_rn(a.z, __fmul_rn(v.z, k)); a.w = __fadd_rn(a.w, __fmul_rn(v.w, k));
  } else {
    ffma2(a.x, a.y, v.x, v.y, t.kk[m]);
    ffma2(a.z, a.w, v.z, v.w, t.kk[m]);
  }
}

// L2 residency hints for the pyramid stores.  The smoothed image L_l is what the next kernel of the
// chain reads back in full (level l+1 is made from it), the gradients are only gathered later, at a
// few thousand footprints, by the tracker.  A 4K level 0 is 100 MB of stores through a 126 MB L2 that
// still holds the previous frame: left alone, most of L_0 is gone again before level_fused_kernel
// asks for it (ncu, no cache flush: 33 MB of DRAM reads for level 1 = all of L_0).  c_l2_hints (env
// KLT_B200_L2_HINTS) bit 0: L_l is stored evict_last; bit 1: gx_l / gy_l are stored evict_first.
// Measured on the 4K step (us): 0: 72.93, 1: 74.54 (the tracker's gradient gathers miss: 20.8 -> 22.9),
// 2: 72.33 (level 1: 24.7 -> 22.9), 3: 73.96.  Default 2.
__constant__ int c_l2_hints = 2;
__device__ __forceinline__ unsigned long long store_policy(bool keep) {
  unsigned long long p_keep, p_drop, p_norm;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p_keep));
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p_drop));
  asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p_norm));
  return keep ? ((c_l2_hints & 1) ? p_keep : p_norm) : ((c_l2_hints & 2) ? p_drop : p_norm);
}
__device__ __forceinline__ void stg128(float* p, const float4& v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w), "l"(pol)
               : "memory");
}

static constexpr int FUSED_RG = 3;       // gradient radius the fused kernels are built for

// Programmatic dependent launch: a CTA of the per-frame chain that finds its tile queue empty lets
// the successor kernel start launching (its CTAs become resident as ours retire and run their
// prologue), and every kernel waits for its predecessor's memory before it touches any of it.
// Hides the launch latency and the drain / fill bubble at each kernel boundary of a frame: 94.3 ->
// 82.2 us per 4K step on B200.  The trigger point matters (measured): at kernel start the step
// takes 132 us, at the claim of the last tile 94.7 us (no gain), at queue-empty 82.2 us.  Both
// instructions are no-ops when the launch did not ask for programmatic serialisation.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- the persistent tile queue of the fused kernels -----------------------------------------------
// Tiles are handed out dynamically: a launch covers the tiles [tile0, ntiles) (whole tile rows when
// a frame is built band by band behind its upload); tile0 + counter[0] - base is the next tile
// index.  Every CTA performs (tiles it processed + 1) atomicAdds, so after the launch the counter
// stands at base + (ntiles - tile0) + gridDim.x, which the host uses as the next launch's base (no
// reset needed).
// (The kernels take it __grid_constant__, so that each field is read from the parameter bank where it
// is used, like a scalar parameter.)
struct TileQueue {
  int tiles_x;                       // tile (x, y) is tile index y * tiles_x + x
  int tile0, ntiles;
  unsigned* counter;
  unsigned base;
};
// One CTA's loop over the queue, tile origin (x0, y0) = (tile % tiles_x, tile / tiles_x) * (TX, TY),
// b = border(x0, y0) (the tile meets a zero band or an image edge):
//   front(x0, y0, b): the stages that consume the source box; barrier; claim of the next tile and the
//                     TMA load of its box (box(x0, y0): the box's start coordinates) into box_dst;
//   back(x0, y0, b):  the remaining stages; barrier.
// The claim is made one tile ahead, so the next box's load latency hides behind the back stages.
// sched: 16 B of shared memory (the mbarrier, then the next tile index).  WAIT_FIRST: griddepcontrol.wait
// before the first claim (the kernel reads what its predecessor wrote); else in front of the first back
// stage, i.e. after the first load and front stages.  Dependents are released when the queue is empty.
template <int TX, int TY, bool WAIT_FIRST, class Border, class Box, class Front, class Back>
__device__ __forceinline__ void tile_queue(const TileQueue& q, const CUtensorMap* map, void* box_dst,
                                           unsigned box_bytes, unsigned char* sched, Border border, Box box,
                                           Front front, Back back) {
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(sched);
  volatile int* s_next = reinterpret_cast<volatile int*>(sched + 8);
  const int tid = threadIdx.x, tiles_x = q.tiles_x;
  auto claim = [&]() {
    if (tid == 0) {
      const int t = q.tile0 + (int)(atomicAdd(q.counter, 1u) - q.base);
      *s_next = t;
      if (t < q.ntiles) {
        mbar_expect_tx(bar, box_bytes);
        const int2 c = box((t % tiles_x) * TX, (t / tiles_x) * TY);
        tma_load_2d(box_dst, map, c.x, c.y, bar);
      }
    }
  };
  if (tid == 0) {
    mbar_init(bar, 1);
    // descriptor fetch overlaps the predecessor's tail (we may be resident before it has finished)
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<unsigned long long>(map)) : "memory");
  }
  if (WAIT_FIRST) pdl_wait();
  claim();
  __syncthreads();
  int tile = *s_next;
  unsigned phase = 0;
  bool waited = WAIT_FIRST;
  while (tile < q.ntiles) {
    const int x0 = (tile % tiles_x) * TX, y0 = (tile / tiles_x) * TY;
    const bool b = border(x0, y0);
    mbar_wait(bar, phase);
    phase ^= 1;
    front(x0, y0, b);
    __syncthreads();                 // source box consumed; everybody has read s_next
    claim();
    if (!waited) { pdl_wait(); waited = true; }
    back(x0, y0, b);
    __syncthreads();                 // the back stages' buffers are free for the next tile
    tile = *s_next;
  }
  if (!waited) pdl_wait();            // (a CTA that got no tile)
  pdl_launch_dependents();            // queue empty: the next kernel of the chain may move in
}

// barrier among the NTH threads of a tile (== __syncthreads())
template <int NTH = 256>
__device__ __forceinline__ void tile_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NTH) : "memory"); }

// ---- stage C: horizontal DoG and Gaussian of a level tile ---------------------------------
// sL [LH][LP]: tile col c <-> global x0-4+c.   sHd, sHg [LH][HP]: col c <-> global x0+c.
// 8 outputs per thread from a 16-float window (4 x LDS.128); a warp covers 8 groups x 4 rows
// (TX = 64) or 4 groups x 8 rows (TX = 32); a quarter warp is 4 groups x 2 rows, conflict free
// because LP/4 and HP/4 are odd.
template <bool EXACT, bool BORDER, int TX, int LH, int LP, int HP, int NTH = 256>
__device__ __forceinline__ void stage_hgrad(const float* sL, float* sHd, float* sHg, const TapsF& tg,
                                            const TapsF& td, int x0, int W) {
  constexpr int RG = FUSED_RG;
  constexpr int NGC = TX / 8;                       // groups per row: 8 or 4
  constexpr int RPW = 32 / NGC;                     // rows per warp: 4 or 8
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & 3, rpar = (lane >> 2) & 1, rem = lane >> 3;
  const int g = NGC == 8 ? 4 * (rem & 1) + sub : sub;
  const int rl = NGC == 8 ? 2 * (rem >> 1) + rpar : 2 * rem + rpar;
  for (int rb = warp * RPW; rb < LH; rb += (NTH / 32) * RPW) {
    const int r = rb + rl;
    if (r < LH) {
      float win[16];
      const float* p = sL + r * LP + 8 * g;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const float4 t = lds128(p + 4 * v);
        win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
      }
      float od[8], og[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float a = 0.0f, b = 0.0f;
#pragma unroll
        for (int m = 0; m < 2 * RG + 1; ++m)
          if (m != RG) a = mac<EXACT>(a, win[q + 1 + m], td.k[m]);        // centre tap is 0
#pragma unroll
        for (int m = 0; m < 2 * RG + 1; ++m) b = mac<EXACT>(b, win[q + 1 + m], tg.k[m]);
        if (BORDER) {
          const int xg = x0 + 8 * g + q;
          if (xg < RG || xg >= W - RG) { a = 0.0f; b = 0.0f; }
        }
        od[q] = a; og[q] = b;
      }
      float4* dd = reinterpret_cast<float4*>(sHd + r * HP + 8 * g);
      float4* dg = reinterpret_cast<float4*>(sHg + r * HP + 8 * g);
      dd[0] = make_float4(od[0], od[1], od[2], od[3]);
      dd[1] = make_float4(od[4], od[5], od[6], od[7]);
      dg[0] = make_float4(og[0], og[1], og[2], og[3]);
      dg[1] = make_float4(og[4], og[5], og[6], og[7]);
    }
  }
}

// ---- the next pyramid level (subsampling 2, radius 5) from a level tile on chip ----------------
// L_{l+1}(X, Y) = S(2X+1, 2Y+1), S the separable Gaussian of L_l; a tile with origin (x0, y0) (both
// even) makes the block X = x0/2 .. x0/2+TX/2-1, Y = y0/2 .. y0/2+TY/2-1, from L_l rows y0-4 ..
// y0+TY+4 and columns x0-4 .. x0+TX+4.  Same operation sequence as lv_p1_item / P2 of
// level_fused_kernel: taps in increasing order, horizontal before vertical, zero bands on the
// source coordinate.
static constexpr int NEXT_R = 5;
// horizontal pass at the kept columns, every source row.  sL [NR][SP]: col c <-> x0-4+c, row r <->
// y0-4+r.  sN [NR][NP]: col c <-> x0/2+c.  Lane mapping of stage_hgrad (a quarter warp is 4 groups x
// 2 rows, conflict free on the loads because SP/4 is odd); the row units go to the warps in reverse
// order, because the last warps are the ones stage_hgrad leaves idle in its last pass.
template <bool EXACT, bool BORDER, int TX, int NR, int SP, int NP, int NTH = 256>
__device__ __forceinline__ void stage_hnext(const float* sL, float* sN, const TapsF& tp, int x0, int Wsrc) {
  constexpr int R = NEXT_R;
  constexpr int NG = TX / 8;                        // groups of 4 kept columns: 8 or 4
  constexpr int RPW = 32 / NG, NW = NTH / 32, NU = (NR + RPW - 1) / RPW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & 3, rpar = (lane >> 2) & 1, rem = lane >> 3;
  const int g = NG == 8 ? 4 * (rem & 1) + sub : sub;
  const int rl = NG == 8 ? 2 * (rem >> 1) + rpar : 2 * rem + rpar;
  for (int u = NW - 1 - warp; u < NU; u += NW) {
    const int r = u * RPW + rl;
    if (r < NR) {
      float win[20];
      const float* p = sL + r * SP + 8 * g;
#pragma unroll
      for (int v = 0; v < 5; ++v) {
        const float4 t = lds128(p + 4 * v);
        win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
      }
      float o[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float acc = 0.0f;
#pragma unroll
        for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[2 * q + m], tp.k[m]);
        if (BORDER) {
          const int xs = x0 + 8 * g + 2 * q + 1;
          if (xs < R || xs >= Wsrc - R) acc = 0.0f;
        }
        o[q] = acc;
      }
      *reinterpret_cast<float4*>(sN + r * NP + 4 * g) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}
// vertical pass at the kept rows, stored to L_{l+1}: items of 4 columns x 1 row, handed out from the
// last thread down (the gy half of stage_vgrad_both, whose derivative pass skips its centre tap, or
// its idle threads, comes first).
template <bool EXACT, bool BORDER, int TX, int TY, int NP, int NTH = 256>
__device__ __forceinline__ void stage_vnext(const float* sN, const TapsF& tp, float* __restrict__ out, int npitch,
                                            int x0, int y0, int Hsrc, int Wn, int Hn) {
  constexpr int R = NEXT_R;
  constexpr int NG = TX / 8, ITEMS = NG * (TY / 2);
  const unsigned long long pol = store_policy(true);        // read back by the next kernel of the chain
  for (int i = NTH - 1 - (int)threadIdx.x; i < ITEMS; i += NTH) {
    const int yl = i / NG, g = i - yl * NG;
    const float* src = sN + (2 * yl) * NP + 4 * g;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int m = 0; m < 2 * R + 1; ++m) fma4(acc, lds128(src + m * NP), tp, m, EXACT);
    const int X = x0 / 2 + 4 * g, Y = y0 / 2 + yl;
    if (BORDER) {
      const int ys = 2 * Y + 1;
      if (ys < R || ys >= Hsrc - R) acc = make_float4(0.f, 0.f, 0.f, 0.f);
      if (X < Wn && Y < Hn) stg128(out + (size_t)Y * npitch + X, acc, pol);
    } else {
      stg128(out + (size_t)Y * npitch + X, acc, pol);
    }
  }
}

// ---- stage D: vertical 7-tap pass, 4 columns x PY rows per thread, straight to HBM ------------
// scatter form: every loaded row feeds the outputs it belongs to, taps in increasing order
// (== the reference's summation order for each output).
template <bool EXACT, bool BORDER, int PY, int HP, bool SKIP_CENTRE>
__device__ __forceinline__ void stage_vgrad(const float* __restrict__ src, const TapsF& tk,
                                            float* __restrict__ out, int opitch, int xg, int yg0,
                                            int W, int H) {
  constexpr int R = FUSED_RG;
  const unsigned long long pol = store_policy(false);
  float4 acc[PY];
#pragma unroll
  for (int q = 0; q < PY; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int i = 0; i < PY + 2 * R; ++i) {
    const float4 v = lds128(src + i * HP);
#pragma unroll
    for (int q = 0; q < PY; ++q) {
      const int m = i - q;
      if (m >= 0 && m <= 2 * R && !(SKIP_CENTRE && m == R)) fma4(acc[q], v, tk, m, EXACT);
    }
  }
#pragma unroll
  for (int q = 0; q < PY; ++q) {
    const int yg = yg0 + q;
    if (BORDER) {
      if (yg < R || yg >= H - R) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (xg < W && yg < H) stg128(out + (size_t)yg * opitch + xg, acc[q], pol);
    } else {
      stg128(out + (size_t)yg * opitch + xg, acc[q], pol);
    }
  }
}

// gx = V_gauss(Hd), gy = V_deriv(Hg); first half of the CTA does gx, second half gy (warp uniform)
template <bool EXACT, bool BORDER, int TX, int TY, int PY, int HP, int NTH = 256>
__device__ __forceinline__ void stage_vgrad_both(const float* sHd, const float* sHg, const TapsF& tg,
                                                 const TapsF& td, float* out_gx, float* out_gy,
                                                 int opitch, int x0, int y0, int W, int H) {
  constexpr int NCG = TX / 4, NRB = TY / PY, ITEMS = NCG * NRB;       // per output image
  constexpr int HALF = NTH / 2;
  static_assert(ITEMS <= HALF, "stage D mapping");
  const int tid = threadIdx.x;
  const int t = tid & (HALF - 1);
  if (t < ITEMS) {
    const int blk = t / NCG, j = t - blk * NCG;
    if (tid < HALF)
      stage_vgrad<EXACT, BORDER, PY, HP, false>(sHd + (blk * PY) * HP + 4 * j, tg, out_gx, opitch,
                                                x0 + 4 * j, y0 + blk * PY, W, H);
    else
      stage_vgrad<EXACT, BORDER, PY, HP, true>(sHg + (blk * PY) * HP + 4 * j, td, out_gy, opitch,
                                               x0 + 4 * j, y0 + blk * PY, W, H);
  }
}

// ============================================================================================
// level 0
// ============================================================================================
// TY_: tile height; PYB_ / PYD_: output rows per thread of the two vertical stages; CPS_: resident
// CTAs per SM the kernel is compiled for (register budget).  NX_: the tile also makes its block of
// L1 (subsampling 2, radius 5): L0 is computed XR rows above, XH - XR rows below and one column
// right of what the gradients need, and the horizontal L1 pass gets a buffer of its own.
template <int TY_, int PYB_, int PYD_, int CPS_, bool NX_ = false>
struct L0GeoT {
  static constexpr int TX = 64, TY = TY_, PYB = PYB_, PYD = PYD_, CPS = CPS_;
  static constexpr bool NX = NX_;
  static constexpr int RS = 2, RG = FUSED_RG;                          // smoothing / gradient radii
  static constexpr int XR = NX ? NEXT_R - 1 - RG : 0, XH = NX ? 2 * (NEXT_R - 1 - RG) + 1 : 0;
  static constexpr int U8_W = 96, U8_H = TY + 2 * (RS + RG) + XH;      // col c <-> x0-16+c
  static constexpr int HS_P = 76, HS_H = U8_H;                         // col c <-> x0-4+c, row r <-> y0-5-XR+r
  static constexpr int L0_P = 76, L0_H = TY + 2 * RG + XH;             // row r <-> y0-3-XR+r
  static constexpr int HG_P = 68, HG_H = TY + 2 * RG;                  // col c <-> x0+c, row r <-> y0-3+r
  static constexpr int NGB = NX ? 19 : 18;                             // stage B column groups of 4
  static constexpr int N1_P = TX / 2 + 4;                              // horizontal L1 pass, col c <-> x0/2+c
  static constexpr int OFF_U8 = 0;
  static constexpr int OFF_HS = U8_W * U8_H;
  static constexpr int OFF_L0 = OFF_HS + HS_H * HS_P * 4;
  static constexpr int OFF_HD = OFF_HS;                                // Hd reuses Hs
  static constexpr int OFF_HG = OFF_L0 + L0_H * L0_P * 4;
  static constexpr int OFF_N1 = OFF_HG + HG_H * HG_P * 4;
  static constexpr int OFF_BAR = OFF_N1 + (NX ? L0_H * N1_P * 4 : 0);
  static constexpr int SMEM = OFF_BAR + 16;
  static_assert(L0_H % PYB == 0 && TY % PYD == 0 && (TX / 4) * (TY / PYD) <= 128 && (L0_H / PYB) * NGB <= 256, "stage B / D mapping");
  static_assert(HG_H * HG_P <= HS_H * HS_P && 4 * NGB <= L0_P && 8 * 9 + (NX ? 4 : 0) <= HS_P, "buffer shapes");
  static_assert(CPS * (SMEM + 1024) <= 228 * 1024, "CPS resident CTAs must fit into the SM's shared memory");
};
using L0Geo = L0GeoT<64, 5, 8, 3>;       // (tile width, halo and radii are the same for every variant)

// stage A item: NOUT (8, or 4 for the last column group of the NX geometry) outputs (Hs cols
// 8g..8g+NOUT-1 <-> global x0-4+8g+q) of row r from 12 u8 pixels
template <class G, bool EXACT, bool BORDER, int NOUT = 8>
__device__ __forceinline__ void l0_stage_a_item(const unsigned char* sU8, float* sHs, const TapsF& ts,
                                                int r, int g, int x0, int W) {
  constexpr int RS = G::RS;
  const uint2 wa = *reinterpret_cast<const uint2*>(sU8 + r * G::U8_W + 8 * g + 8);
  const uint2 wb = *reinterpret_cast<const uint2*>(sU8 + r * G::U8_W + 8 * g + 16);
  float px[12];                                         // global cols x0-6+8g .. x0+5+8g
  px[0] = u8_to_float(wa.x, 2); px[1] = u8_to_float(wa.x, 3);
  px[2] = u8_to_float(wa.y, 0); px[3] = u8_to_float(wa.y, 1);
  px[4] = u8_to_float(wa.y, 2); px[5] = u8_to_float(wa.y, 3);
  px[6] = u8_to_float(wb.x, 0); px[7] = u8_to_float(wb.x, 1);
  px[8] = u8_to_float(wb.x, 2); px[9] = u8_to_float(wb.x, 3);
  px[10] = u8_to_float(wb.y, 0); px[11] = u8_to_float(wb.y, 1);
  float o[8];
#pragma unroll
  for (int q = 0; q < NOUT; ++q) {
    float acc = 0.0f;
#pragma unroll
    for (int m = 0; m < 2 * RS + 1; ++m) acc = mac<EXACT>(acc, px[q + m], ts.k[m]);
    if (BORDER) {
      const int xg = x0 - 4 + 8 * g + q;
      if (xg < RS || xg >= W - RS) acc = 0.0f;
    }
    o[q] = acc;
  }
  float4* dst = reinterpret_cast<float4*>(sHs + r * G::HS_P + 8 * g);
  dst[0] = make_float4(o[0], o[1], o[2], o[3]);
  if (NOUT == 8) dst[1] = make_float4(o[4], o[5], o[6], o[7]);
}

template <class G, bool EXACT, bool BORDER>
__device__ __forceinline__ void l0_fused_tile(unsigned char* smem, int W, const TapsF& ts, int x0) {
  const unsigned char* sU8 = smem + G::OFF_U8;
  float* sHs = reinterpret_cast<float*>(smem + G::OFF_HS);
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;

  // ---- stage A: horizontal Gaussian, u8 -> Hs: 9 groups of 8 columns x 74 rows -------------
  {
    const int sub = lane & 3, rpar = (lane >> 2) & 1, half = (lane >> 3) & 1, rpair = lane >> 4;
    for (int rb = warp * 4; rb < G::HS_H; rb += 32) {
      const int r = rb + 2 * rpair + rpar;
      if (r < G::HS_H) l0_stage_a_item<G, EXACT, BORDER>(sU8, sHs, ts, r, 4 * half + sub, x0, W);
    }
    if (tid < G::HS_H) l0_stage_a_item<G, EXACT, BORDER>(sU8, sHs, ts, tid, 8, x0, W);   // 9th group
    else if (G::NX && tid < 2 * G::HS_H)                                                   // col x0+68
      l0_stage_a_item<G, EXACT, BORDER, 4>(sU8, sHs, ts, tid - G::HS_H, 9, x0, W);
  }
}

template <class G, bool EXACT, bool BORDER>
__device__ __forceinline__ void l0_fused_tile_rest(unsigned char* smem, int W, int H, const TapsF& ts,
                                                   const TapsF& tg, const TapsF& td, const TapsF& tp,
                                                   float* __restrict__ out_img,
                                                   float* __restrict__ out_gx,
                                                   float* __restrict__ out_gy, int opitch,
                                                   float* __restrict__ out_l1, int l1pitch, int W1, int H1,
                                                   int x0, int y0) {
  constexpr int RS = G::RS, RG = G::RG, XR = G::XR;
  float* sHs = reinterpret_cast<float*>(smem + G::OFF_HS);
  float* sL0 = reinterpret_cast<float*>(smem + G::OFF_L0);
  float* sHd = reinterpret_cast<float*>(smem + G::OFF_HD);
  float* sHg = reinterpret_cast<float*>(smem + G::OFF_HG);
  float* sN1 = reinterpret_cast<float*>(smem + G::OFF_N1);
  const int tid = threadIdx.x;

  // ---- stage B: vertical Gaussian, Hs -> L0 (shared + HBM) ------------------------------------
  // NGB column groups of 4 (col c <-> x0-4+c) x NBLK row blocks of PYB (14 x 5 for the 64-row tile).
  // The first 16 * NBLK threads take groups 0..15 (a quarter warp = 8 consecutive groups of one row
  // block: contiguous 128 B), the next NH * NBLK the halo groups.
  constexpr int NBLK = G::L0_H / G::PYB, NH = G::NGB - 16;
  if (tid < G::NGB * NBLK) {
    constexpr int PY = G::PYB;
    const unsigned long long pol_img = store_policy(true);
    int blk, j;
    if (tid < 16 * NBLK) { blk = tid >> 4; j = tid & 15; }
    else { const int t2 = tid - 16 * NBLK; blk = t2 / NH; j = 16 + (t2 - blk * NH); }
    float4 acc[PY];
#pragma unroll
    for (int q = 0; q < PY; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* src = sHs + (blk * PY) * G::HS_P + 4 * j;
#pragma unroll
    for (int i = 0; i < PY + 2 * RS; ++i) {            // L0 row rr needs Hs rows rr .. rr+2RS
      const float4 v = lds128(src + i * G::HS_P);
#pragma unroll
      for (int q = 0; q < PY; ++q) {
        const int m = i - q;
        if (m >= 0 && m <= 2 * RS) fma4(acc[q], v, ts, m, EXACT);
      }
    }
    const int xg = x0 - 4 + 4 * j;
#pragma unroll
    for (int q = 0; q < PY; ++q) {
      const int rr = blk * PY + q;
      const int yg = y0 - RG - XR + rr;
      if (BORDER) {
        if (yg < RS || yg >= H - RS) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      *reinterpret_cast<float4*>(sL0 + rr * G::L0_P + 4 * j) = acc[q];
      if (j >= 1 && j <= 16 && rr >= RG + XR && rr < RG + XR + G::TY) {
        if (!BORDER || (xg < W && yg < H))
          stg128(out_img + (size_t)yg * opitch + xg, acc[q], pol_img);
      }
    }
  }
  tile_sync();

  stage_hgrad<EXACT, BORDER, G::TX, G::HG_H, G::L0_P, G::HG_P>(sL0 + XR * G::L0_P, sHd, sHg, tg, td, x0, W);
  if (G::NX) stage_hnext<EXACT, BORDER, G::TX, G::L0_H, G::L0_P, G::N1_P>(sL0, sN1, tp, x0, W);
  tile_sync();
  stage_vgrad_both<EXACT, BORDER, G::TX, G::TY, G::PYD, G::HG_P>(sHd, sHg, tg, td, out_gx, out_gy, opitch,
                                                            x0, y0, W, H);
  if (G::NX) stage_vnext<EXACT, BORDER, G::TX, G::TY, G::N1_P>(sN1, tp, out_l1, l1pitch, x0, y0, H, W1, H1);
}

template <class G, bool EXACT>
__global__ void __launch_bounds__(256, G::CPS)
l0_fused_kernel(const __grid_constant__ CUtensorMap map, int W, int H, const __grid_constant__ TileQueue q,
                TapsF ts, TapsF tg, TapsF td, float* __restrict__ out_img,
                float* __restrict__ out_gx, float* __restrict__ out_gy, int opitch,
                TapsF tp, float* __restrict__ out_l1, int l1pitch, int W1, int H1) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // tiles whose 8-pixel margin stays inside the image never meet a zero band
  auto border = [&](int x0, int y0) { return (x0 < 8) || (y0 < 8) || (x0 + G::TX + 8 > W) || (y0 + G::TY + 8 > H); };
  // Nothing this kernel READS comes from its predecessor in the stream (the u8 frame is resident, or
  // its upload is ordered by an event the launch itself waited for); only the pyramid slot it WRITES
  // may still be in use (the previous frame's tracker reads the other two slots and the feature
  // arrays).  So the first tile's load and horizontal pass run before griddepcontrol.wait -- under
  // the predecessor's tail -- and the wait sits in front of the first global store.
  tile_queue<G::TX, G::TY, false>(
      q, &map, smem_raw + G::OFF_U8, G::U8_W * G::U8_H, smem_raw + G::OFF_BAR, border,
      [&](int x0, int y0) { return make_int2(x0 - 16, y0 - (G::RS + G::RG + G::XR)); },
      [&](int x0, int y0, bool border) {
        if (border) l0_fused_tile<G, EXACT, true>(smem_raw, W, ts, x0);
        else l0_fused_tile<G, EXACT, false>(smem_raw, W, ts, x0);
      },
      // (stage D reads Hd, aliased on Hs, and Hg: the barrier after it keeps the next stage A out)
      [&](int x0, int y0, bool border) {
        if (border)
          l0_fused_tile_rest<G, EXACT, true>(smem_raw, W, H, ts, tg, td, tp, out_img, out_gx, out_gy, opitch, out_l1,
                                             l1pitch, W1, H1, x0, y0);
        else
          l0_fused_tile_rest<G, EXACT, false>(smem_raw, W, H, ts, tg, td, tp, out_img, out_gx, out_gy, opitch, out_l1,
                                              l1pitch, W1, H1, x0, y0);
      });
}

// ============================================================================================
// levels >= 1: one pyramid step (Gaussian at the kept samples) + gradients
// ============================================================================================
template <int SS, int R, int TX, int TY>
struct LvGeo {
  static constexpr int RG = FUSED_RG;
  static constexpr int LW = TX + 8, LH = TY + 2 * RG;                  // level tile, col c <-> x0-4+c
  static constexpr int NGL = LW / 4;                                   // column groups of 4
  static constexpr int LP = LW + 4;                                    // odd number of chunks
  static constexpr int HP = TX + 4;
  static constexpr int NW1 = 3 * SS + 2 * R + 1;                       // source window of 4 kept outputs
  static constexpr int NV1 = (NW1 + 3) / 4;
  static constexpr int SW0 = SS * 4 * (NGL - 1) + 4 * NV1;
  static constexpr int SW = ((SW0 / 4) & 1) ? SW0 : SW0 + 4;           // source box width, odd chunks
  static constexpr int SH = SS * (LH - 1) + 2 * R + 1;                 // source box height
  static constexpr int XOFF = SS / 2 - R - 4 * SS;                     // source col of tile col 0, minus SS*x0
  static constexpr int YOFF = SS / 2 - R - RG * SS;
  static_assert(XOFF % 4 == 0, "source box must start on a 16 B boundary");
  static_assert((LP / 4) % 2 == 1 && (HP / 4) % 2 == 1 && (SW / 4) % 2 == 1, "odd chunk pitches");
  static constexpr int OFF_SRC = 0;
  static constexpr int OFF_HP = SW * SH * 4;
  // pitch of the horizontal-pass buffer: 64 B more than a multiple of 128 B, so that the two rows a
  // quarter warp stores in P1 (4 groups x 16 B each) fall into disjoint bank halves (ncu: the 72-float
  // pitch cost 88 % extra wavefronts on that store)
  static constexpr int HPP = ((LW * 4 + 127) / 128) * 32 + (((LW * 4) % 128) <= 64 && ((LW * 4) % 128) != 0 ? -16 : 16);
  static_assert(HPP >= LW && (HPP * 4) % 128 == 64, "Hp pitch");
  static constexpr int HP_BYTES = SH * HPP * 4, HDG_BYTES = 2 * LH * HP * 4;
  static constexpr int OFF_L = OFF_HP + (HP_BYTES > HDG_BYTES ? HP_BYTES : HDG_BYTES);
  static constexpr int OFF_HD = OFF_HP;                                // Hd, Hg reuse Hp (dead after P2)
  static constexpr int OFF_HG = OFF_HD + LH * HP * 4;
  static constexpr int OFF_BAR = OFF_L + LH * LP * 4;
  static constexpr int SMEM = OFF_BAR + 16;
};

// P1 item: 4 kept outputs (tile cols 4g..4g+3) of source row r
template <bool EXACT, bool BORDER, int SS, int R, int TX, int TY>
__device__ __forceinline__ void lv_p1_item(const float* sSrc, float* sHp, const TapsF& tp, int r, int g,
                                           int x0, int Wsrc) {
  using G = LvGeo<SS, R, TX, TY>;
  float win[4 * G::NV1];
  const float* p = sSrc + r * G::SW + SS * 4 * g;
#pragma unroll
  for (int v = 0; v < G::NV1; ++v) {
    const float4 t = lds128(p + 4 * v);
    win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
  }
  float o[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float acc = 0.0f;
#pragma unroll
    for (int m = 0; m < 2 * R + 1; ++m) acc = mac<EXACT>(acc, win[SS * q + m], tp.k[m]);
    if (BORDER) {
      const int xs = SS * (x0 - 4 + 4 * g + q) + SS / 2;
      if (xs < R || xs >= Wsrc - R) acc = 0.0f;
    }
    o[q] = acc;
  }
  *reinterpret_cast<float4*>(sHp + r * G::HPP + 4 * g) = make_float4(o[0], o[1], o[2], o[3]);
}

template <bool EXACT, bool BORDER, int SS, int R, int TX, int TY, int NTH = 256>
__device__ __forceinline__ void lv_stage_p1(const unsigned char* smem, const TapsF& tp, int x0, int Wsrc) {
  using G = LvGeo<SS, R, TX, TY>;
  const float* sSrc = reinterpret_cast<const float*>(smem + G::OFF_SRC);
  float* sHp = const_cast<float*>(reinterpret_cast<const float*>(smem + G::OFF_HP));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // a warp covers 8 groups x 4 rows; quarter warp = (8/SS) groups x SS rows (conflict free, see top)
  int g8, rl;
  if (SS == 2) { g8 = 4 * ((lane >> 3) & 1) + (lane & 3); rl = 2 * (lane >> 4) + ((lane >> 2) & 1); }
  else         { g8 = 2 * (lane >> 3) + (lane & 1);       rl = (lane >> 1) & 3; }
  constexpr int NMAIN = (G::NGL / 8) * 8, NCH = NMAIN / 8, NRB = (G::SH + 3) / 4;
  for (int u = warp; u < NRB * NCH; u += NTH / 32) {
    const int rbk = u / NCH, ch = u - rbk * NCH;
    const int r = 4 * rbk + rl;
    if (r < G::SH) lv_p1_item<EXACT, BORDER, SS, R, TX, TY>(sSrc, sHp, tp, r, 8 * ch + g8, x0, Wsrc);
  }
  constexpr int NTAIL = G::NGL - NMAIN;
  for (int it = tid; it < G::SH * NTAIL; it += NTH) {
    const int r = it / NTAIL, g = NMAIN + it - r * NTAIL;
    lv_p1_item<EXACT, BORDER, SS, R, TX, TY>(sSrc, sHp, tp, r, g, x0, Wsrc);
  }
}

template <bool EXACT, bool BORDER, int SS, int R, int TX, int TY, int NTH = 256>
__device__ __forceinline__ void lv_stage_rest(unsigned char* smem, const TapsF& tp, const TapsF& tg,
                                              const TapsF& td, int Hsrc, int W, int H,
                                              float* __restrict__ out_img, float* __restrict__ out_gx,
                                              float* __restrict__ out_gy, int opitch, int x0, int y0) {
  using G = LvGeo<SS, R, TX, TY>;
  constexpr int RG = G::RG;
  const float* sHp = reinterpret_cast<const float*>(smem + G::OFF_HP);
  float* sL = reinterpret_cast<float*>(smem + G::OFF_L);
  float* sHd = reinterpret_cast<float*>(smem + G::OFF_HD);
  float* sHg = reinterpret_cast<float*>(smem + G::OFF_HG);
  const int tid = threadIdx.x;

  // ---- P2: vertical Gaussian at the kept rows, Hp -> level tile (shared + HBM) -----------------
  // item = 4 columns x 2 level rows; level row rr needs Hp rows SS*rr .. SS*rr+2R
  {
    constexpr int NMAIN = (G::NGL / 8) * 8, NPAIR = G::LH / 2, NTAIL = G::NGL - NMAIN;
    static_assert(G::LH % 2 == 0, "level tile height must be even");
    constexpr int NR2 = SS + 2 * R + 1;
    const unsigned long long pol_img = store_policy(true);
    for (int it = tid; it < NPAIR * G::NGL; it += NTH) {
      int pr, j;
      if (it < NPAIR * NMAIN) { pr = it / NMAIN; j = it - pr * NMAIN; }
      else { const int t2 = it - NPAIR * NMAIN; pr = t2 / NTAIL; j = NMAIN + t2 - pr * NTAIL; }
      float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
      const float* src = sHp + (SS * 2 * pr) * G::HPP + 4 * j;
#pragma unroll
      for (int i = 0; i < NR2; ++i) {
        const float4 v = lds128(src + i * G::HPP);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int m = i - SS * q;
          if (m >= 0 && m <= 2 * R) fma4(acc[q], v, tp, m, EXACT);
        }
      }
      const int xg = x0 - 4 + 4 * j;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int rr = 2 * pr + q;
        const int yg = y0 - RG + rr;
        if (BORDER) {
          const int ys = SS * yg + SS / 2;
          if (ys < R || ys >= Hsrc - R) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        *reinterpret_cast<float4*>(sL + rr * G::LP + 4 * j) = acc[q];
        if (j >= 1 && j <= G::NGL - 2 && rr >= RG && rr < RG + TY) {
          if (!BORDER || (xg < W && yg < H))
            stg128(out_img + (size_t)yg * opitch + xg, acc[q], pol_img);
        }
      }
    }
  }
  tile_sync<NTH>();
  stage_hgrad<EXACT, BORDER, TX, G::LH, G::LP, G::HP, NTH>(sL, sHd, sHg, tg, td, x0, W);
  tile_sync<NTH>();
  // output rows per thread of the last stage: as few as the thread count allows (fewer rows = more items)
  constexpr int PY = (TX / 4) * (TY / 2) <= NTH / 2 ? 2 : ((TX / 4) * (TY / 4) <= NTH / 2 ? 4 : 8);
  stage_vgrad_both<EXACT, BORDER, TX, TY, PY, G::HP, NTH>(sHd, sHg, tg, td, out_gx, out_gy, opitch, x0, y0, W, H);
}

// W,H: size of the level being produced; Wsrc,Hsrc: size of the level it is made from.
// NTH threads per CTA: 256, or 512 for the big-tile shapes whose shared-memory footprint allows only two
// CTAs per SM (16 warps per SM leave the tile's four-stage chain latency bound; 32 do not).
template <int SS, int R, int TX, int TY>
__host__ __device__ constexpr int lv_threads() { return (LvGeo<SS, R, TX, TY>::SMEM > 75 * 1024 && SS == 2) ? 512 : 256; }
template <int SS, int R, int TX, int TY, bool EXACT>
__global__ void __launch_bounds__((lv_threads<SS, R, TX, TY>()), (LvGeo<SS, R, TX, TY>::SMEM <= 75 * 1024) ? 3 : 2)
level_fused_kernel(const __grid_constant__ CUtensorMap map, int Wsrc, int Hsrc, int W, int H,
                   const __grid_constant__ TileQueue q, TapsF tp, TapsF tg, TapsF td,
                   float* __restrict__ out_img, float* __restrict__ out_gx,
                   float* __restrict__ out_gy, int opitch) {
  using G = LvGeo<SS, R, TX, TY>;
  constexpr int NTH = lv_threads<SS, R, TX, TY>();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // interior tiles (margins derived in DESIGN.md) never meet a zero band at either level
  auto border = [&](int x0, int y0) { return (x0 < 8) || (y0 < 8) || (x0 + TX + 16 > W) || (y0 + TY + 16 > H); };
  // (waits before its first claim: the source level is written by the previous kernel)
  tile_queue<TX, TY, true>(
      q, &map, smem_raw + G::OFF_SRC, G::SW * G::SH * 4, smem_raw + G::OFF_BAR, border,
      [&](int x0, int y0) { return make_int2(SS * x0 + G::XOFF, SS * y0 + G::YOFF); },
      [&](int x0, int y0, bool border) {
        if (border) lv_stage_p1<EXACT, true, SS, R, TX, TY, NTH>(smem_raw, tp, x0, Wsrc);
        else lv_stage_p1<EXACT, false, SS, R, TX, TY, NTH>(smem_raw, tp, x0, Wsrc);
      },
      [&](int x0, int y0, bool border) {
        if (border)
          lv_stage_rest<EXACT, true, SS, R, TX, TY, NTH>(smem_raw, tp, tg, td, Hsrc, W, H, out_img, out_gx, out_gy, opitch, x0, y0);
        else
          lv_stage_rest<EXACT, false, SS, R, TX, TY, NTH>(smem_raw, tp, tg, td, Hsrc, W, H, out_img, out_gx, out_gy, opitch, x0, y0);
      });
}

// ============================================================================================
// levels >= 1 of a subsampling-2, radius-5 pyramid whose level 0 came from the NX geometry:
// L_l -> gx_l, gy_l (+ L_{l+1} when NX).  The pyramid step of level l has already been done by the
// previous kernel of the chain, from the tile it held on chip, so a tile only loads its own part of
// L_l plus the halo of the two passes (76 x 41 floats for 64 x 32) and runs two stages:
//   1: horizontal DoG / Gaussian (stage_hgrad) + horizontal pass of the next level
//   2: vertical Gaussian / DoG (stage_vgrad_both) + vertical pass and store of the next level
// ============================================================================================
template <int TX, int TY>
struct ChGeo {
  static constexpr int RG = FUSED_RG, RN = NEXT_R;
  static constexpr int SW = TX + 12, SH = TY + 2 * RN - 1;             // col c <-> x0-4+c, row r <-> y0-4+r
  static constexpr int HP = TX + 4, GH = TY + 2 * RG;                  // Hd / Hg: col c <-> x0+c, row r <-> y0-3+r
  static constexpr int NP = TX / 2 + 4;                                // next level's horizontal pass
  static_assert(SW >= TX + 2 * RN - 1 && (SW / 4) % 2 == 1 && (HP / 4) % 2 == 1, "box width / odd chunk pitches");
  static_assert(RN - 1 - RG >= 0, "the gradient rows lie inside the box");
  static constexpr int OFF_SRC = 0;
  static constexpr int OFF_HD = OFF_SRC + SW * SH * 4;
  static constexpr int OFF_HG = OFF_HD + GH * HP * 4;
  static constexpr int OFF_N = OFF_HG + GH * HP * 4;
  static constexpr int OFF_BAR = OFF_N + SH * NP * 4;
  static constexpr int SMEM = OFF_BAR + 16;
};

// W,H: size of level l; Wn,Hn: size of level l+1 (unused without NX).
template <int TX, int TY, bool NX, bool EXACT>
__global__ void __launch_bounds__(256, 4)
level_chain_kernel(const __grid_constant__ CUtensorMap map, int W, int H, int Wn, int Hn,
                   const __grid_constant__ TileQueue q, TapsF tp, TapsF tg, TapsF td, float* __restrict__ out_gx,
                   float* __restrict__ out_gy, int opitch, float* __restrict__ out_next, int npitch) {
  using G = ChGeo<TX, TY>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const float* sL = reinterpret_cast<const float*>(smem_raw + G::OFF_SRC);
  const float* sLg = sL + (G::RN - 1 - G::RG) * G::SW;
  float* sHd = reinterpret_cast<float*>(smem_raw + G::OFF_HD);
  float* sHg = reinterpret_cast<float*>(smem_raw + G::OFF_HG);
  float* sN = reinterpret_cast<float*>(smem_raw + G::OFF_N);
  // output rows per thread of stage 2: as few as the thread count allows (fewer rows = more items)
  constexpr int PY = (TX / 4) * (TY / 2) <= 128 ? 2 : ((TX / 4) * (TY / 4) <= 128 ? 4 : 8);
  // tiles whose 8-pixel margin stays inside level l meet no zero band of either pass and no edge
  auto border = [&](int x0, int y0) { return (x0 < 8) || (y0 < 8) || (x0 + TX + 8 > W) || (y0 + TY + 8 > H); };
  // (waits before its first claim: L_l is written by the previous kernel)
  tile_queue<TX, TY, true>(
      q, &map, smem_raw + G::OFF_SRC, G::SW * G::SH * 4, smem_raw + G::OFF_BAR, border,
      [&](int x0, int y0) { return make_int2(x0 - 4, y0 + 1 - G::RN); },
      [&](int x0, int y0, bool border) {
        if (border) {
          stage_hgrad<EXACT, true, TX, G::GH, G::SW, G::HP>(sLg, sHd, sHg, tg, td, x0, W);
          if (NX) stage_hnext<EXACT, true, TX, G::SH, G::SW, G::NP>(sL, sN, tp, x0, W);
        } else {
          stage_hgrad<EXACT, false, TX, G::GH, G::SW, G::HP>(sLg, sHd, sHg, tg, td, x0, W);
          if (NX) stage_hnext<EXACT, false, TX, G::SH, G::SW, G::NP>(sL, sN, tp, x0, W);
        }
      },
      [&](int x0, int y0, bool border) {
        if (border) {
          stage_vgrad_both<EXACT, true, TX, TY, PY, G::HP>(sHd, sHg, tg, td, out_gx, out_gy, opitch, x0, y0, W, H);
          if (NX) stage_vnext<EXACT, true, TX, TY, G::NP>(sN, tp, out_next, npitch, x0, y0, H, Wn, Hn);
        } else {
          stage_vgrad_both<EXACT, false, TX, TY, PY, G::HP>(sHd, sHg, tg, td, out_gx, out_gy, opitch, x0, y0, W, H);
          if (NX) stage_vnext<EXACT, false, TX, TY, G::NP>(sN, tp, out_next, npitch, x0, y0, H, Wn, Hn);
        }
      });
}
