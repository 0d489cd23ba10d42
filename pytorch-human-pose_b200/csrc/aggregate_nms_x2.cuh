// Specialised fused aggregation + NMS kernel for the standard HigherHRNet single-scale layout:
//   hm_lo, tag at 1/4 resolution, hm_hi at 1/2 resolution, output at full resolution
//   (lo --x2--> hi, mean, --x2--> out ; tag --x4--> out).
// Included by aggregate_nms.cu (needs AggArgs).  Bit-identical to the generic kernel: the taps and
// weights below are what axis_tap() yields for exact x2 / x4 ratios (all weights are exact in f32),
// including the clamped first/last rows and columns.
//
// Work decomposition (B200: issue-bound otherwise -- the generic kernel spends ~370 instructions
// per output pixel; this one ~65, which leaves the kernel bound by HBM writes):
//   * one CTA = a band of RB output rows x (128 * NW) columns of one (image, joint) plane;
//   * phase 0 (tag bounds): the quarter-res tile of the first tag component is staged (16-byte loads, one
//     warp per tile row) and every word of the band gets the per-(4 rows x word) range of the tags its
//     pixels interpolate from (tag_bmin / tag_bmax, the refine prefilter).  The tag tile aliases the
//     half-res tile, so shared memory stays at 30 KB (6 CTAs/SM).  The full-resolution tag map is not
//     written here: the tag stages interpolate the few tags they read (tag_at), and aggregate_tags_kernel
//     writes the map for callers that keep one;
//   * phase 1 (all threads): flip-averaged quarter-res / half-res tiles -> smem, tile interiors 16-byte
//     aligned, two rows per batch so that all loads of a batch are in flight before the first store;
//   * phase 2 (all threads): stage mean S at half resolution, in place, exact torch arithmetic
//     (compile-time taps for bands that touch neither the first nor the last image rows);
//   * phase 3 (per warp, no CTA barrier): every lane owns 4 adjacent output columns and walks
//     down the rows with everything in registers: horizontal interpolation of each half-res row
//     once, vertical interpolation per row, one 16-byte store of the heatmap, 5-wide row maximum via
//     warp shuffles (halo columns from a per-warp prologue), 5-tall column maximum in a register
//     window, survivor test, and per-32-pixel-word mask / maxima reduced over the 8 lanes of the word.
#pragma once

namespace x2 {

constexpr int RB = 32;                 // output rows per CTA band (multiple of 4)
constexpr int SR = RB / 2 + 4;         // half-res rows staged
constexpr int LR = RB / 4 + 4;         // quarter-res rows staged (hm_lo)
constexpr int TR = RB / 4 + 2;         // quarter-res rows staged (tags)
constexpr int NROWS = RB + 4;          // output rows walked (band + 2 halo rows on each side)

__host__ __device__ inline int SC(int NW) { return 64 * NW + 8; }   // half-res cols: hx0-4 .. (interior 16B aligned)
__host__ __device__ inline int LC(int NW) { return 32 * NW + 8; }   // quarter-res cols: lx0-4 ..
__host__ __device__ inline size_t smem_floats(int NW) {
  // the tag tile (TR * LC <= SR * SC floats) aliases the half-res tile
  return (size_t)SR * SC(NW) + (size_t)LR * LC(NW) + (size_t)NW * NROWS * 4 + 4 * SR + 8;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// x2 tap of output index o (input size I): generic axis_tap specialised, used in phase 2 only
__device__ __forceinline__ void tap_x2(int o, int I, int& i0, int& i1, float& w0, float& w1) {
  if (o == 0) { i0 = 0; i1 = (I > 1) ? 1 : 0; w0 = 1.f; w1 = 0.f; return; }
  if (o & 1) { i0 = o >> 1; w0 = 0.75f; w1 = 0.25f; }
  else       { i0 = (o >> 1) - 1; w0 = 0.25f; w1 = 0.75f; }
  i1 = (i0 < I - 1) ? i0 + 1 : i0;
}

// Stage a ROWS x COLS tile (origin (yo, xo), coordinates clamped to the map = border replication)
// into shared memory.  COLS = 4 halo + interior + 4 halo columns, the interior starting at a
// 16-byte aligned column of the map.  One warp per tile row, two rows per batch (all loads of a
// batch are in flight before the first is consumed).  VEC: 16-byte loads/stores for the interior
// (the flipped operand is read as the mirrored 16 bytes and reversed in registers), scalars for the
// 8 halo columns and for any part right of the map.
//   AVG = false: dst = p[y][x]      AVG = true: dst = (p[y][x] + pf[y][w-1-x]) * 0.5   (flip averaging, model.py:90)
// Input element type: float32 (inference), IEEE half (the validation-time caller runs the network under fp16
// autocast, module.py:78) or bfloat16 (bf16 autocast).  16-bit values are widened on load -- exactly -- and
// everything after is float32 arithmetic.
template <typename T> struct In;
template <> struct In<float> {
  static __device__ __forceinline__ float4 ld4(const float* q) { return __ldg(reinterpret_cast<const float4*>(q)); }
  static __device__ __forceinline__ float ld1(const float* q) { return __ldg(q); }
};
template <> struct In<__half> {
  static __device__ __forceinline__ float4 ld4(const __half* q) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(q));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  static __device__ __forceinline__ float ld1(const __half* q) { return __half2float(__ldg(q)); }
};
template <> struct In<__nv_bfloat16> {   // a bfloat16 is the upper 16 bits of the float32 of the same value
  static __device__ __forceinline__ float4 ld4(const __nv_bfloat16* q) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(q));
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
  }
  static __device__ __forceinline__ float ld1(const __nv_bfloat16* q) {
    return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short*>(q)) << 16);
  }
};

template <bool AVG>
__device__ __forceinline__ float stage_combine(float v, float f) {
  return AVG ? __fmul_rn(__fadd_rn(v, f), 0.5f) : v;
}

template <bool AVG, int ROWS, int COLS, int NW, bool VEC, typename T = float>
__device__ __forceinline__ void stage_tile(float* __restrict__ dst, const T* __restrict__ p,
                                           const T* __restrict__ pf, int yo, int xo, int h, int w,
                                           int warp, int lane) {
  constexpr int RPB = 2;
  const int xm = w - 1;
  if (VEC) {
    constexpr int NV = (COLS - 8) / 4, VIT = (NV + 31) / 32;
#pragma unroll 1
    for (int r0 = warp * RPB; r0 < ROWS; r0 += NW * RPB) {
      float4 v[RPB][VIT], f[RPB][VIT];
      float hv[RPB], hf[RPB];
#pragma unroll
      for (int j = 0; j < RPB; ++j) {
        const int r = r0 + j;
        const int row = clampi(yo + r, 0, h - 1) * w;
#pragma unroll
        for (int u = 0; u < VIT; ++u) {
          const int q = lane + 32 * u;
          const int x = xo + 4 + 4 * q;
          v[j][u] = make_float4(0.f, 0.f, 0.f, 0.f);
          f[j][u] = v[j][u];
          if (r < ROWS && q < NV) {
            if (x + 3 <= xm) {
              v[j][u] = In<T>::ld4(p + row + x);
              if (AVG) {
                const float4 t = In<T>::ld4(pf + row + (xm - x - 3));
                f[j][u] = make_float4(t.w, t.z, t.y, t.x);
              }
            } else {   // right of the map: replicate the last column
              float tv[4], tf[4];
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const int xc = min(x + c, xm);
                tv[c] = In<T>::ld1(p + row + xc);
                tf[c] = AVG ? In<T>::ld1(pf + row + (xm - xc)) : 0.f;
              }
              v[j][u] = make_float4(tv[0], tv[1], tv[2], tv[3]);
              f[j][u] = make_float4(tf[0], tf[1], tf[2], tf[3]);
            }
          }
        }
        hv[j] = 0.f; hf[j] = 0.f;
        if (r < ROWS && lane < 8) {
          const int c = (lane < 4) ? lane : COLS - 8 + lane;
          const int x = clampi(xo + c, 0, xm);
          hv[j] = In<T>::ld1(p + row + x);
          if (AVG) hf[j] = In<T>::ld1(pf + row + (xm - x));
        }
      }
#pragma unroll
      for (int j = 0; j < RPB; ++j) {
        const int r = r0 + j;
        if (r >= ROWS) break;
#pragma unroll
        for (int u = 0; u < VIT; ++u) {
          const int q = lane + 32 * u;
          if (q < NV)
            *reinterpret_cast<float4*>(dst + r * COLS + 4 + 4 * q) =
                make_float4(stage_combine<AVG>(v[j][u].x, f[j][u].x), stage_combine<AVG>(v[j][u].y, f[j][u].y),
                            stage_combine<AVG>(v[j][u].z, f[j][u].z), stage_combine<AVG>(v[j][u].w, f[j][u].w));
        }
        if (lane < 8) dst[r * COLS + ((lane < 4) ? lane : COLS - 8 + lane)] = stage_combine<AVG>(hv[j], hf[j]);
      }
    }
  } else {
    constexpr int NIT = (COLS + 31) / 32;
#pragma unroll 1
    for (int r0 = warp * RPB; r0 < ROWS; r0 += NW * RPB) {
      float v[RPB][NIT], f[RPB][NIT];
#pragma unroll
      for (int j = 0; j < RPB; ++j) {
        const int r = r0 + j;
        const int row = clampi(yo + r, 0, h - 1) * w;
#pragma unroll
        for (int u = 0; u < NIT; ++u) {
          const int c = lane + 32 * u;
          v[j][u] = 0.f; f[j][u] = 0.f;
          if (r < ROWS && c < COLS) {
            const int x = clampi(xo + c, 0, xm);
            v[j][u] = In<T>::ld1(p + row + x);
            if (AVG) f[j][u] = In<T>::ld1(pf + row + (xm - x));
          }
        }
      }
#pragma unroll
      for (int j = 0; j < RPB; ++j) {
        const int r = r0 + j;
#pragma unroll
        for (int u = 0; u < NIT; ++u) {
          const int c = lane + 32 * u;
          if (r < ROWS && c < COLS) dst[r * COLS + c] = stage_combine<AVG>(v[j][u], f[j][u]);
        }
      }
    }
  }
}

// The NMS half of the column walk, shared by the x2 and the multi-scale kernel.  A lane owns 4 adjacent
// output columns and is fed their values row by row (t = index of the row in the walk, row y = ys + t, rows
// outside the image carry -inf).  Every row is stored to the aggregated heatmap (if it belongs to the band),
// reduced to its 5-wide row maximum (own 4 + 2 from each neighbour lane, the strip's halo columns from
// `edge`), and pushed into a register window: r0..r3 = row maxima of rows y-4..y-1, vq0 / vq1 = values of
// rows y-2 / y-1.  The centre row y-2 then gets its 5-tall column maximum, survivor bits (grouping.py:80-83)
// and the per-word side arrays (survivor mask, maximum of the survivors, maximum of the raw values).
template <int RB>
struct NmsColumnWalk {
  float r0[4], r1[4], r2[4], r3[4], vq0[4], vq1[4];
  float* hm_plane;
  const float* edge;
  size_t wbase;
  int ys, lane, shl;
  bool active, word_writer;

  __device__ __forceinline__ void init(const AggArgs& a, int b, int k, int X0, int ys_, const float* edge_, bool active_,
                                       int lane_) {
#pragma unroll
    for (int c = 0; c < 4; ++c) { r0[c] = r1[c] = r2[c] = r3[c] = -INFINITY; vq0[c] = vq1[c] = -INFINITY; }
    hm_plane = a.agg_hm + ((size_t)b * a.K + k) * a.H * a.W + X0;
    wbase = ((size_t)b * a.K + k) * a.H * a.wpr + (X0 >> 5);
    edge = edge_;
    ys = ys_; lane = lane_; active = active_;
    word_writer = active_ && (lane_ & 7) == 0;
    shl = 4 * (lane_ & 7);
  }

  __device__ __forceinline__ void row(const AggArgs& a, int t, const float (&v)[4]) {
    const int H = a.H, W = a.W;
    const int y = ys + t;
    if (t >= 2 && t < RB + 2 && y < H && active)
      *reinterpret_cast<float4*>(hm_plane + (size_t)y * W) = make_float4(v[0], v[1], v[2], v[3]);
    float l2 = __shfl_up_sync(kFull, v[2], 1), l3 = __shfl_up_sync(kFull, v[3], 1);
    float q0 = __shfl_down_sync(kFull, v[0], 1), q1 = __shfl_down_sync(kFull, v[1], 1);
    if (lane == 0) { const float2 e = *reinterpret_cast<const float2*>(edge + t * 4); l2 = e.x; l3 = e.y; }
    if (lane == 31) { const float2 e = *reinterpret_cast<const float2*>(edge + t * 4 + 2); q0 = e.x; q1 = e.y; }
    const float pb = fmaxf(v[0], v[1]), pc = fmaxf(v[2], v[3]);
    float rm[4];
    rm[0] = max3(fmaxf(l2, l3), pb, v[2]);
    rm[1] = max3(l3, pb, pc);
    rm[2] = max3(pb, pc, q0);
    rm[3] = max3(v[1], pc, fmaxf(q0, q1));
    const int yc = y - 2;
    if (t >= 4 && yc < H) {   // uniform over the CTA
      const float m0 = max3(max3(r0[0], r1[0], r2[0]), r3[0], rm[0]);
      const float m1 = max3(max3(r0[1], r1[1], r2[1]), r3[1], rm[1]);
      const float m2 = max3(max3(r0[2], r1[2], r2[2]), r3[2], rm[2]);
      const float m3 = max3(max3(r0[3], r1[3], r2[3]), r3[3], rm[3]);
      const bool k0 = (m0 == vq0[0]), k1 = (m1 == vq0[1]), k2 = (m2 == vq0[2]), k3 = (m3 == vq0[3]);
      // NMS'd value of a suppressed pixel is +-0; its sign cannot change any comparison made on the word maximum
      float wm4 = fmaxf(fmaxf(k0 ? vq0[0] : 0.f, k1 ? vq0[1] : 0.f), fmaxf(k2 ? vq0[2] : 0.f, k3 ? vq0[3] : 0.f));
      float hm4 = fmaxf(fmaxf(vq0[0], vq0[1]), fmaxf(vq0[2], vq0[3]));
      unsigned bits = ((k0 ? 1u : 0u) | (k1 ? 2u : 0u) | (k2 ? 4u : 0u) | (k3 ? 8u : 0u)) << shl;
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        bits |= __shfl_xor_sync(kFull, bits, o);
        hm4 = fmaxf(hm4, __shfl_xor_sync(kFull, hm4, o));
        wm4 = fmaxf(wm4, __shfl_xor_sync(kFull, wm4, o));
      }
      if (word_writer) {
        const size_t w = wbase + (size_t)yc * a.wpr;
        a.mask[w] = bits;
        a.wmax[w] = wm4;
        a.hmax[w] = hm4;
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      r0[c] = r1[c]; r1[c] = r2[c]; r2[c] = r3[c]; r3[c] = rm[c];
      vq0[c] = vq1[c]; vq1[c] = v[c];
    }
  }
};

// Tag bounds of one band: per (4 rows x 32 columns) the range of the first tag component's quarter-res
// sources (tag_bmin / tag_bmax, the refine prefilter).  Every tag of an output pixel is an x4 bilinear
// combination (results.py:229-230) of the 3 x 3 quarter-res tags around it, so it lies in that range.  sT is
// the staged tile of the first component ([TR][tc], origin column txo, tile row r = quarter-res row
// y0/4 - 1 + r); the lane covers output columns X0..X0+3 and the RB rows from y0.  Called by the lanes
// whose columns are inside the image (W % 32 == 0: whole 8-lane word groups).
template <int RB, int TR>
__device__ __forceinline__ void tag_bounds_x4_band(const AggArgs& a, const float* __restrict__ sT, int tc, int txo,
                                                   int X0, int y0, int b, int k, int lane) {
  const int H = a.H;
  const int tb = (X0 >> 2) - 1 - txo;          // index of T[q-1] in a tile row, q = this lane's quarter-res column
  auto range = [&](int r, float& mn, float& mx) {
    const float* t = sT + r * tc + tb;
    const float t0 = t[0], t1 = t[1], t2 = t[2];
    mn = fminf(fminf(t0, t1), t2); mx = fmaxf(fmaxf(t0, t1), t2);
  };
  const unsigned amask = __activemask();      // W % 32 == 0: whole 8-lane word groups are active
  float mnA, mxA, mnB, mxB, mnC, mxC;
  range(0, mnA, mxA);
  range(1, mnB, mxB);
  const int HB = (H + 3) >> 2;
  const size_t bbase = (((size_t)b * a.K + k) * HB + (y0 >> 2)) * a.wpr + (X0 >> 5);
#pragma unroll 1
  for (int g = 0; g < RB / 4; ++g) {
    range(g + 2, mnC, mxC);
    // band of rows y0+4g .. y0+4g+3 reads tile rows g, g+1, g+2: bounds over the 8 lanes of the word
    if (y0 + 4 * g < H) {
      float mn = fminf(fminf(mnA, mnB), mnC), mx = fmaxf(fmaxf(mxA, mxB), mxC);
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        mn = fminf(mn, __shfl_xor_sync(amask, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(amask, mx, o));
      }
      if ((lane & 7) == 0) {
        a.tmin[bbase + (size_t)g * a.wpr] = mn;
        a.tmax[bbase + (size_t)g * a.wpr] = mx;
      }
    }
    mnA = mnB; mxA = mxB; mnB = mnC; mxB = mxC;
  }
}

template <int NW, typename T>
__global__ void __launch_bounds__(32 * NW) agg_nms_x2_kernel(const AggArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int sc = 64 * NW + 8, lc = 32 * NW + 8, tc = 32 * NW + 8;
  float* sS = smem;                              // [SR][sc]   hi average, then stage mean S
  float* sL = sS + SR * sc;                      // [LR][lc]   flip-averaged hm_lo
  float* sT = smem;                              // [TR][tc]   first tag component -- aliases sS, read (phase 0) before sS is staged
  float* sEdge = sL + LR * lc;                   // [NW][NROWS][4] halo-column values per warp
  int* sRowI0 = (int*)(sEdge + NW * NROWS * 4);  // [SR] phase-2 vertical taps (rows of sL)
  int* sRowI1 = sRowI0 + SR;
  float* sRowW0 = (float*)(sRowI1 + SR);
  float* sRowW1 = sRowW0 + SR;
  float* sNegInf = sRowW1 + SR;                  // [8] dummy row for lanes right of the image

  const ScaleDev& S = a.sc[0];
  const int tid = threadIdx.x;
  constexpr int nthr = 32 * NW;
  const int warp = tid >> 5, lane = tid & 31;
  const int bk = blockIdx.z, b = bk / a.K, k = bk % a.K, kf = a.flip[k];
  const int H = a.H, W = a.W;
  const int x0 = blockIdx.x * 128 * NW, y0 = blockIdx.y * RB;
  const int hxo = x0 / 2 - 4, hyo = y0 / 2 - 2;     // origins of the half-res tile
  const int lxo = x0 / 4 - 4, lyo = y0 / 4 - 2;     // origins of the quarter-res hm tile
  const int txo = x0 / 4 - 4, tyo = y0 / 4 - 1;     // origins of the tag tile

  const int xw = x0 + 128 * warp;                 // first column of this warp's strip
  const int X0 = xw + 4 * lane;                   // this lane's 4 output columns
  const bool active = X0 < W;

  // ---------------- phase 0a: stage the first tag component (aliases the half-res tile) -------------
  {
    const T* tg0 = reinterpret_cast<const T*>(a.tag) + (size_t)b * a.tag_sb + (size_t)k * a.tag_sc;
    if (a.in_vec_ok) stage_tile<false, TR, tc, NW, true>(sT, tg0, (const T*)nullptr, tyo, txo, a.th, a.tw, warp, lane);
    else stage_tile<false, TR, tc, NW, false>(sT, tg0, (const T*)nullptr, tyo, txo, a.th, a.tw, warp, lane);
  }
  __syncthreads();
  // ---------------- phase 0b: tag bounds (refine prefilter) ------------------------------------------
  if (active) tag_bounds_x4_band<RB, TR>(a, sT, tc, txo, X0, y0, b, k, lane);
  __syncthreads();   // every warp is done with the tag tile before the half-res tile overwrites it

  // ---------------- phase 1: stage the heatmap inputs -------------------------------------------------
  {
    const T* lo = reinterpret_cast<const T*>(S.lo) + (size_t)b * S.lo_sb + (size_t)k * S.lo_sc;
    const T* hi = reinterpret_cast<const T*>(S.hi) + (size_t)b * S.hi_sb + (size_t)k * S.hi_sc;
    const T* lof = S.lo_f ? reinterpret_cast<const T*>(S.lo_f) + (size_t)b * S.lof_sb + (size_t)kf * S.lof_sc : nullptr;
    const T* hif = S.hi_f ? reinterpret_cast<const T*>(S.hi_f) + (size_t)b * S.hif_sb + (size_t)kf * S.hif_sc : nullptr;
#define HPD_STAGE_ALL(VEC_)                                                                                    \
  do {                                                                                                         \
    if (lof) {                                                                                                 \
      stage_tile<true, LR, lc, NW, VEC_>(sL, lo, lof, lyo, lxo, S.lh, S.lw, warp, lane);                       \
      stage_tile<true, SR, sc, NW, VEC_>(sS, hi, hif, hyo, hxo, S.hh, S.hw, warp, lane);                       \
    } else {                                                                                                   \
      stage_tile<false, LR, lc, NW, VEC_>(sL, lo, (const T*)nullptr, lyo, lxo, S.lh, S.lw, warp, lane);        \
      stage_tile<false, SR, sc, NW, VEC_>(sS, hi, (const T*)nullptr, hyo, hxo, S.hh, S.hw, warp, lane);        \
    }                                                                                                          \
  } while (0)
    if (a.in_vec_ok) HPD_STAGE_ALL(true); else HPD_STAGE_ALL(false);
#undef HPD_STAGE_ALL
  }
  if (tid < 8) sNegInf[tid] = -INFINITY;
  if (tid < SR) {   // vertical taps of phase 2: half-res row -> rows of sL
    int i0, i1; float w0, w1;
    tap_x2(clampi(hyo + tid, 0, S.hh - 1), S.lh, i0, i1, w0, w1);
    sRowI0[tid] = i0 - lyo; sRowI1[tid] = i1 - lyo; sRowW0[tid] = w0; sRowW1[tid] = w1;
  }
  __syncthreads();

  // ---------------- phase 2: S = (up2(lo) + hi) * 0.5 in place (results.py:225-226) -------------
  // Bands that touch neither the first nor the last rows of the image need no clamping, so the row
  // taps are compile-time: the quarter-res rows are interpolated horizontally once per column
  // (registers) and combined vertically; the two border bands take the table-driven path.
  const bool interior_band = (y0 >= RB) && (y0 + 2 * RB <= H);
  for (int c = tid; c < sc; c += nthr) {
    int c0, c1; float wx0, wx1;
    tap_x2(clampi(hxo + c, 0, S.hw - 1), S.lw, c0, c1, wx0, wx1);
    c0 -= lxo; c1 -= lxo;
    if (interior_band) {
      float hq[LR];
#pragma unroll
      for (int i = 0; i < LR; ++i) hq[i] = fmaf(wx0, sL[i * lc + c0], __fmul_rn(wx1, sL[i * lc + c1]));
#pragma unroll
      for (int r = 0; r < SR; ++r) {
        // half-res row hyo + r (hyo even): even -> quarter rows (k-1, k) = tile rows (r/2, r/2+1), weights (.25,.75);
        // odd -> (k, k+1) = tile rows ((r-1)/2+1, (r-1)/2+2), weights (.75,.25)
        const int i0 = (r & 1) ? (r >> 1) + 1 : (r >> 1);
        const float up = (r & 1) ? fmaf(0.75f, hq[i0], __fmul_rn(0.25f, hq[i0 + 1]))
                                 : fmaf(0.25f, hq[i0], __fmul_rn(0.75f, hq[i0 + 1]));
        sS[r * sc + c] = __fmul_rn(__fadd_rn(up, sS[r * sc + c]), 0.5f);
      }
    } else {
#pragma unroll 4
      for (int r = 0; r < SR; ++r) {
        const float* r0 = sL + sRowI0[r] * lc;
        const float* r1 = sL + sRowI1[r] * lc;
        const float up = lerp2(wx0, wx1, sRowW0[r], sRowW1[r], r0[c0], r0[c1], r1[c0], r1[c1]);
        sS[r * sc + c] = __fmul_rn(__fadd_rn(up, sS[r * sc + c]), 0.5f);
      }
    }
  }
  __syncthreads();

  // ---------------- phase 3a: per-warp prologue, values of the 4 halo columns ------------------
  const int ys = y0 - 2;                          // first walked row (even)
  float* edge = sEdge + warp * NROWS * 4;
  // 4 columns x NROWS rows = 144 independent values, spread over all 32 lanes (value i = lane + 32u:
  // row t = i / 4, column e = i % 4); each is the same two-step lerp the walk performs.
#pragma unroll
  for (int u = 0; u < (NROWS * 4 + 31) / 32; ++u) {
    const int i = lane + 32 * u;
    if (i < NROWS * 4) {
      const int t = i >> 2, e = i & 3;
      const int xe = (e < 2) ? xw - 2 + e : xw + 126 + e;            // xw-2, xw-1, xw+128, xw+129
      const int y = ys + t;
      float v = -INFINITY;
      if (xe >= 0 && xe < W && y >= 0 && y < H) {
        // xe >= 126 whenever it is inside the image, so no first-column special case here
        const int h = xe >> 1;
        const int ca = ((xe & 1) ? h : h - 1) - hxo;
        const float wa = (xe & 1) ? 0.75f : 0.25f, wb = (xe & 1) ? 0.25f : 0.75f;
        // rows of the half-res tile: even y = 2j -> (j-1, j) = (t/2, t/2+1); odd -> (j, j+1) = ((t-1)/2+1, +2);
        // the first image row clamps to (row 0, row 1) with weights (1, 0)
        const bool odd = t & 1, first = (y == 0);
        const int ra = (odd || first) ? (t >> 1) + 1 : (t >> 1);
        const float wya = first ? 1.f : (odd ? 0.75f : 0.25f), wyb = first ? 0.f : (odd ? 0.25f : 0.75f);
        const float* s0 = sS + ra * sc + ca;
        const float ha = fmaf(wa, s0[0], __fmul_rn(wb, s0[1]));
        const float hb = fmaf(wa, s0[sc], __fmul_rn(wb, s0[sc + 1]));
        v = fmaf(wya, ha, __fmul_rn(wyb, hb));
      }
      edge[i] = v;
    }
  }
  __syncwarp();

  // ---------------- phase 3b: walk the rows, 4 columns per lane ------------------------------------
  // Four rows per loop iteration so that the register windows (4 row-maxima rows, 2 value rows,
  // 2 interpolated half-res rows) rotate by renaming instead of by moves.
  {
    const bool x_first = (X0 == 0);
    const float wa0 = x_first ? 1.f : 0.25f, wb0 = x_first ? 0.f : 0.75f;
    const float NINF = -INFINITY;
    // lanes right of the image read a dummy row of -inf (stride 0), which makes all their values -inf
    const float* srow = active ? (sS + 64 * warp + 2 * lane + 3) : sNegInf + 1;   // &S[h0-1]
    const int sstride = active ? sc : 0;
    auto hpass = [&](int r, float (&h)[4]) {
      const float* sp = srow + r * sstride;
      const float2 mid = *reinterpret_cast<const float2*>(sp + 1);      // S[h0], S[h0+1] (8-byte aligned)
      const float2 p = make_float2(sp[0], mid.x);
      const float2 q = make_float2(mid.y, sp[3]);
      const float a0 = x_first ? p.y : p.x, b0 = x_first ? q.x : p.y;
      h[0] = fmaf(wa0, a0, __fmul_rn(wb0, b0));
      h[1] = fmaf(0.75f, p.y, __fmul_rn(0.25f, q.x));
      h[2] = fmaf(0.25f, p.y, __fmul_rn(0.75f, q.x));
      h[3] = fmaf(0.75f, q.x, __fmul_rn(0.25f, q.y));
    };
    float hA[4], hB[4], hC[4], hD[4];
    hpass(0, hA);
    hpass(1, hB);
    NmsColumnWalk<RB> nms;
    nms.init(a, b, k, X0, ys, edge, active, lane);
    auto process_row = [&](int t, const float (&v)[4]) { nms.row(a, t, v); };

#pragma unroll 1
    for (int it = 0; it < NROWS / 4; ++it) {
      const int t = 4 * it, y = ys + t;            // y = 2 (mod 4); half-res rows j-1..j+2 = tile rows 2it..2it+3
      hpass(2 * it + 2, hC);
      hpass(2 * it + 3, hD);
      float v[4];
      // row y (even): taps (hA, hB)
      if (y >= 0 && y < H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(0.25f, hA[c], __fmul_rn(0.75f, hB[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      process_row(t, v);
      // row y+1 (odd): taps (hB, hC)
      if (y + 1 >= 0 && y + 1 < H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(0.75f, hB[c], __fmul_rn(0.25f, hC[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      process_row(t + 1, v);
      // row y+2 (even): taps (hB, hC); the first image row clamps to (row 0, row 1) with weights (1, 0)
      if (y + 2 < H) {
        if (y + 2 == 0) {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = fmaf(1.f, hC[c], __fmul_rn(0.f, hD[c]));
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = fmaf(0.25f, hB[c], __fmul_rn(0.75f, hC[c]));
        }
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      process_row(t + 2, v);
      // row y+3 (odd): taps (hC, hD)
      if (y + 3 < H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(0.75f, hC[c], __fmul_rn(0.25f, hD[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      process_row(t + 3, v);
#pragma unroll
      for (int c = 0; c < 4; ++c) { hA[c] = hC[c]; hB[c] = hD[c]; }
    }
  }

}

}  // namespace x2
