// Specialised fused aggregation + NMS kernel for single-stage heads (HRNet with the associative-embedding head
// and no deconvolution): heatmaps and tags at 1/4 resolution, output at full resolution
//   (hm --x4--> out ; tag --x4--> out).
// Included by aggregate_nms.cu after aggregate_nms_x2.cuh, whose device functions it shares: the tile staging,
// the tag bounds and the NMS column walk.  Bit-identical to the generic kernel: for an exact x4 ratio axis_tap()
// gives output column 4q + j the taps (q-1, q) with weights (0.375, 0.625) / (0.125, 0.875) for j = 0 / 1 and
// (q, q+1) with (0.875, 0.125) / (0.625, 0.375) for j = 2 / 3 -- all exact in f32 -- except that columns (rows)
// 0 and 1 clamp to (0, 1) with (1, 0); past the last column the staged tile replicates the border, which is the
// generic kernel's i1 == i0 clamp.
//
//   * one CTA = a band of RB output rows x (128 * NW) columns of one (image, joint) plane, as in the x2 kernel;
//   * phase 0 (tag bounds): as in the x2 kernel; the tag tile aliases the heatmap tile;
//   * phase 1: flip-averaged quarter-res tile -> smem (there is no half-res stage and no stage mean: the mean of
//     one stage is the stage itself);
//   * phase 2 (per warp, no CTA barrier): every lane owns 4 adjacent output columns, i.e. one quarter-res column
//     q, and walks down the rows: each quarter-res row is interpolated horizontally once (taps q-1, q, q+1), two
//     such rows give the four output rows 4r+2 .. 4r+5, which go through x2::NmsColumnWalk.
#pragma once

namespace x4 {

using x2::LR;
using x2::NROWS;
using x2::RB;
using x2::TR;

__host__ __device__ inline size_t smem_floats(int NW) {
  // the tag tile (TR rows) aliases the heatmap tile (LR rows), both 32 * NW + 8 columns wide
  return (size_t)LR * (32 * NW + 8) + (size_t)NW * NROWS * 4 + 8;
}

template <int NW, typename T>
__global__ void __launch_bounds__(32 * NW) agg_nms_x4_kernel(const AggArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int lc = 32 * NW + 8;
  float* sL = smem;                              // [LR][lc]   flip-averaged heatmap, tile row i = quarter-res row lyo + i
  float* sT = smem;                              // [TR][lc]   first tag component -- aliases sL, read (phase 0) before sL is staged
  float* sEdge = sL + LR * lc;                   // [NW][NROWS][4] halo-column values per warp
  float* sNegInf = sEdge + NW * NROWS * 4;       // [8] dummy row for lanes right of the image

  const ScaleDev& S = a.sc[0];   // one stage: lo and hi are the same map
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int bk = blockIdx.z, b = bk / a.K, k = bk % a.K, kf = a.flip[k];
  const int H = a.H, W = a.W;
  const int x0 = blockIdx.x * 128 * NW, y0 = blockIdx.y * RB;
  const int lxo = x0 / 4 - 4, lyo = y0 / 4 - 2;     // origin of the heatmap tile
  const int txo = x0 / 4 - 4, tyo = y0 / 4 - 1;     // origin of the tag tile

  const int xw = x0 + 128 * warp;                 // first column of this warp's strip
  const int X0 = xw + 4 * lane;                   // this lane's 4 output columns
  const bool active = X0 < W;

  // ---------------- phase 0: tag bounds (refine prefilter), as in the x2 kernel ------------------------
  {
    const T* tg0 = reinterpret_cast<const T*>(a.tag) + (size_t)b * a.tag_sb + (size_t)k * a.tag_sc;
    if (a.in_vec_ok) x2::stage_tile<false, TR, lc, NW, true>(sT, tg0, (const T*)nullptr, tyo, txo, a.th, a.tw, warp, lane);
    else x2::stage_tile<false, TR, lc, NW, false>(sT, tg0, (const T*)nullptr, tyo, txo, a.th, a.tw, warp, lane);
  }
  __syncthreads();
  if (active) x2::tag_bounds_x4_band<RB, TR>(a, sT, lc, txo, X0, y0, b, k, lane);
  __syncthreads();   // every warp is done with the tag tile before the heatmap tile overwrites it

  // ---------------- phase 1: the flip-averaged heatmap tile ---------------------------------------------
  {
    const T* hm = reinterpret_cast<const T*>(S.hi) + (size_t)b * S.hi_sb + (size_t)k * S.hi_sc;
    const T* hmf = S.hi_f ? reinterpret_cast<const T*>(S.hi_f) + (size_t)b * S.hif_sb + (size_t)kf * S.hif_sc : nullptr;
    if (a.in_vec_ok) {
      if (hmf) x2::stage_tile<true, LR, lc, NW, true>(sL, hm, hmf, lyo, lxo, S.hh, S.hw, warp, lane);
      else x2::stage_tile<false, LR, lc, NW, true>(sL, hm, (const T*)nullptr, lyo, lxo, S.hh, S.hw, warp, lane);
    } else {
      if (hmf) x2::stage_tile<true, LR, lc, NW, false>(sL, hm, hmf, lyo, lxo, S.hh, S.hw, warp, lane);
      else x2::stage_tile<false, LR, lc, NW, false>(sL, hm, (const T*)nullptr, lyo, lxo, S.hh, S.hw, warp, lane);
    }
  }
  if (tid < 8) sNegInf[tid] = -INFINITY;
  __syncthreads();

  // ---------------- phase 2a: per-warp prologue, values of the 4 halo columns --------------------------
  const int ys = y0 - 2;                          // first walked row (y0 - 2 = 2 mod 4)
  float* edge = sEdge + warp * NROWS * 4;
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
        const int jx = xe & 3, ca = ((jx < 2) ? (xe >> 2) - 1 : (xe >> 2)) - lxo;
        const float wa = jx == 0 ? 0.375f : (jx == 1 ? 0.125f : (jx == 2 ? 0.875f : 0.625f));
        const float wb = jx == 0 ? 0.625f : (jx == 1 ? 0.875f : (jx == 2 ? 0.125f : 0.375f));
        const int jy = y & 3;
        const bool first = y < 2;                 // rows 0 and 1 clamp to (row 0, row 1) with weights (1, 0)
        const int ra = (first ? 0 : ((jy < 2) ? (y >> 2) - 1 : (y >> 2))) - lyo;
        const float wya = first ? 1.f : (jy == 0 ? 0.375f : (jy == 1 ? 0.125f : (jy == 2 ? 0.875f : 0.625f)));
        const float wyb = first ? 0.f : (jy == 0 ? 0.625f : (jy == 1 ? 0.875f : (jy == 2 ? 0.125f : 0.375f)));
        const float* s0 = sL + ra * lc + ca;
        const float ha = fmaf(wa, s0[0], __fmul_rn(wb, s0[1]));
        const float hb = fmaf(wa, s0[lc], __fmul_rn(wb, s0[lc + 1]));
        v = fmaf(wya, ha, __fmul_rn(wyb, hb));
      }
      edge[i] = v;
    }
  }
  __syncwarp();

  // ---------------- phase 2b: walk the rows, 4 columns per lane -------------------------------------------
  {
    const bool x_first = (X0 == 0);
    const float NINF = -INFINITY;
    // lanes right of the image read a dummy row of -inf (stride 0), which makes all their values -inf
    const float* srow = active ? (sL + 32 * warp + lane + 3) : sNegInf + 1;   // &T[q-1]
    const int sstride = active ? lc : 0;
    // horizontal x4 pass of tile row r: the lane's 4 output columns from T[q-1], T[q], T[q+1]
    auto hpass = [&](int r, float (&h)[4]) {
      const float* sp = srow + r * sstride;
      const float tm = sp[0], t0 = sp[1], tp = sp[2];
      if (x_first) {   // columns 0 and 1: taps (0, 1) with weights (1, 0)
        h[0] = fmaf(1.f, t0, __fmul_rn(0.f, tp));
        h[1] = h[0];
      } else {
        h[0] = fmaf(0.375f, tm, __fmul_rn(0.625f, t0));
        h[1] = fmaf(0.125f, tm, __fmul_rn(0.875f, t0));
      }
      h[2] = fmaf(0.875f, t0, __fmul_rn(0.125f, tp));
      h[3] = fmaf(0.625f, t0, __fmul_rn(0.375f, tp));
    };
    x2::NmsColumnWalk<RB> nms;
    nms.init(a, b, k, X0, ys, edge, active, lane);
    float hA[4], hB[4];
    hpass(1, hA);                                 // quarter-res row y0/4 - 1
#pragma unroll 1
    for (int it = 0; it < NROWS / 4; ++it) {
      // rows y .. y+3 (y = 2 mod 4) all interpolate between quarter-res rows r = (y-2)/4 (hA) and r+1 (hB)
      const int t = 4 * it, y = ys + t;
      hpass(it + 2, hB);
      float v[4];
      // row y (4r+2): (0.875, 0.125)
      if (y >= 0 && y < H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(0.875f, hA[c], __fmul_rn(0.125f, hB[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      nms.row(a, t, v);
      // row y+1 (4r+3): (0.625, 0.375)
      if (y + 1 >= 0 && y + 1 < H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(0.625f, hA[c], __fmul_rn(0.375f, hB[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
      nms.row(a, t + 1, v);
      if (y + 2 == 0) {
        // rows 0 and 1 of the image: quarter-res rows (0, 1) = (hB, next row) with weights (1, 0)
        float hC[4];
        hpass(it + 3, hC);
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = fmaf(1.f, hB[c], __fmul_rn(0.f, hC[c]));
        nms.row(a, t + 2, v);
        nms.row(a, t + 3, v);
      } else {
        // row y+2 (4(r+1)+0): (0.375, 0.625)
        if (y + 2 < H) {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = fmaf(0.375f, hA[c], __fmul_rn(0.625f, hB[c]));
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = NINF;
        }
        nms.row(a, t + 2, v);
        // row y+3 (4(r+1)+1): (0.125, 0.875)
        if (y + 3 < H) {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = fmaf(0.125f, hA[c], __fmul_rn(0.875f, hB[c]));
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = NINF;
        }
        nms.row(a, t + 3, v);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) hA[c] = hB[c];
    }
  }
}

}  // namespace x4
