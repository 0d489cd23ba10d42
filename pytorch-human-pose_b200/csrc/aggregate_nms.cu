// Stage (a)+(b): fused flip/scale aggregation of the network outputs into full-resolution
// heatmaps, with the 5x5 max-pool NMS evaluated on the same tile while it is still in shared memory.
//
// Reference semantics reproduced bit-exactly (paths relative to /root/reference):
//   model.py:85-96       per stage (pred + flipW(flip_pred)[:, FLIP]) / 2 ; tags kept separate (E = 2)
//   results.py:225       hm_lo --bilinear--> hm_hi size          (F.interpolate, align_corners=False)
//   results.py:226       stage mean, rounded to f32
//   results.py:227       --bilinear--> (H, W)
//   results.py:229-230   every tag map --bilinear--> (H, W), stacked with E innermost
//   grouping.py:80-83    keep = (maxpool5x5(x) == x)   (-inf padding)
// plus, for num_scales > 1, torch.stack(per_scale).mean(0) (sequential sum, true division).
//
// The NMS'd map itself is never written.  Per 32-pixel word of each image row the kernel emits
// the survivor bit mask, the maximum NMS'd value (top-k prefilter) and the maximum raw value
// (refine prefilter); together 3/32 of one map.
//
// The full-resolution tag map (results.py:229-230) has one producer, aggregate_tags_kernel (tag_at per
// pixel).  The decode does not need it: the tag stages interpolate the few tags they read.  When a caller
// asks for the map, launch_aggregate_nms runs that kernel after the aggregation kernel.
//
// This file holds the GENERIC kernel (any resize ratios, any number of scales).  It is the
// correctness anchor; aggregate_nms_x2.cuh specialises the standard single-scale x2/x2/x4 case and
// aggregate_nms_ms.cuh the multi-scale one.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#ifdef HPD_MS_PROFILE
#include <cstdio>
#endif

namespace hpd {

constexpr int TW = 64, TH = 32, HALO = 2;
constexpr int OT_R = TH + 2 * HALO, OT_C = TW + 2 * HALO;
constexpr int kAggThreads = 256;

struct ScaleDev {
  const float *lo, *hi, *lo_f, *hi_f;   // first and last heatmap stage (the same map for a single-stage head)
  long long lo_sb, lo_sc, hi_sb, hi_sc, lof_sb, lof_sc, hif_sb, hif_sc;
  int lh, lw, hh, hw;
  float s_lo_y, s_lo_x;  // lo -> hi   ( (float)lh / hh )
  float s_hi_y, s_hi_x;  // hi -> out
};

// One heatmap stage of one scale (the un-flipped and, with the flip test, the flipped-run map) as the generic kernel
// reads it.
struct StageDev {
  const float *p, *pf;
  long long sb, sc, fsb, fsc;
  int h, w;
  float s_y, s_x;        // this stage -> the last stage
};

struct AggArgs {
  ScaleDev sc[HPD_MAX_SCALES];
  int n_scales;
  const float* tag;   // tag-scale map, first component (the tag bounds)
  long long tag_sb, tag_sc;
  int th, tw;
  int B, K, H, W, wpr;
  int flip[HPD_MAX_KPTS];
  float* agg_hm;
  uint32_t* mask;
  float* wmax;
  float* hmax;
  float* tmin;     // [B,K,(H+3)/4,wpr] bounds of tag component 0 per 4 rows x word
  float* tmax;
  float* nms_out;  // standalone NMS only
  int LO_R, LO_C, HI_R, HI_C;
  int vec_ok;
  int in_vec_ok;   // inputs allow 16-byte loads (aligned bases, strides multiples of 4 elements)
  int in_vec_ok_all;   // ... for every scale
  int dtype;       // HPD_F32 / HPD_F16 / HPD_BF16: the const float* input members point at elements of this type
  // Heads with other than two heatmap stages (generic kernel only; the specialised kernels read sc[] alone, whose
  // layout is unchanged): stages per scale, and the stages between the first (sc[].lo) and the last (sc[].hi).
  int n_stages[HPD_MAX_SCALES];
  StageDev mid[HPD_MAX_SCALES][HPD_MAX_STAGES - 2];
};

// Stage i of scale s: sc[s].lo, mid[s][i-1] or sc[s].hi.
__device__ __forceinline__ StageDev stage_of(const AggArgs& a, int s, int i) {
  const ScaleDev& S = a.sc[s];
  if (i == a.n_stages[s] - 1) return StageDev{S.hi, S.hi_f, S.hi_sb, S.hi_sc, S.hif_sb, S.hif_sc, S.hh, S.hw, 1.f, 1.f};
  if (i == 0) return StageDev{S.lo, S.lo_f, S.lo_sb, S.lo_sc, S.lof_sb, S.lof_sc, S.lh, S.lw, S.s_lo_y, S.s_lo_x};
  return a.mid[s][i - 1];
}

// ---------------------------------------------------------------------------------------------
// NMS on a (TH+4)x(TW+4) tile already in shared memory (pixels outside the image hold -inf).
// rowM is scratch [OT_R][TW].  Plane pointers are already offset to this (image, joint).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void nms_tile(const float* __restrict__ outT, float* __restrict__ rowM, int x0, int y0,
                                         int H, int W, int wpr, uint32_t* __restrict__ mask,
                                         float* __restrict__ wmax, float* __restrict__ hmax,
                                         float* __restrict__ tmin, float* __restrict__ tmax,
                                         float* __restrict__ nms_out) {
  const int tid = threadIdx.x;
  for (int i = tid; i < OT_R * TW; i += kAggThreads) {
    const int r = i / TW, c = i % TW;
    const float* p = outT + r * OT_C + c;
    rowM[i] = fmaxf(fmaxf(fmaxf(p[0], p[1]), fmaxf(p[2], p[3])), p[4]);
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  constexpr int kWarps = kAggThreads / 32;
  for (int r = warp; r < TH; r += kWarps) {
    const int y = y0 + r;
    if (y >= H) break;
#pragma unroll
    for (int half = 0; half < TW / 32; ++half) {
      const int c = half * 32 + lane;
      const int x = x0 + c;
      if (x0 + half * 32 >= W) break;
      const float* q = rowM + r * TW + c;
      const float m = fmaxf(fmaxf(fmaxf(q[0], q[TW]), fmaxf(q[2 * TW], q[3 * TW])), q[4 * TW]);
      const float v = outT[(r + HALO) * OT_C + c + HALO];
      const bool inside = x < W;
      const bool keep = inside && (m == v);
      const float nv = keep ? v : __fmul_rn(v, 0.0f);
      const uint32_t bits = __ballot_sync(kFull, keep);
      const float ninf = -INFINITY;
      // word maximum of the NMS'd values; a suppressed pixel contributes +0 (the sign of its x*0 is
      // irrelevant to every comparison made on the word maximum)
      const float wm = warp_max_float(inside ? (keep ? v : 0.0f) : ninf);
      const float hm = warp_max_float(inside ? v : ninf);
      if (lane == 0) {
        const size_t w = (size_t)y * wpr + (x0 >> 5) + half;
        mask[w] = bits;
        wmax[w] = wm;
        hmax[w] = hm;
        if (tmin != nullptr && (y & 3) == 0) {   // this kernel derives no tag bound: "anything"
          const size_t wb = (size_t)(y >> 2) * wpr + (x0 >> 5) + half;
          tmin[wb] = -INFINITY;
          tmax[wb] = INFINITY;
        }
      }
      if (nms_out != nullptr && inside) nms_out[(size_t)y * W + x] = nv;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// generic fused kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAggThreads) agg_nms_generic_kernel(const AggArgs a) {
  extern __shared__ float smem[];
  float* outT = smem;                         // [OT_R][OT_C]
  float* rowM = outT + OT_R * OT_C;           // [OT_R][TW]
  float* hiT = rowM + OT_R * TW;              // [HI_R][HI_C]
  float* loT = hiT + a.HI_R * a.HI_C;         // [LO_R][LO_C]
  // tap tables: index pairs (relative to the source tile origin) and weights
  int* oc_i0 = (int*)(loT + a.LO_R * a.LO_C); // out col -> hi tile col        [OT_C]
  int* oc_i1 = oc_i0 + OT_C;
  float* oc_w0 = (float*)(oc_i1 + OT_C);
  float* oc_w1 = oc_w0 + OT_C;
  int* or_i0 = (int*)(oc_w1 + OT_C);          // out row -> hi tile row        [OT_R]
  int* or_i1 = or_i0 + OT_R;
  float* or_w0 = (float*)(or_i1 + OT_R);
  float* or_w1 = or_w0 + OT_R;
  int* hc_i0 = (int*)(or_w1 + OT_R);          // hi col -> lo tile col         [HI_C]
  int* hc_i1 = hc_i0 + a.HI_C;
  float* hc_w0 = (float*)(hc_i1 + a.HI_C);
  float* hc_w1 = hc_w0 + a.HI_C;
  int* hr_i0 = (int*)(hc_w1 + a.HI_C);        // hi row -> lo tile row         [HI_R]
  int* hr_i1 = hr_i0 + a.HI_R;
  float* hr_w0 = (float*)(hr_i1 + a.HI_R);
  float* hr_w1 = hr_w0 + a.HI_R;

  const int tid = threadIdx.x;
  const int bk = blockIdx.z, b = bk / a.K, k = bk % a.K, kf = a.flip[k];
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const int H = a.H, W = a.W;
  const int oxa = max(x0 - HALO, 0), oxb = min(x0 + TW + HALO, W) - 1;
  const int oya = max(y0 - HALO, 0), oyb = min(y0 + TH + HALO, H) - 1;

  for (int s = 0; s < a.n_scales; ++s) {
    const ScaleDev& S = a.sc[s];
    const int ns = a.n_stages[s];
    const int hxa = axis_tap(S.s_hi_x, oxa, S.hw, W).i0, hxb = axis_tap(S.s_hi_x, oxb, S.hw, W).i1;
    const int hya = axis_tap(S.s_hi_y, oya, S.hh, H).i0, hyb = axis_tap(S.s_hi_y, oyb, S.hh, H).i1;
    const int nhx = hxb - hxa + 1, nhy = hyb - hya + 1;
    const int per = min(nhx, kAggThreads), groups = kAggThreads / per;   // last-stage tile: column-owned passes
    const int rg = tid / per;

    for (int i = tid; i < OT_C; i += kAggThreads) {
      const int ox = x0 - HALO + i;
      if (ox >= 0 && ox < W) {
        const Tap t = axis_tap(S.s_hi_x, ox, S.hw, W);
        oc_i0[i] = t.i0 - hxa; oc_i1[i] = t.i1 - hxa; oc_w0[i] = t.w0; oc_w1[i] = t.w1;
      } else {
        oc_i0[i] = -1;
      }
    }
    for (int i = tid; i < OT_R; i += kAggThreads) {
      const int oy = y0 - HALO + i;
      if (oy >= 0 && oy < H) {
        const Tap t = axis_tap(S.s_hi_y, oy, S.hh, H);
        or_i0[i] = t.i0 - hya; or_i1[i] = t.i1 - hya; or_w0[i] = t.w0; or_w1[i] = t.w1;
      } else {
        or_i0[i] = -1;
      }
    }
    // stages 0..ns-2: flip-averaged tile (model.py:90) resized to the last stage (results.py:46-54) and summed
    // into hiT in stage order (results.py:226: torch.stack(...).mean(0) sums sequentially)
    for (int si = 0; si + 1 < ns; ++si) {
      const StageDev St = stage_of(a, s, si);
      const int lxa = axis_tap(St.s_x, hxa, St.w, S.hw).i0, lxb = axis_tap(St.s_x, hxb, St.w, S.hw).i1;
      const int lya = axis_tap(St.s_y, hya, St.h, S.hh).i0, lyb = axis_tap(St.s_y, hyb, St.h, S.hh).i1;
      const int nlx = lxb - lxa + 1, nly = lyb - lya + 1;
      for (int i = tid; i < nhx; i += kAggThreads) {
        const Tap t = axis_tap(St.s_x, hxa + i, St.w, S.hw);
        hc_i0[i] = t.i0 - lxa; hc_i1[i] = t.i1 - lxa; hc_w0[i] = t.w0; hc_w1[i] = t.w1;
      }
      for (int i = tid; i < nhy; i += kAggThreads) {
        const Tap t = axis_tap(St.s_y, hya + i, St.h, S.hh);
        hr_i0[i] = t.i0 - lya; hr_i1[i] = t.i1 - lya; hr_w0[i] = t.w0; hr_w1[i] = t.w1;
      }
      {
        const size_t po = (size_t)b * St.sb + (size_t)k * St.sc, pfo = (size_t)b * St.fsb + (size_t)kf * St.fsc;
        const int lper = min(nlx, kAggThreads), lgroups = kAggThreads / lper;
        const int lrg = tid / lper;
        if (lrg < lgroups)
          for (int c = tid % lper; c < nlx; c += lper) {
            const int x = lxa + c;
            for (int r = lrg; r < nly; r += lgroups) {
              const int rowo = (lya + r) * St.w;
              float v = in_elem(St.p, po + rowo + x, a.dtype);
              if (St.pf) v = __fmul_rn(__fadd_rn(v, in_elem(St.pf, pfo + rowo + (St.w - 1 - x), a.dtype)), 0.5f);
              loT[r * a.LO_C + c] = v;
            }
          }
      }
      __syncthreads();
      // A thread owns one column (its taps stay in registers) and strides over the rows.
      if (rg < groups)
        for (int c = tid % per; c < nhx; c += per) {
          const int c0 = hc_i0[c], c1 = hc_i1[c];
          const float cw0 = hc_w0[c], cw1 = hc_w1[c];
          for (int r = rg; r < nhy; r += groups) {
            const float* r0 = loT + hr_i0[r] * a.LO_C;
            const float* r1 = loT + hr_i1[r] * a.LO_C;
            const float up = lerp2(cw0, cw1, hr_w0[r], hr_w1[r], r0[c0], r0[c1], r1[c0], r1[c1]);
            hiT[r * a.HI_C + c] = si == 0 ? up : __fadd_rn(hiT[r * a.HI_C + c], up);
          }
        }
      __syncthreads();   // loT and the hc / hr taps are rewritten by the next stage
    }
    // last stage, flip-averaged, ends the sum; the stage mean divides by ns (two stages: exactly today's * 0.5)
    {
      const StageDev St = stage_of(a, s, ns - 1);
      const size_t po = (size_t)b * St.sb + (size_t)k * St.sc, pfo = (size_t)b * St.fsb + (size_t)kf * St.fsc;
      const float nst = (float)ns;
      if (rg < groups)
        for (int c = tid % per; c < nhx; c += per) {
          const int x = hxa + c;
          for (int r = rg; r < nhy; r += groups) {
            const int rowo = (hya + r) * St.w;
            float v = in_elem(St.p, po + rowo + x, a.dtype);
            if (St.pf) v = __fmul_rn(__fadd_rn(v, in_elem(St.pf, pfo + rowo + (St.w - 1 - x), a.dtype)), 0.5f);
            if (ns > 1) v = __fdiv_rn(__fadd_rn(hiT[r * a.HI_C + c], v), nst);
            hiT[r * a.HI_C + c] = v;
          }
        }
    }
    __syncthreads();
    // full-resolution tile with halo (results.py:227); scales accumulate sequentially.  Column-owned too.
    {
      constexpr int kGroups = kAggThreads / OT_C;   // 3 row groups of OT_C threads
      const int c = tid % OT_C, rg = tid / OT_C;
      if (rg < kGroups) {
        const int c0 = oc_i0[c];
        const int c1 = c0 >= 0 ? oc_i1[c] : 0;
        const float cw0 = c0 >= 0 ? oc_w0[c] : 0.f, cw1 = c0 >= 0 ? oc_w1[c] : 0.f;
        const bool last = a.n_scales > 1 && s == a.n_scales - 1;
        const float nsc = (float)a.n_scales;
        for (int r = rg; r < OT_R; r += kGroups) {
          const int ri0 = or_i0[r];
          float v = -INFINITY;
          if (ri0 >= 0 && c0 >= 0) {
            const float* r0 = hiT + ri0 * a.HI_C;
            const float* r1 = hiT + or_i1[r] * a.HI_C;
            v = lerp2(cw0, cw1, or_w0[r], or_w1[r], r0[c0], r0[c1], r1[c0], r1[c1]);
            if (s > 0) v = __fadd_rn(outT[r * OT_C + c], v);
            if (last) v = __fdiv_rn(v, nsc);
          }
          outT[r * OT_C + c] = v;
        }
      }
    }
    __syncthreads();
  }

  // aggregated heatmap tile -> HBM
  {
    float* dst = a.agg_hm + ((size_t)b * a.K + k) * H * W;
    for (int i = tid; i < TH * TW / 4; i += kAggThreads) {
      const int r = i / (TW / 4), c = (i % (TW / 4)) * 4;
      const int y = y0 + r, x = x0 + c;
      if (y >= H || x >= W) continue;
      const float* src = outT + (r + HALO) * OT_C + c + HALO;
      if (a.vec_ok) {
        *reinterpret_cast<float4*>(dst + (size_t)y * W + x) = make_float4(src[0], src[1], src[2], src[3]);
      } else {
        for (int j = 0; j < 4 && x + j < W; ++j) dst[(size_t)y * W + x + j] = src[j];
      }
    }
  }
  // NMS words
  {
    const size_t plane = (size_t)b * a.K + k;
    nms_tile(outT, rowM, x0, y0, H, W, a.wpr, a.mask + plane * H * a.wpr, a.wmax + plane * H * a.wpr,
             a.hmax + plane * H * a.wpr, a.tmin + plane * ((H + 3) / 4) * a.wpr, a.tmax + plane * ((H + 3) / 4) * a.wpr,
             nullptr);
  }
}

}  // namespace hpd
namespace hpd {
#include "aggregate_nms_x2.cuh"
#include "aggregate_nms_x4.cuh"
#include "aggregate_nms_ms.cuh"
}  // namespace hpd
namespace hpd {

// ---------------------------------------------------------------------------------------------
// standalone NMS (grouping.py:80-83) for callers that hand in aggregated maps
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAggThreads) nms_kernel(const float* __restrict__ hm, int K, int H, int W, int wpr,
                                                          uint32_t* mask, float* wmax, float* hmax, float* tmin, float* tmax,
                                                          float* nms_out) {
  __shared__ float outT[OT_R * OT_C];
  __shared__ float rowM[OT_R * TW];
  const int tid = threadIdx.x;
  const size_t plane = blockIdx.z;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const float* src = hm + plane * H * W;
  for (int i = tid; i < OT_R * OT_C; i += kAggThreads) {
    const int r = i / OT_C, c = i % OT_C;
    const int y = y0 - HALO + r, x = x0 - HALO + c;
    outT[i] = (y >= 0 && y < H && x >= 0 && x < W) ? src[(size_t)y * W + x] : -INFINITY;
  }
  __syncthreads();
  nms_tile(outT, rowM, x0, y0, H, W, wpr, mask + plane * H * wpr, wmax + plane * H * wpr, hmax + plane * H * wpr,
           tmin + plane * ((H + 3) / 4) * wpr, tmax + plane * ((H + 3) / 4) * wpr, nms_out ? nms_out + plane * H * W : nullptr);
}

// ---------------------------------------------------------------------------------------------
// standalone bilinear resize (BaseKeypointsResult.match_heatmaps_size / resize_heatmaps[_list],
// results.py:46-67): one thread per 4 output pixels of a row
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) resize_kernel(const float* __restrict__ in, long long in_sb, long long in_sc,
                                                     int C, int ih, int iw, float* __restrict__ out, int oh, int ow,
                                                     float sy, float sx) {
  const int plane = blockIdx.z;
  const int y = blockIdx.y;
  const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (x4 >= ow) return;
  const float* src = in + (size_t)(plane / C) * in_sb + (size_t)(plane % C) * in_sc;
  const Tap ty = axis_tap(sy, y, ih, oh);
  const float* r0 = src + (size_t)ty.i0 * iw;
  const float* r1 = src + (size_t)ty.i1 * iw;
  float* o = out + ((size_t)plane * oh + y) * ow;
  for (int j = 0; j < 4 && x4 + j < ow; ++j) {
    const Tap tx = axis_tap(sx, x4 + j, iw, ow);
    o[x4 + j] = lerp2(tx.w0, tx.w1, ty.w0, ty.w1, r0[tx.i0], r0[tx.i1], r1[tx.i0], r1[tx.i1]);
  }
}

// ---------------------------------------------------------------------------------------------
// the full-resolution tag map alone (hpd_aggregate_tags): one thread per output pixel, E-innermost stores
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) aggregate_tags_kernel(const TagSource s, float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, row = blockIdx.z;
  if (x >= s.W) return;
  float t[HPD_MAX_EMB];
  tag_at(s, row / s.K, row % s.K, y, x, t);
  float* o = out + (((size_t)row * s.H + y) * s.W + x) * s.E;
  for (int e = 0; e < s.E; ++e) o[e] = t[e];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
namespace {

// Largest source-tile extent any output tile needs along one axis of the nested resize lo -> hi -> out:
// out span (tile + halo) -> mid (hi) extent -> inner (lo) extent.
void axis_extents(int out_size, int tile, int halo, int mid_size, float s_mid, int in_size, float s_in, int* mid_ext,
                  int* in_ext) {
  int me = 1, ie = 1;
  for (int o0 = 0; o0 < out_size; o0 += tile) {
    const int oa = o0 - halo < 0 ? 0 : o0 - halo;
    const int ob = (o0 + tile + halo < out_size ? o0 + tile + halo : out_size) - 1;
    const int ma = axis_tap(s_mid, oa, mid_size, out_size).i0, mb = axis_tap(s_mid, ob, mid_size, out_size).i1;
    me = mb - ma + 1 > me ? mb - ma + 1 : me;
    const int ia = axis_tap(s_in, ma, in_size, mid_size).i0, ib = axis_tap(s_in, mb, in_size, mid_size).i1;
    ie = ib - ia + 1 > ie ? ib - ia + 1 : ie;
  }
  *mid_ext = me;
  *in_ext = ie;
}

int check_map(const HpdMap& m, const char* name, bool required) {
  if (m.ptr == nullptr) {
    if (required) { set_error("%s: missing", name); return HPD_EINVAL; }
    return HPD_OK;
  }
  if (m.h <= 0 || m.w <= 0) { set_error("%s: bad size %dx%d", name, m.h, m.w); return HPD_EINVAL; }
  if (m.dtype != HPD_F32 && m.dtype != HPD_F16 && m.dtype != HPD_BF16) { set_error("%s: unsupported dtype code %d", name, m.dtype); return HPD_EINVAL; }
  return HPD_OK;
}

// TagSource over the tag-scale inputs (map = NULL)
int tag_source_from_inputs(const HpdParams* p, const HpdScaleInputs& in, TagSource* s, const char* who) {
  if (in.tag.ptr == nullptr || in.tag.h <= 0 || in.tag.w <= 0 || (in.tag.dtype != HPD_F32 && in.tag.dtype != HPD_F16 &&
                                                                 in.tag.dtype != HPD_BF16)) {
    set_error("%s: the tag map of the tag scale is missing or malformed", who);
    return HPD_EINVAL;
  }
  if ((p->emb == 2) != (in.tag_f.ptr != nullptr)) {
    set_error("%s: emb must be 2 iff the flipped-run tag map is given (got emb=%d)", who, p->emb);
    return HPD_EINVAL;
  }
  if (in.tag_f.ptr && (in.tag_f.h != in.tag.h || in.tag_f.w != in.tag.w || in.tag_f.dtype != in.tag.dtype)) {
    set_error("%s: the flipped-run tag map must have the shape and dtype of the un-flipped one", who);
    return HPD_EINVAL;
  }
  memset(s, 0, sizeof(*s));
  s->tag = (const float*)in.tag.ptr; s->tag_sb = in.tag.stride_b; s->tag_sc = in.tag.stride_c;
  s->tag_f = (const float*)in.tag_f.ptr; s->tagf_sb = in.tag_f.stride_b; s->tagf_sc = in.tag_f.stride_c;
  s->K = p->num_kpts; s->H = p->out_h; s->W = p->out_w; s->E = p->emb;
  s->th = in.tag.h; s->tw = in.tag.w;
  s->s_y = (float)s->th / (float)s->H; s->s_x = (float)s->tw / (float)s->W;   // as launch_aggregate_nms computes them
  s->dtype = in.tag.dtype;
  s->tags_preflipped = p->tags_preflipped;
  for (int k = 0; k < HPD_MAX_KPTS; ++k) s->flip[k] = p->flip_index[k];
  return HPD_OK;
}

}  // namespace

int make_tag_source(const HpdParams* p, const HpdBuffers* buf, TagSource* s, const char* who) {
  if (buf->agg_tags == nullptr) return tag_source_from_inputs(p, buf->tag_inputs, s, who);
  memset(s, 0, sizeof(*s));
  s->map = buf->agg_tags;
  s->K = p->num_kpts; s->H = p->out_h; s->W = p->out_w; s->E = p->emb;
  return HPD_OK;
}

int launch_aggregate_tags(const HpdParams* p, const HpdScaleInputs* scales, float* out, cudaStream_t st) {
  if (!scales || !out) {
    set_error("hpd_aggregate_tags: scales and out are required");
    return HPD_EINVAL;
  }
  TagSource s;
  if (int rc = tag_source_from_inputs(p, scales[p->tag_scale], &s, "hpd_aggregate_tags")) return rc;
  if (p->out_h > 65535) {
    set_error("hpd_aggregate_tags: out_h must be <= 65535");
    return HPD_EINVAL;
  }
  const dim3 grid((p->out_w + 255) / 256, p->out_h, p->batch * p->num_kpts);
  aggregate_tags_kernel<<<grid, 256, 0, st>>>(s, out);
  count_launch();
  return check_launch("aggregate_tags_kernel");
}

namespace {

// Name of stage i of an n-stage scale in error messages: two stages are HigherHRNet's hm_lo / hm_hi.
const char* stage_name(int n, int i) {
  static const char* any[HPD_MAX_STAGES] = {"hm[0]", "hm[1]", "hm[2]", "hm[3]"};
  return n == 2 ? (i == 0 ? "hm_lo" : "hm_hi") : any[i];
}

// The aggregation + NMS kernel alone: agg_hm, the word side arrays and the tag bounds.
int launch_aggregation_kernel(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, cudaStream_t st) {
  if (!scales || !buf->agg_hm || !buf->nms_mask || !buf->nms_wmax || !buf->hm_wmax || !buf->tag_bmin || !buf->tag_bmax) {
    set_error("hpd_aggregate_nms: scales, agg_hm, nms_mask, nms_wmax, hm_wmax, tag_bmin, tag_bmax are required");
    return HPD_EINVAL;
  }
  AggArgs a;
  memset(&a, 0, sizeof(a));
  a.n_scales = p->num_scales;
  a.B = p->batch; a.K = p->num_kpts; a.H = p->out_h; a.W = p->out_w;
  a.wpr = (p->out_w + 31) / 32;
  for (int k = 0; k < HPD_MAX_KPTS; ++k) a.flip[k] = p->flip_index[k];
  const bool flip = scales[0].hm_f[0].ptr != nullptr;
  const int dtype = scales[0].hm[0].dtype;
  a.dtype = dtype;
  const uintptr_t vec_align = dtype == HPD_F32 ? 16 : 8;    // four elements per vector load
  int LO_R = 1, LO_C = 1, HI_R = 1, HI_C = 1;
  for (int s = 0; s < p->num_scales; ++s) {
    const HpdStageInputs& in = scales[s];
    const int ns = in.num_stages;
    if (ns < 1 || ns > HPD_MAX_STAGES) {
      set_error("num_stages must be in [1,%d] (got %d)", HPD_MAX_STAGES, ns);
      return HPD_EINVAL;
    }
    int rc;
    for (int i = 0; i < ns; ++i)
      if ((rc = check_map(in.hm[i], stage_name(ns, i), true))) return rc;
    for (int i = 0; i < ns + 2; ++i) {
      const HpdMap* pair[2] = {i < ns ? &in.hm[i] : (i == ns ? &in.tag : &in.tag_f),
                               i < ns ? &in.hm_f[i] : (i == ns ? &in.tag : &in.tag_f)};
      for (const HpdMap* m : pair)
        if (m->ptr != nullptr && m->dtype != dtype) {
          set_error("all maps of a call must share one dtype");
          return HPD_EINVAL;
        }
    }
    for (int i = 0; i < ns; ++i)
      if (flip != (in.hm_f[i].ptr != nullptr)) {
        set_error("flip inputs must be given for all stages and scales or for none");
        return HPD_EINVAL;
      }
    for (int i = 0; flip && i < ns; ++i)
      if (in.hm_f[i].h != in.hm[i].h || in.hm_f[i].w != in.hm[i].w) {
        set_error("flipped-run maps must have the shapes of the un-flipped run");
        return HPD_EINVAL;
      }
    ScaleDev& S = a.sc[s];
    const HpdMap &lo = in.hm[0], &hi = in.hm[ns - 1], &lof = in.hm_f[0], &hif = in.hm_f[ns - 1];
    S.lo = (const float*)lo.ptr; S.lo_sb = lo.stride_b; S.lo_sc = lo.stride_c;
    S.hi = (const float*)hi.ptr; S.hi_sb = hi.stride_b; S.hi_sc = hi.stride_c;
    S.lo_f = (const float*)lof.ptr; S.lof_sb = lof.stride_b; S.lof_sc = lof.stride_c;
    S.hi_f = (const float*)hif.ptr; S.hif_sb = hif.stride_b; S.hif_sc = hif.stride_c;
    S.lh = lo.h; S.lw = lo.w; S.hh = hi.h; S.hw = hi.w;
    S.s_lo_y = (float)S.lh / (float)S.hh; S.s_lo_x = (float)S.lw / (float)S.hw;
    S.s_hi_y = (float)S.hh / (float)a.H; S.s_hi_x = (float)S.hw / (float)a.W;
    a.n_stages[s] = ns;
    StageDev st[HPD_MAX_STAGES];
    for (int i = 0; i < ns; ++i) {
      StageDev& D = st[i];
      const HpdMap &m = in.hm[i], &mf = in.hm_f[i];
      D.p = (const float*)m.ptr; D.sb = m.stride_b; D.sc = m.stride_c;
      D.pf = (const float*)mf.ptr; D.fsb = mf.stride_b; D.fsc = mf.stride_c;
      D.h = m.h; D.w = m.w;
      D.s_y = (float)D.h / (float)S.hh; D.s_x = (float)D.w / (float)S.hw;
      if (i > 0 && i < ns - 1) a.mid[s][i - 1] = D;
    }
    for (int i = 0; i < (ns > 1 ? ns - 1 : 1); ++i) {   // one stage: the last-stage extents only
      const StageDev& D = st[i];
      int me, ie;
      axis_extents(a.W, TW, HALO, S.hw, S.s_hi_x, D.w, D.s_x, &me, &ie);
      HI_C = me > HI_C ? me : HI_C;
      if (ns > 1) LO_C = ie > LO_C ? ie : LO_C;
      axis_extents(a.H, TH, HALO, S.hh, S.s_hi_y, D.h, D.s_y, &me, &ie);
      HI_R = me > HI_R ? me : HI_R;
      if (ns > 1) LO_R = ie > LO_R ? ie : LO_R;
    }
  }
  {
    const HpdStageInputs& in = scales[p->tag_scale];
    int rc;
    if ((rc = check_map(in.tag, "tag", true))) return rc;
    if ((p->emb == 2) != (in.tag_f.ptr != nullptr)) {
      set_error("emb must be 2 iff the flipped-run tag map is given (got emb=%d)", p->emb);
      return HPD_EINVAL;
    }
    a.tag = (const float*)in.tag.ptr; a.tag_sb = in.tag.stride_b; a.tag_sc = in.tag.stride_c;
    a.th = in.tag.h; a.tw = in.tag.w;
  }
  a.LO_R = LO_R; a.LO_C = LO_C | 1; a.HI_R = HI_R; a.HI_C = HI_C | 1;
  a.agg_hm = buf->agg_hm; a.mask = buf->nms_mask; a.wmax = buf->nms_wmax;
  a.hmax = buf->hm_wmax;
  a.tmin = buf->tag_bmin;
  a.tmax = buf->tag_bmax;
  {
    auto okp = [vec_align](const float* q, long long sb, long long sc_) { return q == nullptr || ((uintptr_t)q % vec_align == 0 && sb % 4 == 0 && sc_ % 4 == 0); };
    a.in_vec_ok_all = 1;
    for (int s = 0; s < a.n_scales; ++s) {
      const ScaleDev& S = a.sc[s];
      if (!(okp(S.lo, S.lo_sb, S.lo_sc) && okp(S.hi, S.hi_sb, S.hi_sc) && okp(S.lo_f, S.lof_sb, S.lof_sc) && okp(S.hi_f, S.hif_sb, S.hif_sc)))
        a.in_vec_ok_all = 0;
      for (int i = 0; i + 2 < a.n_stages[s]; ++i) {
        const StageDev& D = a.mid[s][i];
        if (!(okp(D.p, D.sb, D.sc) && okp(D.pf, D.fsb, D.fsc))) a.in_vec_ok_all = 0;
      }
    }
  }
  a.vec_ok = (a.W % 4 == 0) && ((uintptr_t)a.agg_hm % 16 == 0);

  // standard single-scale x2/x2/x4 layout -> specialised kernel (aggregate_nms_x2.cuh)
  {
    const ScaleDev& S = a.sc[0];
    auto ok = [vec_align](const float* q, long long sb, long long sc_) { return q == nullptr || ((uintptr_t)q % vec_align == 0 && sb % 4 == 0 && sc_ % 4 == 0); };
    const bool fast = !(p->force_generic & 1) && a.n_scales == 1 && a.n_stages[0] == 2 && S.hh == 2 * S.lh && S.hw == 2 * S.lw &&
                      a.H == 2 * S.hh && a.W == 2 * S.hw && a.th == S.lh && a.tw == S.lw && a.W % 32 == 0 && S.lh >= 2 &&
                      S.lw >= 2 && a.vec_ok;
    // single-stage HRNet-AE layout: heatmaps and tags at S/4 -> x4 walk, no half-res stage
    const bool fast1 = !(p->force_generic & 1) && a.n_scales == 1 && a.n_stages[0] == 1 && a.H == 4 * S.hh && a.W == 4 * S.hw &&
                       a.th == S.hh && a.tw == S.hw && a.W % 32 == 0 && S.hh >= 2 && S.hw >= 2 && a.vec_ok;
    if (fast1) {
      a.in_vec_ok = S.hw % 4 == 0 && ok(S.hi, S.hi_sb, S.hi_sc) && ok(S.hi_f, S.hif_sb, S.hif_sc) && ok(a.tag, a.tag_sb, a.tag_sc);
      const int NW = a.W >= 512 ? 4 : (a.W >= 256 ? 2 : 1);
      const size_t smem = sizeof(float) * x4::smem_floats(NW);
      const dim3 grid((a.W + 128 * NW - 1) / (128 * NW), (a.H + x2::RB - 1) / x2::RB, a.B * a.K);
#define HPD_X4_LAUNCH(NW_, T_)                                                                              \
  do {                                                                                                      \
    if (int rc_ = ensure_dynamic_smem((const void*)x4::agg_nms_x4_kernel<NW_, T_>, smem, "agg_nms_x4_kernel")) return rc_; \
    x4::agg_nms_x4_kernel<NW_, T_><<<grid, 32 * NW_, smem, st>>>(a);                                        \
  } while (0)
#define HPD_X4_LAUNCH_T(NW_)                                                                                \
  do {                                                                                                      \
    if (a.dtype == HPD_F16) HPD_X4_LAUNCH(NW_, __half);                                                     \
    else if (a.dtype == HPD_BF16) HPD_X4_LAUNCH(NW_, __nv_bfloat16);                                        \
    else HPD_X4_LAUNCH(NW_, float);                                                                         \
  } while (0)
      if (NW == 4) HPD_X4_LAUNCH_T(4); else if (NW == 2) HPD_X4_LAUNCH_T(2); else HPD_X4_LAUNCH_T(1);
#undef HPD_X4_LAUNCH_T
#undef HPD_X4_LAUNCH
      count_launch();
      return check_launch("agg_nms_x4_kernel");
    }
    if (fast) {
      a.in_vec_ok = S.lw % 4 == 0 && ok(S.lo, S.lo_sb, S.lo_sc) && ok(S.hi, S.hi_sb, S.hi_sc) && ok(S.lo_f, S.lof_sb, S.lof_sc) &&
                    ok(S.hi_f, S.hif_sb, S.hif_sc) && ok(a.tag, a.tag_sb, a.tag_sc);
      const int NW = a.W >= 512 ? 4 : (a.W >= 256 ? 2 : 1);
      const size_t smem = sizeof(float) * x2::smem_floats(NW);
      const dim3 grid((a.W + 128 * NW - 1) / (128 * NW), (a.H + x2::RB - 1) / x2::RB, a.B * a.K);
#define HPD_X2_LAUNCH(NW_, T_)                                                                              \
  do {                                                                                                      \
    if (int rc_ = ensure_dynamic_smem((const void*)x2::agg_nms_x2_kernel<NW_, T_>, smem, "agg_nms_x2_kernel")) return rc_; \
    x2::agg_nms_x2_kernel<NW_, T_><<<grid, 32 * NW_, smem, st>>>(a);                                        \
  } while (0)
#define HPD_X2_LAUNCH_T(NW_)                                                                                \
  do {                                                                                                      \
    if (a.dtype == HPD_F16) HPD_X2_LAUNCH(NW_, __half);                                                     \
    else if (a.dtype == HPD_BF16) HPD_X2_LAUNCH(NW_, __nv_bfloat16);                                        \
    else HPD_X2_LAUNCH(NW_, float);                                                                         \
  } while (0)
      if (NW == 4) HPD_X2_LAUNCH_T(4); else if (NW == 2) HPD_X2_LAUNCH_T(2); else HPD_X2_LAUNCH_T(1);
#undef HPD_X2_LAUNCH_T
#undef HPD_X2_LAUNCH
      count_launch();
      return check_launch("agg_nms_x2_kernel");
    }
  }
  // several scales and / or other hi -> output ratios with the HigherHRNet structure (lo -> hi exactly x2,
  // tags exactly x4) -> column-walking multi-scale kernel (aggregate_nms_ms.cuh)
  {
    bool ok = !(p->force_generic & 1) && a.n_scales <= 3 && a.in_vec_ok_all && a.th * 4 == a.H && a.tw * 4 == a.W && a.W % 32 == 0 && a.H % 4 == 0 &&
              a.W >= 256 && a.vec_ok;
    for (int s = 0; ok && s < a.n_scales; ++s) {
      const ScaleDev& S = a.sc[s];
      ok = a.n_stages[s] == 2 && S.hh == 2 * S.lh && S.hw == 2 * S.lw && S.lh >= 2 && S.lw >= 4 && S.lw % 4 == 0 && S.hw <= a.W &&
           S.hh <= a.H;
    }
    if (ok) {
      // warps (128-column strips) per CTA: the count in 2..5 that pads the row least, the larger on ties
      // (640 columns: 5 -- one CTA per band with every warp busy; 4 would leave 3 of 8 strips empty)
      int NW = 2;
      for (int c = 3; c <= 5; ++c) {
        const int pad_c = (a.W + 128 * c - 1) / (128 * c) * c, pad_n = (a.W + 128 * NW - 1) / (128 * NW) * NW;
        if (pad_c <= pad_n) NW = c;
      }
      ms::Geom g;
      memset(&g, 0, sizeof(g));
      int off = 0;
      for (int s = 0; s < a.n_scales; ++s) {
        const ScaleDev& S = a.sc[s];
        int hc, lc, hr, lr;
        axis_extents(a.W, 128 * NW, 2, S.hw, S.s_hi_x, S.lw, S.s_lo_x, &hc, &lc);
        axis_extents(a.H, ms::RB, 2, S.hh, S.s_hi_y, S.lh, S.s_lo_y, &hr, &lr);
        g.off_s[s] = off;
        g.hr[s] = hr;
        g.hc[s] = (hc + 6 + 3) & ~3;      // origin rounded down / width rounded up to 4 in the kernel
        off += g.hr[s] * g.hc[s];
        g.lr[s] = lr;
        g.lc[s] = (lc + 6 + 3) & ~3;
      }
      const int tag_words = ms::TR * (32 * NW + 8);
      off = off > tag_words ? off : tag_words;
      off = (off + 3) & ~3;
      for (int s = 0; s < a.n_scales; ++s) {
        g.off_lo[s] = off;
        off += (g.lr[s] * g.lc[s] + 3) & ~3;
      }
      g.off_edge = off; off += NW * ms::NROWS * 4;
      g.off_tab = off;  off += 3 * a.n_scales * ms::NROWS;
      g.total = off;
      const size_t smem = sizeof(float) * (size_t)g.total;
      if (smem <= 200 * 1024) {
        const dim3 grid((a.W + 128 * NW - 1) / (128 * NW), (a.H + ms::RB - 1) / ms::RB, a.B * a.K);
#define HPD_MS_LAUNCH(NW_, NS_, T_)                                                                              \
  do {                                                                                                           \
    if (int rc_ = ensure_dynamic_smem((const void*)ms::agg_nms_ms_kernel<NW_, NS_, T_>, smem, "agg_nms_ms_kernel")) return rc_; \
    ms::agg_nms_ms_kernel<NW_, NS_, T_><<<grid, 32 * NW_, smem, st>>>(a, g);                                     \
  } while (0)
#define HPD_MS_NS_T(NW_, T_)                                                                                     \
  do {                                                                                                           \
    if (a.n_scales == 1) HPD_MS_LAUNCH(NW_, 1, T_); else if (a.n_scales == 2) HPD_MS_LAUNCH(NW_, 2, T_); else HPD_MS_LAUNCH(NW_, 3, T_); \
  } while (0)
#define HPD_MS_NS(NW_)                                                                                           \
  do {                                                                                                           \
    if (a.dtype == HPD_F16) HPD_MS_NS_T(NW_, __half);                                                           \
    else if (a.dtype == HPD_BF16) HPD_MS_NS_T(NW_, __nv_bfloat16);                                             \
    else HPD_MS_NS_T(NW_, float);                                                                                \
  } while (0)
        if (NW == 5) HPD_MS_NS(5); else if (NW == 4) HPD_MS_NS(4); else if (NW == 3) HPD_MS_NS(3); else HPD_MS_NS(2);
#undef HPD_MS_NS
#undef HPD_MS_NS_T
#undef HPD_MS_LAUNCH
        count_launch();
        return check_launch("agg_nms_ms_kernel");
      }
    }
  }
  const size_t smem = sizeof(float) * ((size_t)OT_R * OT_C + (size_t)OT_R * TW + (size_t)a.HI_R * a.HI_C +
                                       (size_t)a.LO_R * a.LO_C + 4 * (OT_C + OT_R + a.HI_C + a.HI_R));
  if (smem > 227 * 1024) {
    set_error("resize ratios need %zu bytes of shared memory per tile (> 227 KB)", smem);
    return HPD_EINVAL;
  }
  if (int rc = ensure_dynamic_smem((const void*)agg_nms_generic_kernel, smem, "agg_nms_generic_kernel")) return rc;
  const dim3 grid((a.W + TW - 1) / TW, (a.H + TH - 1) / TH, a.B * a.K);
  agg_nms_generic_kernel<<<grid, kAggThreads, smem, st>>>(a);
  count_launch();
  return check_launch("agg_nms_generic_kernel");
}

}  // namespace

HpdStageInputs two_stage_inputs(const HpdScaleInputs& s) {
  HpdStageInputs r;
  memset(&r, 0, sizeof(r));
  r.hm[0] = s.hm_lo; r.hm[1] = s.hm_hi; r.hm_f[0] = s.hm_lo_f; r.hm_f[1] = s.hm_hi_f;
  r.tag = s.tag; r.tag_f = s.tag_f;
  r.num_stages = 2;
  return r;
}

HpdScaleInputs tag_scale_inputs(const HpdStageInputs& s) {
  HpdScaleInputs r;
  memset(&r, 0, sizeof(r));
  r.tag = s.tag; r.tag_f = s.tag_f;
  return r;
}

int launch_aggregate_nms(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, cudaStream_t st) {
  if (int rc = launch_aggregation_kernel(p, scales, buf, st)) return rc;
  if (!buf->agg_tags) return HPD_OK;
  const HpdScaleInputs tags = tag_scale_inputs(scales[p->tag_scale]);
  HpdParams q = *p;   // launch_aggregate_tags reads scales[tag_scale]
  q.tag_scale = 0;
  return launch_aggregate_tags(&q, &tags, buf->agg_tags, st);
}

int launch_nms(const HpdParams* p, const HpdBuffers* buf, float* nms_out, cudaStream_t st) {
  if (!buf->agg_hm || !buf->nms_mask || !buf->nms_wmax || !buf->hm_wmax || !buf->tag_bmin || !buf->tag_bmax) {
    set_error("hpd_nms: agg_hm, nms_mask, nms_wmax, hm_wmax, tag_bmin, tag_bmax are required");
    return HPD_EINVAL;
  }
  const int H = p->out_h, W = p->out_w, wpr = (W + 31) / 32;
  const dim3 grid((W + TW - 1) / TW, (H + TH - 1) / TH, p->batch * p->num_kpts);
  nms_kernel<<<grid, kAggThreads, 0, st>>>(buf->agg_hm, p->num_kpts, H, W, wpr, buf->nms_mask, buf->nms_wmax,
                                           buf->hm_wmax, buf->tag_bmin, buf->tag_bmax, nms_out);
  count_launch();
  return check_launch("nms_kernel");
}

int launch_resize(const HpdMap* in, int batch, int channels, float* out, int oh, int ow, cudaStream_t st) {
  if (!in || !in->ptr || !out || in->h < 1 || in->w < 1 || oh < 1 || ow < 1 || batch < 1 || channels < 1 ||
      (long long)batch * channels > 65535 || oh > 65535 || in->dtype != HPD_F32) {
    set_error("hpd_resize_bilinear: bad arguments");
    return HPD_EINVAL;
  }
  const dim3 grid(((ow + 3) / 4 + 255) / 256, oh, batch * channels);
  resize_kernel<<<grid, 256, 0, st>>>((const float*)in->ptr, in->stride_b, in->stride_c, channels, in->h, in->w, out, oh, ow,
                                      (float)in->h / (float)oh, (float)in->w / (float)ow);
  count_launch();
  return check_launch("resize_kernel");
}

}  // namespace hpd
