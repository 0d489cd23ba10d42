// Multi-scale / general-ratio fused aggregation + NMS kernel (BASELINE config 3: test scales 0.5/1.0/1.5).
// Included by aggregate_nms.cu after aggregate_nms_x2.cuh (needs AggArgs, x2::stage helpers).
//
// Same column-walking scheme as the x2 kernel (each lane owns 4 adjacent output columns and walks down
// the rows with everything in registers), generalised:
//   * every scale s has its own half-resolution stage-mean tile S_s in shared memory (lo --x2--> hi is
//     always an exact x2 in HigherHRNet; hi --> output uses the general torch taps, e.g. x4, x2, x4/3);
//   * a lane keeps, per scale, the column taps of its 4 columns in registers and a two-row cache of
//     horizontally interpolated S_s rows; the vertical taps of every (scale, output row) come from a small
//     shared table; the scales are summed sequentially and divided by n like torch.stack(...).mean(0);
//   * tags come from one scale and must be an exact x4 (as in the reference); NMS, word side arrays and tag
//     bounds are the x2 kernel's, and like it this kernel writes no tag map;
//   * input elements are float32, IEEE half or bfloat16 (T); 16-bit values are widened exactly as they are loaded,
//     shared memory and all arithmetic stay float32.
// Bit-identical to the generic kernel (tests/test_gpu_stages.py).
#pragma once

namespace ms {

// -DHPD_MS_PROFILE: one CTA in the middle of the grid prints clock64() per phase (development aid)
#ifdef HPD_MS_PROFILE
#define MSP_MARK(i) do { if (prof) pt[i] = clock64(); } while (0)
#else
#define MSP_MARK(i)
#endif

using x2::clampi;
using x2::max3;
using x2::tap_x2;

constexpr int RB = 16;            // output rows per CTA (multiple of 4)
constexpr int NROWS = RB + 4;     // walked rows: band + 2 halo rows on each side
constexpr int TR = RB / 4 + 2;    // quarter-res tag rows staged

struct Geom {                     // shared-memory layout, computed on the host
  int off_s[HPD_MAX_SCALES];      // float offset of S_s
  int hr[HPD_MAX_SCALES], hc[HPD_MAX_SCALES];   // rows / row stride (multiple of 4) of S_s
  int off_lo[HPD_MAX_SCALES];     // quarter-res staging tile of scale s
  int lr[HPD_MAX_SCALES], lc[HPD_MAX_SCALES];
  int off_edge, off_tab, total;
};

// One staged window (a scale's quarter- or half-res rows).  Row r of it is the job "copy nvec vectors of four
// elements from p + r*w, flip-averaged with the vectors running backwards from pf + r*w, to
// smem[dst + r*stride]".
template <typename T>
struct Seg {
  const T* p;                     // first vector of row 0
  const T* pf;                    // mirrored first vector of row 0 in the flipped run's map, or null
  int dst, stride, nvec, w, rows;
};

// vector q (four elements) of a row, widened to float32: one 16-byte load for float, one 8-byte load for 16-bit types
__device__ __forceinline__ float4 ld_vec(const float* p, int q) { return __ldg(reinterpret_cast<const float4*>(p) + q); }
template <typename T>
__device__ __forceinline__ float4 ld_vec(const T* p, int q) { return x2::In<T>::ld4(p + 4 * q); }

// Stage all windows: the rows of all segments form one job list dealt round-robin to the warps; a warp
// keeps two rows in flight (all loads of both issued before the first store).  Vector loads; the flipped
// operand is read as the mirrored vector and reversed in registers (model.py:87-90).
template <int NW, int NSEG, typename T>
__device__ __forceinline__ void stage_segments(float* __restrict__ smem, const Seg<T>* __restrict__ seg, int warp, int lane) {
  constexpr int MAXIT = 4;
  int start[NSEG + 1];
  start[0] = 0;
#pragma unroll
  for (int i = 0; i < NSEG; ++i) start[i + 1] = start[i] + seg[i].rows;
  const int njobs = start[NSEG];
  struct Row { const T* p; const T* pf; float* dst; int nvec; };
  auto locate = [&](int j) {
    Row r{nullptr, nullptr, nullptr, 0};
    if (j < njobs) {
      int sg = 0, first = 0;
#pragma unroll
      for (int i = 1; i < NSEG; ++i)
        if (j >= start[i]) { sg = i; first = start[i]; }
      const Seg<T>& S = seg[sg];
      const int rr = j - first;
      r.p = S.p + (size_t)rr * S.w;
      r.pf = S.pf ? S.pf + (size_t)rr * S.w : nullptr;
      r.dst = smem + S.dst + rr * S.stride;
      r.nvec = S.nvec;
    }
    return r;
  };
  // (the "whole group of 32 vectors is past the row" tests are warp-uniform: real branches, so short
  // rows do not pay for MAXIT predicated-off copies)
  auto load = [&](const Row& r, int qb, float4 (&v)[MAXIT], float4 (&f)[MAXIT]) {
#pragma unroll
    for (int u = 0; u < MAXIT; ++u) {
      if (qb + 32 * u >= r.nvec) break;
      const int q = qb + lane + 32 * u;
      if (q < r.nvec) {
        v[u] = ld_vec(r.p, q);
        if (r.pf) f[u] = ld_vec(r.pf, -q);
      }
    }
  };
  auto store = [&](const Row& r, int qb, const float4 (&v)[MAXIT], const float4 (&f)[MAXIT]) {
#pragma unroll
    for (int u = 0; u < MAXIT; ++u) {
      if (qb + 32 * u >= r.nvec) break;
      const int q = qb + lane + 32 * u;
      if (q < r.nvec) {
        float4 o = v[u];
        if (r.pf) {
          o.x = __fmul_rn(__fadd_rn(v[u].x, f[u].w), 0.5f);
          o.y = __fmul_rn(__fadd_rn(v[u].y, f[u].z), 0.5f);
          o.z = __fmul_rn(__fadd_rn(v[u].z, f[u].y), 0.5f);
          o.w = __fmul_rn(__fadd_rn(v[u].w, f[u].x), 0.5f);
        }
        reinterpret_cast<float4*>(r.dst)[q] = o;
      }
    }
  };
  for (int j = warp; j < njobs; j += 2 * NW) {
    const Row A = locate(j), B = locate(j + NW);
    const int nv = max(A.nvec, B.nvec);
    for (int qb = 0; qb < nv; qb += 32 * MAXIT) {
      float4 va[MAXIT], fa[MAXIT], vb[MAXIT], fb[MAXIT];
      load(A, qb, va, fa);
      load(B, qb, vb, fb);
      store(A, qb, va, fa);
      store(B, qb, vb, fb);
    }
  }
}

template <int NW, int NS, typename T>
__global__ void __launch_bounds__(32 * NW, 16 / NW) agg_nms_ms_kernel(const AggArgs a, const Geom g) {
  extern __shared__ __align__(16) float smem[];
  constexpr int tc = 32 * NW + 8;
  constexpr int nthr = 32 * NW;
  float* sT = smem;                                   // the tag tile aliases the S tiles (consumed first)
  float* sEdge = smem + g.off_edge;
  // out-row -> S_s row taps: [NS][NROWS] x (packed i0 | i1 << 8 | advance << 16, w0, w1); the advance code
  // says how the walk's two cached rows move on: 0 keep both, 1 shift (new i0 = old i1), 2 reload; -1 = the
  // output row is outside the image
  int* rt_pk = (int*)(smem + g.off_tab);
  float* rt_w0 = (float*)(rt_pk + NS * NROWS);
  float* rt_w1 = rt_w0 + NS * NROWS;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int bk = blockIdx.z, b = bk / a.K, k = bk % a.K, kf = a.flip[k];
  const int H = a.H, W = a.W;
  const int x0 = blockIdx.x * 128 * NW, y0 = blockIdx.y * RB;
  const int xw = x0 + 128 * warp;
  const int X0 = xw + 4 * lane;
  const bool active = X0 < W;
  const int ys = y0 - 2;
  const float NINF = -INFINITY;
#ifdef HPD_MS_PROFILE
  const bool prof = tid == 0 && blockIdx.x == 0 && blockIdx.y == gridDim.y / 2 && blockIdx.z == gridDim.z / 2;
  long long pt[8];
#endif
  MSP_MARK(0);

  // windows of every scale this CTA needs (hya, hxa, nhy, nhx, lya, lxa) and the staging jobs for them;
  // published by the first barrier of phase 0
  __shared__ int s_win[HPD_MAX_SCALES][6];
  __shared__ Seg<T> s_seg[2 * HPD_MAX_SCALES];
  if (tid < NS) {
    const int s = tid;
    const ScaleDev& S = a.sc[s];
    const int oya = max(y0 - 2, 0), oyb = min(y0 + RB + 2, H) - 1;
    const int oxa = max(x0 - 2, 0), oxb = min(x0 + 128 * NW + 2, W) - 1;
    const int hya = axis_tap(S.s_hi_y, oya, S.hh, H).i0, hyb = axis_tap(S.s_hi_y, oyb, S.hh, H).i1;
    // column origins are rounded down to a multiple of 4 and widths up, so that rows move as 16-byte vectors
    const int hxa = axis_tap(S.s_hi_x, oxa, S.hw, W).i0 & ~3, hxb = axis_tap(S.s_hi_x, oxb, S.hw, W).i1 | 3;
    const int nhy = hyb - hya + 1, nhx = min(hxb, S.hw - 1) - hxa + 1;
    int t0, t1; float tw0, tw1;
    tap_x2(hya, S.lh, t0, t1, tw0, tw1);
    const int lya = t0;
    tap_x2(hyb, S.lh, t0, t1, tw0, tw1);
    const int nly = t1 - lya + 1;
    tap_x2(hxa, S.lw, t0, t1, tw0, tw1);
    const int lxa = t0 & ~3;
    tap_x2(min(hxb, S.hw - 1), S.lw, t0, t1, tw0, tw1);
    const int nlx = min(t1 | 3, S.lw - 1) - lxa + 1;
    s_win[s][0] = hya; s_win[s][1] = hxa; s_win[s][2] = nhy; s_win[s][3] = nhx; s_win[s][4] = lya; s_win[s][5] = lxa;
    Seg<T>& lo = s_seg[2 * s];
    Seg<T>& hi = s_seg[2 * s + 1];
    lo.p = reinterpret_cast<const T*>(S.lo) + (size_t)b * S.lo_sb + (size_t)k * S.lo_sc + (size_t)lya * S.lw + lxa;
    lo.pf = S.lo_f ? reinterpret_cast<const T*>(S.lo_f) + (size_t)b * S.lof_sb + (size_t)kf * S.lof_sc + (size_t)lya * S.lw + (S.lw - 4 - lxa)
                   : nullptr;
    lo.dst = g.off_lo[s]; lo.stride = g.lc[s]; lo.nvec = nlx >> 2; lo.w = S.lw; lo.rows = nly;
    hi.p = reinterpret_cast<const T*>(S.hi) + (size_t)b * S.hi_sb + (size_t)k * S.hi_sc + (size_t)hya * S.hw + hxa;
    hi.pf = S.hi_f ? reinterpret_cast<const T*>(S.hi_f) + (size_t)b * S.hif_sb + (size_t)kf * S.hif_sc + (size_t)hya * S.hw + (S.hw - 4 - hxa)
                   : nullptr;
    hi.dst = g.off_s[s]; hi.stride = g.hc[s]; hi.nvec = nhx >> 2; hi.w = S.hw; hi.rows = nhy;
  }

  // ---------------- phase 0: tag bounds (x4), identical to the x2 kernel --------------------------------
  {
    const int txo = x0 / 4 - 4, tyo = y0 / 4 - 1;
    const T* tg0 = reinterpret_cast<const T*>(a.tag) + (size_t)b * a.tag_sb + (size_t)k * a.tag_sc;
    x2::stage_tile<false, TR, tc, NW, false, T>(sT, tg0, (const T*)nullptr, tyo, txo, a.th, a.tw, warp, lane);
    __syncthreads();
    if (active) x2::tag_bounds_x4_band<RB, TR>(a, sT, tc, txo, X0, y0, b, k, lane);
    __syncthreads();
  }

  MSP_MARK(1);
  // ---------------- phase 1: flip-averaged quarter- and half-res windows of every scale -> smem ---------
  // (s_seg / s_win were filled at kernel entry; the barrier that ended phase 0 published them)
  stage_segments<NW, 2 * NS, T>(smem, s_seg, warp, lane);
  for (int i = tid; i < NS * NROWS; i += nthr) {     // output row -> S_s rows
    const int s = i / NROWS, t = i - s * NROWS;
    const ScaleDev& S = a.sc[s];
    const int hya = s_win[s][0];
    const int y = ys + t;
    int pk = -1;
    if (y >= 0 && y < H) {
      const Tap tp = axis_tap(S.s_hi_y, y, S.hh, H);
      int adv = 2;
      if (t > 0 && y > 0) {
        const Tap pv = axis_tap(S.s_hi_y, y - 1, S.hh, H);
        adv = (pv.i0 == tp.i0 && pv.i1 == tp.i1) ? 0 : ((pv.i1 == tp.i0) ? 1 : 2);
      }
      pk = (tp.i0 - hya) | ((tp.i1 - hya) << 8) | (adv << 16);
      rt_w0[i] = tp.w0; rt_w1[i] = tp.w1;
    }
    rt_pk[i] = pk;
  }
  __syncthreads();
  // ---------------- phase 2: S_s = (up2(lo_s) + hi_s) * 0.5 in place (results.py:225-226) -----------------
  // A thread owns 4 adjacent half-res columns C..C+3 (C a multiple of 4) of one scale and walks down the
  // rows of S_s: their x2 taps touch the quarter-res columns C/2-1 .. C/2+2 (scalar + aligned pair + scalar);
  // a quarter-res row is interpolated horizontally once (lerp2's inner FMAs) and kept in registers for the
  // two or three half-res rows that use it.  The column groups of all scales form one list.
  {
    int gstart[NS + 1];
    gstart[0] = 0;
#pragma unroll
    for (int s = 0; s < NS; ++s) gstart[s + 1] = gstart[s] + (s_win[s][3] >> 2);
    for (int gi = tid; gi < gstart[NS]; gi += nthr) {
      int s = 0, first = 0;
#pragma unroll
      for (int i = 1; i < NS; ++i)
        if (gi >= gstart[i]) { s = i; first = gstart[i]; }
      const int c4 = gi - first;
      const int lh = a.sc[s].lh, lw = a.sc[s].lw;
      const int hc = g.hc[s], lc = g.lc[s];
      const int hya = s_win[s][0], hxa = s_win[s][1], nhy = s_win[s][2], lya = s_win[s][4], lxa = s_win[s][5];
      float* sp = smem + g.off_s[s] + 4 * c4;
      const int C = hxa + 4 * c4, j = C >> 1;
      const float* lp = smem + g.off_lo[s] + (j - lxa) - lya * lc;
      const bool first_col = (C == 0);
      const int dl = first_col ? 0 : -1;                  // column C/2-1 (unused by the first column's (1,0) tap)
      const int dr = (j + 2 <= lw - 1) ? 2 : 1;           // column C/2+2, replicated at the right border
      auto hp = [&](int i, float (&h)[4]) {
        const float* rp = lp + i * lc;
        const float2 m = *reinterpret_cast<const float2*>(rp);
        const float l = rp[dl], r = rp[dr];
        h[0] = first_col ? fmaf(1.f, m.x, __fmul_rn(0.f, m.y)) : fmaf(0.25f, l, __fmul_rn(0.75f, m.x));
        h[1] = fmaf(0.75f, m.x, __fmul_rn(0.25f, m.y));
        h[2] = fmaf(0.25f, m.x, __fmul_rn(0.75f, m.y));
        h[3] = fmaf(0.75f, m.y, __fmul_rn(0.25f, r));
      };
      float hA[4] = {0.f, 0.f, 0.f, 0.f}, hB[4] = {0.f, 0.f, 0.f, 0.f};
      int ci0 = -1, ci1 = -1;
      for (int r = 0; r < nhy; ++r) {
        int i0, i1; float wy0, wy1;
        tap_x2(hya + r, lh, i0, i1, wy0, wy1);
        if (i0 != ci0) {
          if (i0 == ci1) {
#pragma unroll
            for (int c = 0; c < 4; ++c) hA[c] = hB[c];
          } else {
            hp(i0, hA);
          }
        }
        if (i1 == i0) {
#pragma unroll
          for (int c = 0; c < 4; ++c) hB[c] = hA[c];
        } else if (i1 != ci1) {
          hp(i1, hB);
        }
        ci0 = i0; ci1 = i1;
        float4 v = *reinterpret_cast<const float4*>(sp + r * hc);
        v.x = __fmul_rn(__fadd_rn(fmaf(wy0, hA[0], __fmul_rn(wy1, hB[0])), v.x), 0.5f);
        v.y = __fmul_rn(__fadd_rn(fmaf(wy0, hA[1], __fmul_rn(wy1, hB[1])), v.y), 0.5f);
        v.z = __fmul_rn(__fadd_rn(fmaf(wy0, hA[2], __fmul_rn(wy1, hB[2])), v.z), 0.5f);
        v.w = __fmul_rn(__fadd_rn(fmaf(wy0, hA[3], __fmul_rn(wy1, hB[3])), v.w), 0.5f);
        *reinterpret_cast<float4*>(sp + r * hc) = v;
      }
    }
  }
  __syncthreads();

  MSP_MARK(2);
  int hxa_s[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) hxa_s[s] = s_win[s][1];
  // per-lane column taps of every scale, kept in registers: tile-relative index of the first column's
  // left tap, then per column a 2-bit offset to its own left tap (hw <= W, so 4 adjacent output columns
  // span at most 4 source columns) and 1 bit "right tap = left tap + 1"
  int cbase[NS];
  unsigned cpack[NS];
  float cw1[NS][4];   // w0 is 1 - w1 exactly as axis_tap computes it (recomputed on use)
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    cpack[s] = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const Tap tp = axis_tap(a.sc[s].s_hi_x, min(X0 + c, W - 1), a.sc[s].hw, W);
      if (c == 0) cbase[s] = tp.i0 - hxa_s[s];
      cpack[s] |= (unsigned)(tp.i0 - hxa_s[s] - cbase[s]) << (2 * c);
      cpack[s] |= (unsigned)(tp.i1 - tp.i0) << (8 + c);
      cw1[s][c] = tp.w1;
    }
  }

  // ---------------- phase 3a: values of the 4 halo columns of this warp's strip ------------------------
  float* edge = sEdge + warp * NROWS * 4;
#pragma unroll
  for (int u = 0; u < (NROWS * 4 + 31) / 32; ++u) {
    const int i = lane + 32 * u;
    if (i < NROWS * 4) {
      const int t = i >> 2, e = i & 3;
      const int xe = (e < 2) ? xw - 2 + e : xw + 126 + e;
      const int y = ys + t;
      float v = NINF;
      if (xe >= 0 && xe < W && y >= 0 && y < H) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const Tap tx = axis_tap(a.sc[s].s_hi_x, xe, a.sc[s].hw, W);
          const float* sS = smem + g.off_s[s];
          const int pk = rt_pk[s * NROWS + t];
          const float* r0 = sS + (pk & 0xff) * g.hc[s];
          const float* r1 = sS + ((pk >> 8) & 0xff) * g.hc[s];
          const int c0 = tx.i0 - hxa_s[s], c1 = tx.i1 - hxa_s[s];
          const float vs = lerp2(tx.w0, tx.w1, rt_w0[s * NROWS + t], rt_w1[s * NROWS + t], r0[c0], r0[c1], r1[c0], r1[c1]);
          v = (s == 0) ? vs : __fadd_rn(v, vs);
        }
        if (NS > 1) v = __fdiv_rn(v, (float)NS);
      }
      edge[i] = v;
    }
  }
  __syncwarp();
  MSP_MARK(3);

  // ---------------- phase 3b: walk the rows ---------------------------------------------------------------
  {
    float hX[NS][4], hY[NS][4];   // the two horizontally interpolated S_s rows (i0, i1) of the current output row
    auto hpass = [&](int s, int r, float (&h)[4]) {
      const float* sp = smem + g.off_s[s] + r * g.hc[s];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int i0 = cbase[s] + (int)((cpack[s] >> (2 * c)) & 3u);
        const float v0 = sp[i0], v1 = sp[i0 + (int)((cpack[s] >> (8 + c)) & 1u)];
        h[c] = fmaf(1.f - cw1[s][c], v0, __fmul_rn(cw1[s][c], v1));
      }
    };
    x2::NmsColumnWalk<RB> nms;
    nms.init(a, b, k, X0, ys, edge, active, lane);

    auto row_value = [&](int t, float (&v)[4]) {
      const int y = ys + t;
      if (y < 0 || y >= H) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
        return;
      }
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int pk = rt_pk[s * NROWS + t];
        const float w0 = rt_w0[s * NROWS + t], w1 = rt_w1[s * NROWS + t];
        const int adv = pk >> 16;                   // uniform over the CTA
        if (adv != 0) {
          const int i0 = pk & 0xff, i1 = (pk >> 8) & 0xff;
          if (adv == 1) {
#pragma unroll
            for (int c = 0; c < 4; ++c) hX[s][c] = hY[s][c];
          } else {
            hpass(s, i0, hX[s]);
          }
          if (i1 == i0) {
#pragma unroll
            for (int c = 0; c < 4; ++c) hY[s][c] = hX[s][c];
          } else {
            hpass(s, i1, hY[s]);
          }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float vs = fmaf(w0, hX[s][c], __fmul_rn(w1, hY[s][c]));
          v[c] = (s == 0) ? vs : __fadd_rn(v[c], vs);
        }
      }
      if (NS == 3) {
        // x / 3 as two FMAs around the rounded reciprocal (checked against IEEE division for every
        // finite float: exact for all of them but -0, which with the tiny values takes the real division)
        const float third = 0.333333343267440796f;
        bool odd = false;
#pragma unroll
        for (int c = 0; c < 4; ++c) odd |= fabsf(v[c]) < 1e-30f && __float_as_uint(v[c]) != 0u;
        if (__any_sync(kFull, odd)) {
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = __fdiv_rn(v[c], 3.0f);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float q0 = __fmul_rn(v[c], third);
            v[c] = fmaf(fmaf(-3.0f, q0, v[c]), third, q0);
          }
        }
      } else if (NS > 1) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = __fdiv_rn(v[c], (float)NS);
      }
      if (!active) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = NINF;
      }
    };

    // (not unrolled: with NS scales the body is large, and one copy keeps it in the instruction cache)
#pragma unroll 1
    for (int t = 0; t < NROWS; ++t) {
      float v[4];
      row_value(t, v);
      nms.row(a, t, v);
    }
  }
  MSP_MARK(4);
#ifdef HPD_MS_PROFILE
  if (prof)
    printf("ms profile (cycles): tag bounds %lld, stage+S tiles %lld, taps+halo %lld, walk %lld\n", pt[1] - pt[0], pt[2] - pt[1],
           pt[3] - pt[2], pt[4] - pt[3]);
#endif
}

}  // namespace ms
