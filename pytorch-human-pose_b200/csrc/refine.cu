// Stage (e): quarter-pixel adjust, person score and missing-joint refine
// (/root/reference/src/keypoints/grouping.py:172-191, :276, :193-250, loop :278-282).
//
// The reference's refine makes, for every person, 17 passes over the full-resolution heatmap
// and tag maps (80-96 % of its decode time).  Only joints a person is MISSING can change
// (grouping.py:248), and for such a (person, joint) pair the answer is
//     argmax_pix ( hm[k][pix] - rint(|tags[k][pix] - T_person|) ),  first index on ties,
// where the subtracted term is a non-negative integer, so  value(pix) <= hm[k][pix].
// That bound makes the search sparse:
//   1. adjust_prepare_kernel (one warp per person) adjusts the detected joints, computes the
//      person score and the person's mean tag T, lists the (person, joint) pairs to refine and
//      seeds each pair's running best with the joint's top-k candidates;
//   2. refine_scan_kernel (one CTA per plane, two sweeps) walks the per-word maxima of the raw
//      heatmap (written by the aggregation kernel, 1/32 of a map) and expands only words whose
//      maximum can still beat or tie a pair's running best; bests are 64-bit keys (ordered value,
//      ~index) merged with atomicMax, which implements "largest value, then lowest index" exactly;
//   3. refine_apply_kernel turns the winning pixel into the refined joint.
// All float arithmetic is the reference's float32 sequence (separate mul/add, IEEE sqrt, rint).
#include "common.cuh"

namespace hpd {

namespace {

struct RefineWs {
  unsigned long long* keys;  // [B*K][M]   running best per listed (person, joint)
  float* T;                  // [B][M][2]  mean tag per person
  int32_t* miss_cnt;         // [B*K]
  int32_t* miss_pid;         // [B*K][M]
};

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

RefineWs carve(void* ws, int B, int K, int M) {
  RefineWs r;
  char* p = (char*)ws;
  r.keys = (unsigned long long*)p;
  p += align_up((size_t)B * K * M * 8, 256);
  r.T = (float*)p;
  p += align_up((size_t)B * M * 2 * 4, 256);
  r.miss_cnt = (int32_t*)p;
  p += align_up((size_t)B * K * 4, 256);
  r.miss_pid = (int32_t*)p;
  return r;
}

__device__ __forceinline__ unsigned ordered_u32(float v) {
  const unsigned u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unordered_f32(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ unsigned long long pack_key(float v, int idx) {
  return ((unsigned long long)ordered_u32(v) << 32) | (unsigned)(~(unsigned)idx);
}

// hm - rint(||tag - T||) with the reference's float32 op sequence (grouping.py:221-222);
// "+ 0.0f" folds -0 into +0 so that the ordered-bits compare agrees with np.argmax's ==.
__device__ __forceinline__ float refine_value(float hm, float t0, float t1, float T0, float T1, int E) {
  const float a = __fsub_rn(t0, T0);
  float s = __fmul_rn(a, a);
  if (E > 1) {
    const float b = __fsub_rn(t1, T1);
    s = __fadd_rn(s, __fmul_rn(b, b));
  }
  const float d = __fsqrt_rn(s);
  return __fadd_rn(__fsub_rn(hm, rintf(d)), 0.0f);
}

__device__ __forceinline__ void quarter_offset(const float* __restrict__ m, int H, int W, int xi, int yi, float& x,
                                               float& y) {
  x += (m[(size_t)yi * W + min(xi + 1, W - 1)] > m[(size_t)yi * W + max(xi - 1, 0)]) ? 0.25f : -0.25f;
  y += (m[(size_t)min(yi + 1, H - 1) * W + xi] > m[(size_t)max(yi - 1, 0) * W + xi]) ? 0.25f : -0.25f;
}

// one warp per person, one block per image.  Coordinates come from the top-k stage inside hpd_decode and are
// always inside the map; the standalone adjust / refine twins receive caller-supplied coordinates, which are
// clamped to the map before any read (the Python wrappers reject them where the reference would raise).
__global__ void __launch_bounds__(32 * HPD_MAX_PEOPLE) adjust_prepare_kernel(const float* __restrict__ agg_hm, const TagSource tags,
                                      const int32_t* __restrict__ idx_k, const float* __restrict__ tags_k,
                                      const int32_t* __restrict__ n_person, int K,
                                      int M, int E, int H, int W, int do_adjust, int do_refine,
                                      float* __restrict__ poses, float* __restrict__ person_scores, RefineWs ws) {
  __shared__ float s_score[HPD_MAX_PEOPLE][HPD_MAX_KPTS];
  __shared__ float s_tl[HPD_MAX_PEOPLE][HPD_MAX_KPTS][HPD_MAX_EMB];
  __shared__ int s_cnt[HPD_MAX_KPTS];
  const int b = blockIdx.x;
  const int p = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = 3 + E;
  const int P = n_person[b];
  if (threadIdx.x < HPD_MAX_KPTS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const float* hm_b = agg_hm + (size_t)b * K * H * W;
  float T0 = 0.f, T1 = 0.f;
  bool missing = false;
  if (p < P) {
    float score = 0.f, x = 0.f, y = 0.f;
    float* d = poses + (((size_t)b * M + p) * K + lane) * D;
    if (lane < K) {
      x = d[0]; y = d[1]; score = d[2];
      if (do_adjust && score != 0.f) {   // grouping.py:172-191
        const int xi = min(max((int)x, 0), W - 1), yi = min(max((int)y, 0), H - 1);
        quarter_offset(hm_b + (size_t)lane * H * W, H, W, xi, yi, x, y);
        x += 0.5f; y += 0.5f;
        d[0] = x; d[1] = y;
      }
      s_score[p][lane] = score;
    }
    // tags of the detected joints at the (truncated) adjusted coordinates (grouping.py:206-210)
    const bool has = lane < K && score > 0.f;
    const unsigned hmask = __ballot_sync(kFull, has);
    if (has && do_refine) {
      const int pos = __popc(hmask & ((1u << lane) - 1u));
      const int xi = min(max((int)x, 0), W - 1), yi = min(max((int)y, 0), H - 1);
      float t[HPD_MAX_EMB];
      tag_value(tags, b * K + lane, yi * W + xi, t);
      s_tl[p][pos][0] = t[0];
      s_tl[p][pos][1] = (E > 1) ? t[1] : 0.f;
    }
    __syncwarp();
    if (lane == 0) {
      person_scores[(size_t)b * M + p] =
          __fdiv_rn(__fadd_rn(0.0f, np_sum_pairwise8(&s_score[p][0], K, 1)), (float)K);   // grouping.py:276
      if (do_refine) {
        const int n = __popc(hmask);
        float mv[HPD_MAX_EMB] = {0.f, 0.f};
        if (n > 0) np_mean_vectors(&s_tl[p][0][0], n, E, HPD_MAX_EMB, mv);
        else mv[0] = mv[1] = __int_as_float(0x7fc00000);
        T0 = mv[0]; T1 = mv[1];
        ws.T[((size_t)b * M + p) * 2 + 0] = T0;
        ws.T[((size_t)b * M + p) * 2 + 1] = T1;
      }
    }
    T0 = __shfl_sync(kFull, T0, 0);
    T1 = __shfl_sync(kFull, T1, 0);
    missing = do_refine && lane < K && score == 0.f;
  } else if (p < M && lane == 0) {
    person_scores[(size_t)b * M + p] = 0.f;
  }
  // list the pairs to refine and seed their running best with the joint's top-k candidates
  if (missing) {
    const int slot = atomicAdd(&s_cnt[lane], 1);
    const size_t bk = (size_t)b * K + lane;
    ws.miss_pid[bk * M + slot] = p;
    const float* m = hm_b + (size_t)lane * H * W;
    unsigned long long best = 0ull;
    // eight candidates at a time: their index loads, then their heatmap / tag loads, are all in flight together
    // (one dependent DRAM round trip per candidate made this loop most of the kernel's 30 us).  The candidates'
    // tags are the top-k stage's tags_k (the tags at idx_k), not re-read or re-interpolated.
    for (int j0 = 0; j0 < M; j0 += 8) {
      int idx[8];
      float hv[8], t0[8], t1[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) idx[u] = j0 + u < M ? idx_k[bk * M + j0 + u] : -1;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        hv[u] = t0[u] = t1[u] = 0.f;
        if (idx[u] >= 0) {
          const size_t o = (bk * M + j0 + u) * E;
          hv[u] = m[idx[u]];
          t0[u] = tags_k[o];
          if (E > 1) t1[u] = tags_k[o + 1];
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (idx[u] < 0) continue;
        const unsigned long long key = pack_key(refine_value(hv[u], t0[u], t1[u], T0, T1, E), idx[u]);
        best = key > best ? key : best;
      }
    }
    ws.keys[bk * M + slot] = best;
  }
  __syncthreads();
  if (threadIdx.x < K) ws.miss_cnt[(size_t)b * K + threadIdx.x] = do_refine ? s_cnt[threadIdx.x] : 0;
}

constexpr int kScanWarps = 16;

// One CTA per (image, joint) plane that has pairs to refine.  Two sweeps over the plane's word maxima, the 32-word
// chunks dealt round-robin to the warps: sweep 0 expands only words whose raw maximum reaches the joint's M-th
// top-k score (the words around the strongest peaks), sweep 1 the rest.  The running bests live in shared memory
// (re-read at every chunk, merged with atomicMax as soon as they improve), so after sweep 0 almost every remaining
// word is pruned by its maximum instead of being climbed flank by flank in index order; the word maxima of
// sweep 1 are re-read from cache.  (Round 1 ran the sweeps as two launches of 8 CTAs per plane with the bests in
// global memory: twice the chunk bookkeeping, and an L2 round trip per chunk for the bests.)
// Tags of the 32 pixels (y, x0 + lane) of one image row word, loaded by the whole warp (lanes right of the image
// get the last column's).  From the map: one load per lane and component.  Interpolated: the word's pixels share
// their two source rows and span a few source columns (10 at the x4 tag resolution), so every distinct source value
// is loaded once, by the lane of its column, and shuffled to the lanes whose taps use it -- instead of four loads per
// lane and component.  Bit-identical to tag_at.
__device__ __forceinline__ void word_tags(const TagSource& s, int b, int k, int y, int x0, int lane, float& t0, float& t1) {
  const int x = min(x0 + lane, s.W - 1);
  t1 = 0.f;
  if (s.map != nullptr) {
    const float* q = s.map + (((size_t)b * s.K + k) * s.H * s.W + (size_t)y * s.W + x) * s.E;
    t0 = q[0];
    if (s.E > 1) t1 = q[1];
    return;
  }
  const Tap tx = axis_tap(s.s_x, x, s.tw, s.W), ty = axis_tap(s.s_y, y, s.th, s.H);
  const int c_lo = __shfl_sync(kFull, tx.i0, 0);
  const int span = __shfl_sync(kFull, tx.i1, 31) - c_lo + 1;   // taps are monotone in x
  if (span > 32) {   // a tag map finer than the output: too many distinct taps to share
    float t[HPD_MAX_EMB];
    tag_at(s, b, k, y, x, t);
    t0 = t[0];
    if (s.E > 1) t1 = t[1];
    return;
  }
  const int j0 = tx.i0 - c_lo, j1 = tx.i1 - c_lo;
  float out[HPD_MAX_EMB] = {0.f, 0.f};
#pragma unroll
  for (int e = 0; e < HPD_MAX_EMB; ++e) {
    if (e >= s.E) break;
    const bool unflip = (e == 1) && !s.tags_preflipped;
    const float* p = (e == 0) ? s.tag : s.tag_f;
    const size_t po = (e == 0) ? (size_t)b * s.tag_sb + (size_t)k * s.tag_sc
                               : (size_t)b * s.tagf_sb + (size_t)(unflip ? s.flip[k] : k) * s.tagf_sc;
    float v0 = 0.f, v1 = 0.f;
    if (lane < span) {
      const int c = c_lo + lane;
      const size_t col = (size_t)(unflip ? s.tw - 1 - c : c);
      v0 = in_elem(p, po + (size_t)ty.i0 * s.tw + col, s.dtype);
      v1 = in_elem(p, po + (size_t)ty.i1 * s.tw + col, s.dtype);
    }
    const float v00 = __shfl_sync(kFull, v0, j0), v01 = __shfl_sync(kFull, v0, j1);
    const float v10 = __shfl_sync(kFull, v1, j0), v11 = __shfl_sync(kFull, v1, j1);
    out[e] = lerp2(tx.w0, tx.w1, ty.w0, ty.w1, v00, v01, v10, v11);
  }
  t0 = out[0];
  t1 = out[1];
}

__global__ void __launch_bounds__(kScanWarps * 32) refine_scan_kernel(const float* __restrict__ agg_hm,
                                                                      const TagSource tags,
                                                                      const float* __restrict__ hmax,
                                                                      const float* __restrict__ tag_bmin,
                                                                      const float* __restrict__ tag_bmax,
                                                                      const float* __restrict__ scores_k,
                                                                      int K, int M, int E, int H, int W, int wpr,
                                                                      RefineWs ws) {
  const int bk = blockIdx.x;
  const int cnt = ws.miss_cnt[bk];
  if (cnt == 0) return;
  __shared__ unsigned long long s_best[32];
  const int b = bk / K;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nwords = H * wpr;
  const float* m = agg_hm + (size_t)bk * H * W;
  const float* hx = hmax + (size_t)bk * nwords;
  const int HB = (H + 3) >> 2;
  const float* tlo = tag_bmin + (size_t)bk * HB * wpr;
  const float* thi = tag_bmax + (size_t)bk * HB * wpr;
  const float split = scores_k[(size_t)bk * M + M - 1];
  unsigned long long* gkeys = s_best;
  if (threadIdx.x < 32) s_best[threadIdx.x] = threadIdx.x < cnt ? ws.keys[(size_t)bk * M + threadIdx.x] : ~0ull;
  __syncthreads();

  // lane q < cnt tracks listed pair q
  float T0 = 0.f, T1 = 0.f;
  unsigned long long best = ~0ull;
  if (lane < cnt) {
    const int p = ws.miss_pid[(size_t)bk * M + lane];
    T0 = ws.T[((size_t)b * M + p) * 2 + 0];
    T1 = ws.T[((size_t)b * M + p) * 2 + 1];
  }
  const int w_end = nwords;

  constexpr int kStep = 32 * kScanWarps;
  for (int pass_id = 0; pass_id < 2; ++pass_id) {
  // the word maxima of the next two chunks of this warp are already on their way while one is processed
  float hv_n1 = (32 * warp + lane < w_end) ? hx[32 * warp + lane] : -INFINITY;
  float hv_n2 = (32 * warp + kStep + lane < w_end) ? hx[32 * warp + kStep + lane] : -INFINITY;
  for (int base = 32 * warp; base < w_end; base += kStep) {
    const int wd = base + lane;
    const float hv = hv_n1;
    hv_n1 = hv_n2;
    hv_n2 = (wd + 2 * kStep < w_end) ? hx[wd + 2 * kStep] : -INFINITY;
    if (lane < cnt) best = *(volatile unsigned long long*)(gkeys + lane);   // newest bests of all warps of the plane
    // A word matters to a pair if  max(hm) - rint(min distance to the pair's tag)  can reach the pair's
    // running best: the distance is bounded from below through the band's range of the first tag
    // component (tag_bmin / tag_bmax, minus a slack that covers the rounding of the interpolation).
    auto reach = [&](float hmx, float lo_, float hi_, float Tq) {   // ordered upper bound of the value
      const float slack = 1e-4f * (1.f + fabsf(Tq) + fmaxf(fabsf(lo_), fabsf(hi_)));
      const float dmin = fmaxf(fmaxf(fmaxf(lo_ - Tq, Tq - hi_), 0.f) - slack, 0.f);
      return ordered_u32(__fadd_rn(__fsub_rn(hmx, rintf(dmin)), 0.0f));
    };
    const bool mine = wd < w_end && ((pass_id == 0) ? (hv >= split) : !(hv >= split));
    // cheap test first: the word's maximum against the smallest running best of all pairs (most chunks end here,
    // before the tag bounds -- an integer division and two more loads -- are touched)
    const unsigned thr = __reduce_min_sync(kFull, (unsigned)(best >> 32));
    const unsigned hv_o = ordered_u32(__fadd_rn(hv, 0.0f));
    if (!__any_sync(kFull, mine && hv_o >= thr)) continue;
    float lo = 0.f, hi = 0.f;
    if (mine) {
      const int yw = wd / wpr;
      const int bi = (yw >> 2) * wpr + (wd - yw * wpr);
      lo = tlo[bi];
      hi = thi[bi];
    }
    const unsigned chunk_max = __reduce_max_sync(kFull, mine ? hv_o : 0u);
    bool viable = false;
    for (int q = 0; q < cnt; ++q) {
      const unsigned bq = (unsigned)(__shfl_sync(kFull, best, q) >> 32);
      if (bq > chunk_max) continue;                       // no word of this chunk reaches pair q
      const float Tq = __shfl_sync(kFull, T0, q);
      viable = viable || (reach(hv, lo, hi, Tq) >= bq);
    }
    uint32_t pass = __ballot_sync(kFull, mine && viable);
    while (pass) {
      const int l = __ffs(pass) - 1;
      pass &= pass - 1;
      const float hw_f = __shfl_sync(kFull, hv, l), lo_l = __shfl_sync(kFull, lo, l), hi_l = __shfl_sync(kFull, hi, l);
      // only the pairs this word can still reach
      uint32_t todo = __ballot_sync(kFull, lane < cnt && reach(hw_f, lo_l, hi_l, T0) >= (unsigned)(best >> 32));
      if (!todo) continue;
      const int w2 = base + l;
      const int y = w2 / wpr, x0 = (w2 - y * wpr) * 32;
      const bool valid = x0 + lane < W;
      const int idx = y * W + x0 + lane;
      float pv = 0.f, t0, t1;
      if (valid) pv = m[idx];
      word_tags(tags, b, bk - b * K, y, x0, lane, t0, t1);
      bool improved = false;
      while (todo) {
        const int q = __ffs(todo) - 1;
        todo &= todo - 1;
        const unsigned long long bq = __shfl_sync(kFull, best, q);
        const float v = refine_value(pv, t0, t1, __shfl_sync(kFull, T0, q), __shfl_sync(kFull, T1, q), E);
        const unsigned vo = valid ? ordered_u32(v) : 0u;
        if (!__any_sync(kFull, vo >= (unsigned)(bq >> 32))) continue;
        const unsigned vmax = __reduce_max_sync(kFull, vo);
        const int first = __ffs(__ballot_sync(kFull, vo == vmax)) - 1;    // lowest index among equal values
        const unsigned long long wbest = ((unsigned long long)vmax << 32) | (unsigned)(~(unsigned)(y * W + x0 + first));
        if (wbest > bq) {
          if (lane == q) best = wbest;
          improved = true;
        }
      }
      if (improved && lane < cnt) atomicMax(gkeys + lane, best);
    }
  }
  __syncthreads();      // every warp has finished this sweep: the next one prunes against the merged bests
  }
  if (threadIdx.x < cnt) ws.keys[(size_t)bk * M + threadIdx.x] = s_best[threadIdx.x];
}

// One block per image.  Phase 1 turns each listed pair's winning pixel into the refined joint (grouping.py:236-249).
// Phase 2 -- the epilogue of the whole decode -- writes the image's result record (HpdRecordLayout): the grouped
// joints / person scores / count / flags as they are, plus the COCO record of bin/eval.py:31-47 with the joints
// back-projected to the raw image through the image's inverse affine matrix (results.py:158-171,189-201,244):
// np.dot(M, [x, y, 1.0]) in float64 -- OpenBLAS's dgemv order fma(m2, 1, fma(m0, x, m1*y)) -- then rounded to
// float32 because the reference writes it into a float32 array (results.py:165-170); the empty-scene fallback's
// pseudo-person is float64 throughout with every score 0.01 (grouping.py:262-269), so its row stays unrounded.
__global__ void __launch_bounds__(256) refine_apply_kernel(const float* __restrict__ agg_hm, int do_refine, int K, int M,
                                                           int E, int H, int W, float* __restrict__ poses,
                                                           const float* __restrict__ person_scores,
                                                           const int32_t* __restrict__ n_person,
                                                           const int32_t* __restrict__ flags, RefineWs ws,
                                                           uint8_t* __restrict__ records,
                                                           const double* __restrict__ inv_affine, HpdRecordLayout L,
                                                           double fallback_score) {
  const int b = blockIdx.x;
  const int D = 3 + E;
  if (do_refine) {
    for (int i = threadIdx.x; i < K * M; i += blockDim.x) {   // (joint, slot)
      const int k = i / M, slot = i - k * M;
      const int bk = b * K + k;
      if (slot >= ws.miss_cnt[bk]) continue;
      const int p = ws.miss_pid[(size_t)bk * M + slot];
      const unsigned long long key = ws.keys[(size_t)bk * M + slot];
      const int idx = (int)(~(unsigned)key);
      const float* m = agg_hm + (size_t)bk * H * W;
      const float val = m[idx];
      if (!(val > 0.f)) continue;     // grouping.py:248 (the pair is listed only if its score == 0)
      const int y = idx / W, x = idx % W;
      float fx = (float)x + 0.5f, fy = (float)y + 0.5f;
      quarter_offset(m, H, W, x, y, fx, fy);
      float* d = poses + (((size_t)b * M + p) * K + k) * D;
      d[0] = fx; d[1] = fy; d[2] = val;
    }
  }
  if (records == nullptr) return;
  __syncthreads();
  uint8_t* row = records + (size_t)b * L.row_bytes;
  const int P = n_person[b];
  const int flag = flags[b];
  const float* src = poses + (size_t)b * M * K * D;
  float* r_poses = (float*)(row + L.off_poses);
  for (int i = threadIdx.x; i < M * K * D; i += blockDim.x) r_poses[i] = src[i];
  float* r_scores = (float*)(row + L.off_person_scores);
  for (int i = threadIdx.x; i < M; i += blockDim.x) r_scores[i] = person_scores[(size_t)b * M + i];
  if (threadIdx.x == 0) {
    *(int32_t*)(row + L.off_n_person) = P;
    *(int32_t*)(row + L.off_flags) = flag;
  }
  double m0 = 1.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 1.0, m5 = 0.0;
  if (inv_affine) {
    const double* a = inv_affine + (size_t)b * 6;
    m0 = a[0]; m1 = a[1]; m2 = a[2]; m3 = a[3]; m4 = a[4]; m5 = a[5];
  }
  const bool fallback = flag & 1;
  double* coco = (double*)(row + L.off_coco);
  for (int i = threadIdx.x; i < M * (K + 1); i += blockDim.x) {
    const int p = i / (K + 1), k = i - p * (K + 1);
    double* c = coco + (size_t)p * L.coco_stride;
    if (k == K) {   // "score": obj_scores[i].mean().item(), bin/eval.py:45
      c[3 * K] = p < P ? (fallback ? fallback_score : (double)person_scores[(size_t)b * M + p]) : 0.0;
      continue;
    }
    double X = 0.0, Y = 0.0, V = 0.0;
    if (p < P) {
      const double x = (double)src[((size_t)p * K + k) * D], y = (double)src[((size_t)p * K + k) * D + 1];
      if (inv_affine) {
        X = fma(m2, 1.0, fma(m0, x, __dmul_rn(m1, y)));
        Y = fma(m5, 1.0, fma(m3, x, __dmul_rn(m4, y)));
      } else {
        X = x; Y = y;
      }
      if (!fallback) { X = (double)(float)X; Y = (double)(float)Y; }
      V = 1.0;
    }
    c[3 * k] = X; c[3 * k + 1] = Y; c[3 * k + 2] = V;
  }
}

}  // namespace

size_t refine_workspace_bytes(const HpdParams* p) {
  const size_t B = p->batch, K = p->num_kpts, M = p->max_people;
  return align_up(B * K * M * 8, 256) + align_up(B * M * 2 * 4, 256) + align_up(B * K * 4, 256) +
         align_up(B * K * M * 4, 256);
}

int launch_adjust_refine(const HpdParams* p, const HpdBuffers* buf, void* wsp, size_t ws_bytes, cudaStream_t st) {
  if (!buf->agg_hm || !buf->hm_wmax || !buf->tag_bmin || !buf->tag_bmax || !buf->idx_k || !buf->scores_k || !buf->poses ||
      !buf->person_scores || !buf->n_person || (p->do_refine && !buf->tags_k)) {
    set_error("hpd_adjust_refine: agg_hm, hm_wmax, tag_bmin, tag_bmax, idx_k, scores_k, poses, person_scores, n_person and "
              "(refine) tags_k are required");
    return HPD_EINVAL;
  }
  TagSource tags;
  if (int rc = make_tag_source(p, buf, &tags, "hpd_adjust_refine")) return rc;
  if (!wsp || ws_bytes < refine_workspace_bytes(p)) {
    set_error("hpd_adjust_refine: workspace of %zu bytes required, got %zu", refine_workspace_bytes(p), ws_bytes);
    return HPD_EWORKSPACE;
  }
  if ((uintptr_t)wsp % 8 != 0) {
    set_error("hpd_adjust_refine: workspace must be 8-byte aligned");
    return HPD_EINVAL;
  }
  const int B = p->batch, K = p->num_kpts, M = p->max_people, E = p->emb, H = p->out_h, W = p->out_w;
  const int wpr = (W + 31) / 32;
  RefineWs ws = carve(wsp, B, K, M);
  adjust_prepare_kernel<<<B, 32 * M, 0, st>>>(buf->agg_hm, tags, buf->idx_k, buf->tags_k, buf->n_person, K, M, E, H, W,
                                              p->do_adjust, p->do_refine, buf->poses, buf->person_scores, ws);
  count_launch();
  int rc = check_launch("adjust_prepare_kernel");
  if (rc) return rc;
  if (p->do_refine) {
    refine_scan_kernel<<<B * K, kScanWarps * 32, 0, st>>>(buf->agg_hm, tags, buf->hm_wmax, buf->tag_bmin, buf->tag_bmax,
                                                          buf->scores_k, K, M, E, H, W, wpr, ws);
    count_launch();
    if ((rc = check_launch("refine_scan_kernel"))) return rc;
  }
  if (!p->do_refine && !buf->records) return HPD_OK;
  if (buf->records && (!buf->flags || (uintptr_t)buf->records % 8 != 0)) {
    set_error("hpd_adjust_refine: records need flags and an 8-byte aligned buffer");
    return HPD_EINVAL;
  }
  // the fallback pseudo-person's score: np.mean of K float64 copies of 0.01 (numpy's pairwise-8 order)
  double fb_score;
  {
    const double v = 0.01;
    if (K < 8) {
      fb_score = -0.0;
      for (int i = 0; i < K; ++i) fb_score += v;
    } else {
      double r[8];
      for (int j = 0; j < 8; ++j) r[j] = v;
      int i = 8;
      for (; i < K - (K % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += v;
      fb_score = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
      for (; i < K; ++i) fb_score += v;
    }
    fb_score /= (double)K;
  }
  refine_apply_kernel<<<B, 256, 0, st>>>(buf->agg_hm, p->do_refine, K, M, E, H, W, buf->poses, buf->person_scores,
                                         buf->n_person, buf->flags, ws, buf->records, buf->inv_affine,
                                         record_layout(K, M, E), fb_score);
  count_launch();
  return check_launch("refine_apply_kernel");
}

}  // namespace hpd
