// Stage (d): associative-embedding grouping -- MPPEHeatmapParser.match_by_tag
// (/root/reference/src/keypoints/grouping.py:85-145), py_max_match (:55-59, munkres 1.1.4
// Munkres.compute) and the empty-scene fallback of parse (:262-269).
//
// One CTA of four warps per image.  The 17 joint steps are strictly sequential and every step
// works on at most 32 detections x 32 persons, so the kernel is latency-bound by design
// (bench.py reports microseconds per image instead of a bandwidth fraction).  All four warps run
// the same control flow on replicated registers (lane r = detection r / person r / matrix row r);
// the float64 work is split between them: the cost matrix by (detection, person) pair, the
// Hungarian solver's matrix by column (warp w keeps columns 8w..8w+7 of every row in registers),
// exchanged through shared memory at the two points of steps 1 and 6 where a row needs all its
// columns.  Only warp 0 writes the tag lists and the output.
//
// Exactness notes (SURVEY.md App. A.5 / B):
//   * det_thr and tag_thr are compared in float64; costs are float64:
//       cost = rint(sqrt(sum_e (tag_e - mean_e)^2)) * 100 - score     (no contraction anywhere)
//   * the mean tag of a person is numpy's float32 np.mean over its tag list (pairwise-8 for
//     E = 1, sequential for E = 2);
//   * persons are dict entries keyed by the float32 value of tag[0]: an equal key overwrites that
//     person's joint and resets its tag list; only the first M persons are match candidates or
//     outputs, later ones are counted but not stored;
//   * the Hungarian solver replays munkres 1.1.4 step by step: lane r owns matrix row r and a
//     32-bit mask of its zero entries, so "find the last uncovered zero in cyclic order" is bit
//     arithmetic; the (C + m) - m update order of step 6 is kept.
//   * library policy, not the reference's: a cost that is not finite or whose magnitude is >= 2^63
//     is replaced by 1e10 (grouping.py:126-128's "cannot match" value) before the solver runs, and
//     flags bit 1 is set.  On such a row munkres 1.1.4 never terminates (a NaN row never gets a
//     zero; step 6's sys.maxsize sentinel stops making zeros above 2^63).  With finite costs below
//     2^63 every step 6 makes a zero, so an augmentation needs at most n step-6 calls; the solver
//     still stops after n (n + 1) of them, sets bit 1 and leaves the step's detections unmatched.
#include "common.cuh"
#ifdef HPD_GROUP_PROFILE
#include <cstdio>
#endif

namespace hpd {

namespace {

constexpr int NP = HPD_MAX_PEOPLE;      // 32
constexpr int CS = NP + 1;              // padded row stride of the float64 matrices

// -DHPD_GROUP_PROFILE: block 0 prints clock64() totals per phase (development aid, off by default)
#ifdef HPD_GROUP_PROFILE
__device__ long long gp_acc[12];
#define GP_BEGIN(t) const long long t = clock64()
#define GP_END(slot, t) do { if (blockIdx.x == 0 && threadIdx.x == 0) gp_acc[slot] += clock64() - (t); } while (0)
#define GP_COUNT(slot) do { if (blockIdx.x == 0 && threadIdx.x == 0) gp_acc[slot] += 1; } while (0)
#else
#define GP_BEGIN(t)
#define GP_END(slot, t)
#define GP_COUNT(slot)
#endif

constexpr int kGroupWarps = 4;
constexpr int CW = NP / kGroupWarps;    // matrix columns per warp
constexpr int TL = HPD_MAX_KPTS * HPD_MAX_EMB + 1;   // odd person stride: lanes hit distinct banks
constexpr int kSolverCapped = -2;       // munkres_cta's result on every lane when its step-6 cap was reached

struct GroupSmem {
  double C[NP][CS];                     // cost matrix as built (real detections x real persons)
  double D[NP][CS];                     // saved distances (diff_saved)
  double pmin[kGroupWarps][NP];         // per-warp partial minima
  unsigned pz[kGroupWarps][NP];         // per-warp partial zero masks
  float keytmp[kGroupWarps][NP];        // per-warp scratch: keys of the persons created in a step
  float taglist[NP * TL];               // person p's tag list: taglist[p*TL + j*HPD_MAX_EMB + e]
};

__device__ __forceinline__ double warp_min_double(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double w = __shfl_xor_sync(kFull, v, o);
    v = (w < v) ? w : v;
  }
  return v;
}

// same for values known to be >= +0 (their bit patterns order like unsigned integers): two
// warp-reduce instructions instead of five shuffle rounds
__device__ __forceinline__ double warp_min_nonneg(double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  const unsigned hi = (unsigned)(u >> 32), lo = (unsigned)u;
  const unsigned mh = __reduce_min_sync(kFull, hi);
  const unsigned ml = __reduce_min_sync(kFull, hi == mh ? lo : 0xffffffffu);
  return __longlong_as_double((long long)(((unsigned long long)mh << 32) | ml));
}

__device__ __forceinline__ double min4(const double (*pm)[NP], int i) {
  const double a = pm[0][i], b = pm[1][i], c = pm[2][i], d = pm[3][i];
  const double ab = (b < a) ? b : a, cd = (d < c) ? d : c;
  return (cd < ab) ? cd : ab;
}

// munkres 1.1.4 Munkres.compute on the n x n matrix: rows < nr and columns < G come from sm.C,
// columns G..n-1 of those rows are 1e10 (grouping.py:126-128), rows nr..n-1 are munkres' zero
// padding.  Returns the starred column of this lane's row (valid for lane < n), or kSolverCapped on
// every lane after n (n + 1) step-6 calls.  Called by all four warps; contains __syncthreads().
__device__ int munkres_cta(GroupSmem& sm, int nr, int G, int n, int lane, int w) {
  const unsigned nmask = (n >= 32) ? kFull : ((1u << n) - 1u);
  const int cap = n * (n + 1);
  int n6 = 0;
  const int cb = w * CW;
  const double kInf = __longlong_as_double(0x7ff0000000000000ll);
  double c[CW];
#pragma unroll
  for (int jj = 0; jj < CW; ++jj) {
    const int j = cb + jj;
    c[jj] = (lane < nr) ? ((j < G) ? sm.C[lane][j] : 1e10) : 0.0;
  }
  unsigned zmask = 0;
  GP_BEGIN(t_s1);
  // step 1: subtract the row minimum
  {
    double m = kInf;
#pragma unroll
    for (int jj = 0; jj < CW; ++jj)
      if (cb + jj < n && c[jj] < m) m = c[jj];
    sm.pmin[w][lane] = m;
    __syncthreads();
    m = min4(sm.pmin, lane);
    unsigned z = 0;
#pragma unroll
    for (int jj = 0; jj < CW; ++jj) {
      c[jj] = __dsub_rn(c[jj], m);
      if (c[jj] == 0.0) z |= 1u << (cb + jj);
    }
    sm.pz[w][lane] = z;
    __syncthreads();
    if (lane < n) zmask = (sm.pz[0][lane] | sm.pz[1][lane] | sm.pz[2][lane] | sm.pz[3][lane]) & nmask;
  }
  GP_END(0, t_s1);
  GP_BEGIN(t_s2);
  // step 2: rows ascending, star the first zero in an uncovered column
  int star = -1;
  unsigned colcov = 0, rowcov = 0;
  // (rows >= n have an empty mask; unrolled so that the shuffles do not sit on the colcov chain)
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const unsigned c = __shfl_sync(kFull, zmask, i) & ~colcov;
    const unsigned low = c & (0u - c);
    if (lane == i && low) star = __ffs(low) - 1;
    colcov |= low;
  }
  colcov = 0;
  int prime = -1;
  GP_END(1, t_s2);
  while (true) {
    // step 3: cover starred columns
    colcov |= __reduce_or_sync(kFull, (lane < n && star >= 0) ? (1u << star) : 0u);
    if (__popc(colcov) >= n) break;
    int z0r = 0, z0c = 0;
    while (true) {
      // step 4
      int row = 0, col = 0;
      bool augment = false;
      GP_BEGIN(t_s4);
      while (true) {
        GP_COUNT(11);
        const unsigned cand = (lane < n && !((rowcov >> lane) & 1u)) ? (zmask & ~colcov & nmask) : 0u;
        const unsigned rows_with = __ballot_sync(kFull, cand != 0u);
        if (!rows_with) break;
        const unsigned hi = rows_with >> row;
        const int r = hi ? (row + __ffs(hi) - 1) : (__ffs(rows_with) - 1);
        const unsigned c = __shfl_sync(kFull, cand, r);
        const unsigned low = c & ((1u << col) - 1u);
        const int cc = low ? (31 - __clz(low)) : (31 - __clz(c));
        if (lane == r) prime = cc;
        const int sc = __shfl_sync(kFull, star, r);
        row = r;
        if (sc >= 0) {
          col = sc;
          rowcov |= 1u << r;
          colcov &= ~(1u << sc);
        } else {
          z0r = r;
          z0c = cc;
          augment = true;
          break;
        }
      }
      GP_END(2, t_s4);
      if (augment) break;
      GP_BEGIN(t_s6);
      GP_COUNT(10);
      // step 6 (the count is uniform over the CTA, so every thread leaves here together)
      if (++n6 > cap) return kSolverCapped;
      double m = 9.223372036854775807e18;
      if (lane < n && !((rowcov >> lane) & 1u)) {
#pragma unroll
        for (int jj = 0; jj < CW; ++jj)
          if (cb + jj < n && !((colcov >> (cb + jj)) & 1u) && m > c[jj]) m = c[jj];
      }
      // after step 1 every entry is >= +0; the sign test keeps the exact path for anything else
      m = __any_sync(kFull, m < 0.0 || m != m) ? warp_min_double(m) : warp_min_nonneg(m);
      if (lane == 0) sm.pmin[w][0] = m;
      __syncthreads();
      m = min4(sm.pmin, 0);
      {
        const bool rc = (rowcov >> lane) & 1u;
        unsigned z = 0;
#pragma unroll
        for (int jj = 0; jj < CW; ++jj) {
          double v = c[jj];
          if (rc) v = __dadd_rn(v, m);
          if (!((colcov >> (cb + jj)) & 1u)) v = __dsub_rn(v, m);
          c[jj] = v;
          if (v == 0.0) z |= 1u << (cb + jj);
        }
        sm.pz[w][lane] = z;
      }
      __syncthreads();
      zmask = (lane < n) ? ((sm.pz[0][lane] | sm.pz[1][lane] | sm.pz[2][lane] | sm.pz[3][lane]) & nmask) : 0u;
      GP_END(3, t_s6);
    }
    // step 5: augment along the alternating star/prime path from Z0
    {
      GP_BEGIN(t_s5);
      int r = z0r, c = z0c;
      while (true) {
        const unsigned b = __ballot_sync(kFull, lane < n && star == c);
        if (lane == r) star = c;
        if (!b) break;
        const int r2 = __ffs(b) - 1;
        c = __shfl_sync(kFull, prime, r2);
        r = r2;
      }
      rowcov = colcov = 0;
      prime = -1;
      GP_END(4, t_s5);
    }
  }
  return star;
}

__global__ void __launch_bounds__(32 * kGroupWarps) group_kernel(const float* __restrict__ scores_k,
                                                                 const int32_t* __restrict__ coords_k,
                                                                 const float* __restrict__ tags_k, int K, int M,
                                                                 int E, double det_thr, double tag_thr,
                                                                 const HpdParams prm, float* __restrict__ poses,
                                                                 int32_t* __restrict__ n_person,
                                                                 int32_t* __restrict__ flags) {
  __shared__ GroupSmem sm;
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int b = blockIdx.x;
  const int D = 3 + E;
  const float* sc_b = scores_k + (size_t)b * K * M;
  const int32_t* co_b = coords_k + (size_t)b * K * M * 2;
  const float* tg_b = tags_k + (size_t)b * K * M * E;
  float* out = poses + (size_t)b * M * K * D;
  for (int i = threadIdx.x; i < M * K * D; i += 32 * kGroupWarps) out[i] = 0.f;

  int fl = 0;         // flags[b], uniform
  int P = 0;          // persons stored (<= M), uniform
  int Ptotal = 0;     // persons created, uniform
  float key = 0.f;    // lane p: dict key of person p
  int ntag = 0;       // lane p: length of person p's tag list

  // lane r holds the rank-r candidate of a joint; loaded one joint step ahead of its use
  struct Cand { float score, x, y, t0, t1; };
  auto load_cand = [&](int it) {
    Cand c{0.f, 0.f, 0.f, 0.f, 0.f};
    if (it < K && lane < M) {
      const int i = prm.joints_order[it] * M + lane;
      c.score = sc_b[i];
      c.x = (float)co_b[2 * i + 0];
      c.y = (float)co_b[2 * i + 1];
      c.t0 = tg_b[(size_t)i * E];
      c.t1 = (E > 1) ? tg_b[(size_t)i * E + 1] : 0.f;
    }
    return c;
  };
  Cand nxt = load_cand(0);

  for (int it = 0; it < K; ++it) {
    // warp 0's tag-list / output writes of the previous step (and the zero fill) are visible to
    // everyone from here on, and nobody still reads the previous step's D
    __syncthreads();
    GP_BEGIN(t_pro);
    const int k = prm.joints_order[it];
    Cand cur = nxt;
    nxt = load_cand(it + 1);
    const unsigned rowmask = __ballot_sync(kFull, lane < M && (double)cur.score > det_thr);
    const int nr = __popc(rowmask);
    if (nr == 0) continue;
    const unsigned detmask = (nr >= 32) ? kFull : ((1u << nr) - 1u);
    if (rowmask != detmask) {
      // scores not sorted (hpd_group called on foreign data): compact the detections to lanes 0..nr-1
      const int src = (lane < nr) ? (int)__fns(rowmask, 0, lane + 1) : 0;
      cur.score = __shfl_sync(kFull, cur.score, src);
      cur.x = __shfl_sync(kFull, cur.x, src);
      cur.y = __shfl_sync(kFull, cur.y, src);
      cur.t0 = __shfl_sync(kFull, cur.t0, src);
      cur.t1 = __shfl_sync(kFull, cur.t1, src);
    }
    // lane a < nr now owns the a-th detection above threshold
    const float a_score = cur.score, a_x = cur.x, a_y = cur.y, a_t0 = cur.t0, a_t1 = cur.t1;
    GP_END(9, t_pro);

    // writes detection a into person p (warp 0's lane a does the stores)
    auto put_joint = [&](int a, int p) {
      if (w == 0 && lane == a) {
        float* d = out + ((size_t)p * K + k) * D;
        d[0] = a_x; d[1] = a_y; d[2] = a_score; d[3] = a_t0;
        if (E > 1) d[4] = a_t1;
      }
    };
    auto put_tag = [&](int a, int p, int j) {
      if (w == 0 && lane == a) {
        sm.taglist[p * TL + j * HPD_MAX_EMB + 0] = a_t0;
        sm.taglist[p * TL + j * HPD_MAX_EMB + 1] = a_t1;
      }
    };
    // dict.setdefault(key)[idx] = joint ; tag_dict[key] = [tag]   (grouping.py:109-111,141-143)
    auto new_or_collide = [&](int a) {
      const float t0 = __shfl_sync(kFull, a_t0, a);
      const unsigned hit = __ballot_sync(kFull, lane < P && key == t0);
      int p;
      if (hit) {
        p = __ffs(hit) - 1;
      } else {
        ++Ptotal;
        if (P < M) {
          p = P++;
          if (lane == p) key = t0;
        } else {
          p = -1;   // person beyond the first M: never read again
        }
      }
      if (p >= 0) {
        put_joint(a, p);
        put_tag(a, p, 0);
        if (lane == p) ntag = 1;
      }
    };

    const int G = P;      // match candidates; 0 until the first person exists (grouping.py:107)
    int star = -1;
    if (G > 0) {
      const int n = max(G, nr);
      GP_BEGIN(t_mean);
      // mean tag per existing person (grouping.py:114)
      float mean0 = 0.f, mean1 = 0.f;
      if (lane < G) {
        float mv[HPD_MAX_EMB];
        np_mean_vectors(&sm.taglist[lane * TL], ntag, E, HPD_MAX_EMB, mv);
        mean0 = mv[0];
        mean1 = (E > 1) ? mv[1] : 0.f;
      }
      GP_END(5, t_mean);
      GP_BEGIN(t_cost);
      // cost matrix (grouping.py:116-128): the nr x G real pairs are spread over the four warps,
      // four independent pairs per thread and round (the float64 sqrt chains overlap); the 1e10
      // columns and zero rows are synthesised when the solver loads its registers
      bool guarded = false;
      {
        constexpr int U = 4;
        const int npairs = nr * G;
        const unsigned inv = (65536u + G - 1) / G;         // i / G == (i * inv) >> 16 for i < 2048
        for (int i0 = 0; i0 < npairs; i0 += 32 * U * kGroupWarps) {
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int i = i0 + (u * kGroupWarps + w) * 32 + lane;
            const int a = min((int)(((unsigned)i * inv) >> 16), nr - 1);
            const int p = (i < npairs) ? i - a * G : 0;
            const float t0 = __shfl_sync(kFull, a_t0, a), t1 = __shfl_sync(kFull, a_t1, a);
            const float sc_a = __shfl_sync(kFull, a_score, a);
            const float m0 = __shfl_sync(kFull, mean0, p), m1 = __shfl_sync(kFull, mean1, p);
            if (i < npairs) {
              const double d0 = __dsub_rn((double)t0, (double)m0);
              double s = __dmul_rn(d0, d0);
              if (E > 1) {
                const double d1 = __dsub_rn((double)t1, (double)m1);
                s = __dadd_rn(s, __dmul_rn(d1, d1));
              }
              const double dn = __dsqrt_rn(s);
              sm.D[a][p] = dn;
              double cst = __dsub_rn(__dmul_rn(rint(dn), 100.0), (double)sc_a);
              if (!(fabs(cst) < 9.223372036854775808e18)) {   // NaN, +-inf, |cost| >= 2^63
                cst = 1e10;
                guarded = true;
              }
              sm.C[a][p] = cst;
            }
          }
        }
      }
      if (__syncthreads_or(guarded)) fl |= 2;
      GP_END(6, t_cost);
      GP_BEGIN(t_mk);
      star = munkres_cta(sm, nr, G, n, lane, w);
      if (star == kSolverCapped) {
        fl |= 2;
        star = -1;
      }
      GP_END(7, t_mk);
    }

    // grouping.py:131-143 (and :107-111 when there is nobody to match against)
    GP_BEGIN(t_asg);
    const bool is_det = lane < nr;
    const bool ok = is_det && star >= 0 && star < G && sm.D[lane][star] < tag_thr;
    const unsigned okmask = __ballot_sync(kFull, ok);
    const unsigned newmask = detmask & ~okmask;
    const bool is_new = (newmask >> lane) & 1u;
    // The detections can be placed all at once unless a new one has the dict key (float32 tag[0])
    // of an existing person or of another new one -- then order matters and the loop below runs.
    bool ordered = false;
    if (newmask) {
      const unsigned same = __match_any_sync(kFull, __float_as_uint(__fadd_rn(a_t0, 0.0f)));
      bool clash = (same & newmask & ~(1u << lane)) != 0u;
#pragma unroll
      for (int p = 0; p < 32; ++p) {
        const float kp = __shfl_sync(kFull, key, p);
        clash |= (p < P) & (kp == a_t0);
      }
      ordered = __any_sync(kFull, is_new && clash);
    }
    if (!ordered) {
      const int nt = __shfl_sync(kFull, ntag, ok ? star : 0);
      const int rank = __popc(newmask & ((1u << lane) - 1u));
      const int cnt = __popc(newmask);
      const int Pn = min(M, P + cnt);
      if (ok) {
        put_joint(lane, star);
        put_tag(lane, star, nt);
      } else if (is_new && P + rank < M) {
        put_joint(lane, P + rank);
        put_tag(lane, P + rank, 0);
      }
      const unsigned got = __reduce_or_sync(kFull, ok ? (1u << star) : 0u);
      if ((got >> lane) & 1u) ntag += 1;
      if (cnt) {
        if (is_new) sm.keytmp[w][rank] = a_t0;
        __syncwarp();
        if (lane >= P && lane < Pn) {
          key = sm.keytmp[w][lane - P];
          ntag = 1;
        }
        __syncwarp();
      }
      P = Pn;
      Ptotal += cnt;
    } else {
      for (int a = 0; a < nr; ++a) {
        if ((okmask >> a) & 1u) {
          const int c = __shfl_sync(kFull, star, a);
          const int nt = __shfl_sync(kFull, ntag, c);
          put_joint(a, c);
          put_tag(a, c, nt);
          if (lane == c) ntag = nt + 1;
        } else {
          new_or_collide(a);
        }
      }
    }
    GP_END(8, t_asg);
  }
#ifdef HPD_GROUP_PROFILE
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    printf("group profile (cycles, image 0): step1 %lld step2 %lld step4 %lld step6 %lld step5 %lld | means %lld cost %lld "
           "munkres %lld assign %lld prologue %lld | step6 calls %lld step4 iterations %lld persons %d\n",
           gp_acc[0], gp_acc[1], gp_acc[2], gp_acc[3], gp_acc[4], gp_acc[5], gp_acc[6], gp_acc[7], gp_acc[8],
           gp_acc[9], gp_acc[10], gp_acc[11], Ptotal);
    for (int i = 0; i < 12; ++i) gp_acc[i] = 0;
  }
#endif

  if (w != 0) return;
  if (Ptotal == 0) {
    // grouping.py:262-269: one pseudo-person from the best candidate of every joint, score := 0.01
    fl |= 1;
    P = 1;
    for (int k = lane; k < K; k += 32) {
      float* d = out + (size_t)k * D;
      d[0] = (float)co_b[(k * M) * 2 + 0];
      d[1] = (float)co_b[(k * M) * 2 + 1];
      d[2] = 0.01f;
      for (int e = 0; e < E; ++e) {
        const float t = tg_b[(size_t)(k * M) * E + e];
        d[3 + e] = (t != t) ? 0.f : t;
      }
    }
  }
  if (lane == 0) {
    n_person[b] = P;
    flags[b] = fl;
  }
}

}  // namespace

int launch_group(const HpdParams* p, const HpdBuffers* buf, cudaStream_t st) {
  if (!buf->scores_k || !buf->coords_k || !buf->tags_k || !buf->poses || !buf->n_person || !buf->flags) {
    set_error("hpd_group: scores_k, coords_k, tags_k, poses, n_person, flags are required");
    return HPD_EINVAL;
  }
  group_kernel<<<p->batch, 32 * kGroupWarps, 0, st>>>(buf->scores_k, buf->coords_k, buf->tags_k, p->num_kpts, p->max_people, p->emb,
                                        p->det_thr, p->tag_thr, *p, buf->poses, buf->n_person, buf->flags);
  count_launch();
  return check_launch("group_kernel");
}

}  // namespace hpd
