// COCO keypoint evaluation on the device: pycocotools cocoeval.py, iouType "keypoints" (computeOks, evaluateImg,
// accumulate) for one category.  The CPU oracle is oracle/coco_eval_oracle.py, which keeps pycocotools' expressions.
//
//   coco_image_kernel       one CTA per image: stable score rank of each detection (mergesort on -score), the
//                           maxDets cut, detection areas (loadRes), the OKS matrix (computeOks) and the greedy
//                           matching of every (area range, threshold) pair, one thread each (evaluateImg).  Writes one
//                           code per (area, threshold, image, rank) and the non-ignored gt count per (area, image).
//   cub radix sort          the kept detections of all images in (image, rank) order, sorted by score descending and
//                           stably: accumulate's np.argsort(-dtScores, kind='mergesort').
//   coco_accumulate_kernel  one CTA per (area, threshold): tp / fp prefix sums in that order, recall and precision
//                           with accumulate's operations, the precision envelope (a suffix maximum) and the
//                           searchsorted lookup of every recall threshold.
//
// Every float64 operation is spelled out (__dadd_rn, ...) and the library builds with -fmad=false.  The one
// operation that is not exact is exp() in the OKS (CUDA's is within 1 ulp; NumPy's differs from libm's in the last
// bit for a few percent of arguments), so OKS values agree within a few ulp and everything after them exactly as long
// as no OKS sits within that distance of a decision.
#include <cub/cub.cuh>

#include "common.cuh"

namespace hpd {
namespace {

constexpr int kImgThreads = 256;
constexpr int kAccThreads = 512;
constexpr int kGtWords = HPD_COCO_MAX_PER_IMAGE / 32;
constexpr int kMaxPairs = HPD_COCO_MAX_AREAS * HPD_COCO_MAX_IOU_THRS;

struct CocoWs {
  double* oks;          // [I][md][G] (outs->oks when given)
  uint8_t* codes;       // [A][T][I][md] (outs->codes when given)
  int32_t* npig_img;    // [A][I]
  int32_t* kept_n;      // [I] min(n, md)
  double* slot_score;   // [I][md] score of the detection of rank r of image i
  uint64_t *keys_in, *keys_out;   // order keys of the slots (0: no detection)
  int32_t *vals_in, *vals_out;    // slot indices
  int32_t* tp_cum;      // [A*T][I*md]
  double* env;          // [A*T][I*md] precision, then its envelope
  void* sort_tmp;
  size_t sort_bytes;
  size_t total;
};

size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// Carves the workspace (base == nullptr: only sizes).  The sort's scratch size comes from CUB itself.
int coco_workspace(const HpdCocoEvalParams* p, uint8_t* base, CocoWs* w) {
  const size_t I = (size_t)p->num_images, md = (size_t)p->max_dets, G = (size_t)p->max_gts;
  const size_t AT = (size_t)p->num_areas * p->num_iou_thrs, N = I * md;
  size_t sort_bytes = 0;
  const cudaError_t e = cub::DeviceRadixSort::SortPairsDescending(
      nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr,
      (int)N, 0, 64);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hpd_coco_eval: sort scratch size query failed: %s", cudaGetErrorString(e));
    return HPD_ECUDA;
  }
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* q = base ? base + off : nullptr;
    off += align256(bytes);
    return q;
  };
  w->oks = (double*)take(N * G * 8);
  w->codes = take(AT * N);
  w->npig_img = (int32_t*)take((size_t)p->num_areas * I * 4);
  w->kept_n = (int32_t*)take(I * 4);
  w->slot_score = (double*)take(N * 8);
  w->keys_in = (uint64_t*)take(N * 8);
  w->keys_out = (uint64_t*)take(N * 8);
  w->vals_in = (int32_t*)take(N * 4);
  w->vals_out = (int32_t*)take(N * 4);
  w->tp_cum = (int32_t*)take(AT * N * 4);
  w->env = (double*)take(AT * N * 8);
  w->sort_tmp = take(sort_bytes);
  w->sort_bytes = sort_bytes;
  w->total = off;
  return HPD_OK;
}

// Descending order of these keys is descending score order with -0.0 == +0.0 (NumPy's comparison); 0 sorts last.
__device__ __forceinline__ uint64_t score_key(double s) {
  if (s == 0.0) s = 0.0;
  const uint64_t u = (uint64_t)__double_as_longlong(s);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// np.max((z, v), axis=0) for one element: maximum(0, v) keeps the first operand unless the second is larger
__device__ __forceinline__ double max0(double v) { return 0.0 >= v ? 0.0 : v; }

// computeOks for one (detection, gt): e = (dx**2 + dy**2) / vars / (area + np.spacing(1)) / 2 over the gt's visible
// joints (all K joints with the distance to the gt box grown by its size when none is visible), then
// np.sum(np.exp(-e)) / len(e) with NumPy's pairwise-8 summation order (n <= 32 < its 128-element block).
__device__ __forceinline__ double oks_pair(const double* xd, const double* yd, const double* gk, const double* bb,
                                           double garea, const double* vars, int K) {
  int k1 = 0;
  for (int k = 0; k < K; ++k) k1 += gk[3 * k + 2] > 0.0;
  const double x0 = __dsub_rn(bb[0], bb[2]), x1 = __dadd_rn(bb[0], __dmul_rn(bb[2], 2.0));
  const double y0 = __dsub_rn(bb[1], bb[3]), y1 = __dadd_rn(bb[1], __dmul_rn(bb[3], 2.0));
  const double den = __dadd_rn(garea, 0x1p-52);
  const int n = k1 > 0 ? k1 : K;
  NpSumF64 acc(n);
  for (int k = 0; k < K; ++k) {
    double dx, dy;
    if (k1 > 0) {
      if (!(gk[3 * k + 2] > 0.0)) continue;
      dx = __dsub_rn(xd[k], gk[3 * k]);
      dy = __dsub_rn(yd[k], gk[3 * k + 1]);
    } else {
      dx = __dadd_rn(max0(__dsub_rn(x0, xd[k])), max0(__dsub_rn(xd[k], x1)));
      dy = __dadd_rn(max0(__dsub_rn(y0, yd[k])), max0(__dsub_rn(yd[k], y1)));
    }
    double e = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    e = __ddiv_rn(__ddiv_rn(__ddiv_rn(e, vars[k]), den), 2.0);
    acc.add(exp(-e));
  }
  return __ddiv_rn(acc.sum(), (double)n);
}

__global__ void __launch_bounds__(kImgThreads) coco_image_kernel(HpdCocoEvalParams p, HpdCocoDets dets, HpdCocoGts gts,
                                                                 CocoWs w) {
  __shared__ double s_score[HPD_COCO_MAX_PER_IMAGE];
  __shared__ double s_x[HPD_MAX_PEOPLE][HPD_MAX_KPTS], s_y[HPD_MAX_PEOPLE][HPD_MAX_KPTS];
  __shared__ double s_darea[HPD_MAX_PEOPLE];
  __shared__ int s_kept[HPD_MAX_PEOPLE];
  __shared__ uint32_t s_ig[HPD_COCO_MAX_AREAS][kGtWords], s_crowd[kGtWords];
  __shared__ uint32_t s_gtm[kMaxPairs][kGtWords];

  const int i = blockIdx.x, tid = threadIdx.x;
  const int K = p.num_kpts, md = p.max_dets, G = p.max_gts, A = p.num_areas, T = p.num_iou_thrs, I = p.num_images;
  const int ps = dets.person_stride;

  const long long row = dets.row_offset[i];
  int n = 0;
  const double* coco = nullptr;
  if (row >= 0) {
    const uint8_t* r = dets.base + row;
    n = min(max(*reinterpret_cast<const int32_t*>(r + dets.off_count), 0), dets.max_per_row);
    coco = reinterpret_cast<const double*>(r + dets.off_coco);
  }
  const int ng = min(max(gts.n_gt[i], 0), G);
  const int nk = min(n, md);

  for (int j = tid; j < n; j += blockDim.x) s_score[j] = coco[(size_t)j * ps + 3 * K];
  for (int q = tid; q < kGtWords; q += blockDim.x) {
    s_crowd[q] = 0;
    for (int a = 0; a < HPD_COCO_MAX_AREAS; ++a) s_ig[a][q] = 0;
    for (int at = 0; at < kMaxPairs; ++at) s_gtm[at][q] = 0;
  }
  __syncthreads();

  // rank of detection j: mergesort of -score keeps equal scores in list order
  for (int j = tid; j < n; j += blockDim.x) {
    const double s = s_score[j];
    int rank = 0;
    for (int q = 0; q < n; ++q) {
      const double o = s_score[q];
      rank += (o > s) || (o == s && q < j);
    }
    if (rank < md) s_kept[rank] = j;
  }
  // _ignore of every gt for every area range, crowd flags
  for (int g = tid; g < ng; g += blockDim.x) {
    const size_t ig = (size_t)i * G + g;
    const double ar = gts.area[ig];
    const uint32_t bit = 1u << (g & 31);
    for (int a = 0; a < A; ++a)
      if (gts.ignore[ig] || ar < p.area_rng[a][0] || ar > p.area_rng[a][1]) atomicOr(&s_ig[a][g >> 5], bit);
    if (gts.iscrowd[ig]) atomicOr(&s_crowd[g >> 5], bit);
  }
  __syncthreads();

  for (int r = tid; r < md; r += blockDim.x) {
    const size_t slot = (size_t)i * md + r;
    const double s = r < nk ? s_score[s_kept[r]] : 0.0;
    w.slot_score[slot] = s;
    w.keys_in[slot] = r < nk ? score_key(s) : 0ull;
    w.vals_in[slot] = (int32_t)slot;
  }
  if (tid == 0) w.kept_n[i] = nk;
  for (int a = tid; a < A; a += blockDim.x) {
    int ignored = 0;
    for (int q = 0; q < kGtWords; ++q) ignored += __popc(s_ig[a][q]);
    w.npig_img[(size_t)a * I + i] = ng - ignored;
  }
  for (int idx = tid; idx < nk * K; idx += blockDim.x) {
    const int r = idx / K, k = idx % K;
    const double* d = coco + (size_t)s_kept[r] * ps;
    s_x[r][k] = d[3 * k];
    s_y[r][k] = d[3 * k + 1];
  }
  __syncthreads();

  // loadRes: area = (x1 - x0) * (y1 - y0) from the min and max over all K joints
  for (int r = tid; r < nk; r += blockDim.x) {
    double x0 = s_x[r][0], x1 = x0, y0 = s_y[r][0], y1 = y0;
    for (int k = 1; k < K; ++k) {
      const double x = s_x[r][k], y = s_y[r][k];
      x0 = x < x0 ? x : x0;
      x1 = x > x1 ? x : x1;
      y0 = y < y0 ? y : y0;
      y1 = y > y1 ? y : y1;
    }
    s_darea[r] = __dmul_rn(__dsub_rn(x1, x0), __dsub_rn(y1, y0));
  }
  double* oks = w.oks + (size_t)i * md * G;
  for (int idx = tid; idx < md * G; idx += blockDim.x) {
    const int r = idx / G, g = idx % G;
    double v = 0.0;
    if (r < nk && g < ng) {
      const size_t ig = (size_t)i * G + g;
      v = oks_pair(s_x[r], s_y[r], gts.kpts + ig * K * 3, gts.bbox + ig * 4, gts.area[ig], p.kpt_vars, K);
    }
    oks[idx] = v;
  }
  __syncthreads();   // the OKS matrix is read back below by other threads of this CTA

  // evaluateImg: one thread per (area range, threshold), detections in rank order.  gts are visited in the order of
  // the stable partition by _ignore: the non-ignored ones, then -- only if none of them matched -- the ignored ones
  // (the `break` of a held non-ignored match on the first ignored gt that is not skipped).
  if (tid < A * T) {
    const int a = tid / T, t = tid % T;
    const double lo = p.area_rng[a][0], hi = p.area_rng[a][1];
    const double bar = p.iou_thrs[t] <= 1.0 - 1e-10 ? p.iou_thrs[t] : 1.0 - 1e-10;   // min([t, 1-1e-10])
    uint32_t* gtm = s_gtm[tid];
    const uint32_t* igw = s_ig[a];
    uint8_t* codes = w.codes + ((size_t)tid * I + i) * md;
    for (int r = 0; r < nk; ++r) {
      double best = bar;
      int m = -1;
      for (int phase = 0; phase < 2 && m < 0; ++phase) {
        for (int g = 0; g < ng; ++g) {
          const uint32_t bit = 1u << (g & 31);
          if (((igw[g >> 5] & bit) != 0) != (phase == 1)) continue;
          if ((gtm[g >> 5] & bit) && !(s_crowd[g >> 5] & bit)) continue;
          const double v = oks[r * G + g];
          if (v < best) continue;
          best = v;
          m = g;
        }
      }
      uint8_t code;
      if (m >= 0) {
        gtm[m >> 5] |= 1u << (m & 31);
        code = (igw[m >> 5] >> (m & 31)) & 1 ? HPD_COCO_IGNORED : HPD_COCO_TP;
      } else {
        code = (s_darea[r] < lo || s_darea[r] > hi) ? HPD_COCO_IGNORED : HPD_COCO_FP;
      }
      codes[r] = code;
    }
    for (int r = nk; r < md; ++r) codes[r] = HPD_COCO_ABSENT;
  }
}

struct MaxOp {
  __device__ __forceinline__ double operator()(double a, double b) const { return b > a ? b : a; }
};

__global__ void __launch_bounds__(kAccThreads) coco_accumulate_kernel(HpdCocoEvalParams p, CocoWs w,
                                                                      HpdCocoEvalOutputs outs) {
  using Reduce = cub::BlockReduce<long long, kAccThreads>;
  using ScanI = cub::BlockScan<int, kAccThreads>;
  using ScanD = cub::BlockScan<double, kAccThreads>;
  __shared__ union {
    typename Reduce::TempStorage reduce;
    typename ScanI::TempStorage scan_i;
    typename ScanD::TempStorage scan_d;
  } tmp;
  __shared__ long long s_tot[2];
  __shared__ int s_pi[HPD_COCO_MAX_REC_THRS];

  const int at = blockIdx.x, a = at / p.num_iou_thrs, t = at % p.num_iou_thrs, tid = threadIdx.x;
  const int I = p.num_images, md = p.max_dets, R = p.num_rec_thrs, A = p.num_areas;
  const size_t cap = (size_t)I * md;

  long long kept = 0, pig = 0;
  for (int i = tid; i < I; i += blockDim.x) {
    kept += w.kept_n[i];
    pig += w.npig_img[(size_t)a * I + i];
  }
  kept = Reduce(tmp.reduce).Sum(kept);
  __syncthreads();
  pig = Reduce(tmp.reduce).Sum(pig);
  if (tid == 0) {
    s_tot[0] = kept;
    s_tot[1] = pig;
  }
  __syncthreads();
  const int N = (int)s_tot[0];
  const long long npig = s_tot[1];
  if (t == 0 && tid == 0 && outs.npig) outs.npig[a] = npig;
  if (npig == 0) {   // accumulate skips this (area, threshold): the arrays keep their -1
    for (int r = tid; r < R; r += blockDim.x) {
      outs.precision[((size_t)t * R + r) * A + a] = -1.0;
      outs.scores[((size_t)t * R + r) * A + a] = -1.0;
    }
    if (tid == 0) outs.recall[(size_t)t * A + a] = -1.0;
    return;
  }
  const uint8_t* codes = w.codes + (size_t)at * cap;
  int32_t* tp_cum = w.tp_cum + (size_t)at * cap;
  double* env = w.env + (size_t)at * cap;
  const double dnpig = (double)npig;

  // tp / fp cumulative sums in global score order; pr = tp / (fp + tp + np.spacing(1))
  int carry_tp = 0, carry_fp = 0;
  for (int base = 0; base < N; base += blockDim.x) {
    const int j = base + tid;
    const int c = j < N ? codes[w.vals_out[j]] : HPD_COCO_ABSENT;
    const int packed = (c == HPD_COCO_TP ? 1 << 16 : 0) | (c == HPD_COCO_FP ? 1 : 0);   // <= kAccThreads per chunk each
    int incl, total;
    ScanI(tmp.scan_i).InclusiveSum(packed, incl, total);
    const int tp = carry_tp + (incl >> 16), fp = carry_fp + (incl & 0xffff);
    if (j < N) {
      tp_cum[j] = tp;
      env[j] = __ddiv_rn((double)tp, __dadd_rn(__dadd_rn((double)fp, (double)tp), 0x1p-52));
    }
    carry_tp += total >> 16;
    carry_fp += total & 0xffff;
    __syncthreads();
  }
  // envelope: the right-to-left walk `if pr[i] > pr[i-1]: pr[i-1] = pr[i]` is the suffix maximum
  double carry = -INFINITY;
  for (int end = N; end > 0; end -= blockDim.x) {
    const int j = end - 1 - tid;
    const double v = j >= 0 ? env[j] : -INFINITY;
    double s, total;
    ScanD(tmp.scan_d).InclusiveScan(v, s, MaxOp(), total);
    if (j >= 0) env[j] = MaxOp()(s, carry);
    carry = MaxOp()(total, carry);
    __syncthreads();
  }
  if (tid == 0) outs.recall[(size_t)t * A + a] = N ? __ddiv_rn((double)tp_cum[N - 1], dnpig) : 0.0;
  // np.searchsorted(rc, recThrs, side='left') with rc = tp / npig
  for (int r = tid; r < R; r += blockDim.x) {
    const double thr = p.rec_thrs[r];
    int lo = 0, hi = N;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ddiv_rn((double)tp_cum[mid], dnpig) < thr) lo = mid + 1;
      else hi = mid;
    }
    s_pi[r] = lo;
  }
  __syncthreads();
  // q[ri] = pr[pi]; ss[ri] = dtScoresSorted[pi] until the first pi == nd raises IndexError: from there on 0
  for (int r = tid; r < R; r += blockDim.x) {
    bool past = false;
    for (int q = 0; q <= r; ++q) past |= s_pi[q] == N;
    const int pi = s_pi[r];
    outs.precision[((size_t)t * R + r) * A + a] = past ? 0.0 : env[pi];
    outs.scores[((size_t)t * R + r) * A + a] = past ? 0.0 : w.slot_score[w.vals_out[pi]];
  }
}

}  // namespace

int validate_coco_params(const HpdCocoEvalParams* p) {
  if (!p) { set_error("hpd_coco_eval: params pointer is NULL"); return HPD_EINVAL; }
  if (p->num_images < 1) { set_error("hpd_coco_eval: num_images must be >= 1 (got %d)", p->num_images); return HPD_EINVAL; }
  if (p->num_kpts < 1 || p->num_kpts > HPD_MAX_KPTS) {
    set_error("hpd_coco_eval: num_kpts must be in [1,%d] (got %d)", HPD_MAX_KPTS, p->num_kpts);
    return HPD_EINVAL;
  }
  if (p->max_dets < 1 || p->max_dets > HPD_MAX_PEOPLE) {
    set_error("hpd_coco_eval: max_dets must be in [1,%d] (got %d)", HPD_MAX_PEOPLE, p->max_dets);
    return HPD_EINVAL;
  }
  if (p->max_gts < 1 || p->max_gts > HPD_COCO_MAX_PER_IMAGE) {
    set_error("hpd_coco_eval: max_gts must be in [1,%d] (got %d)", HPD_COCO_MAX_PER_IMAGE, p->max_gts);
    return HPD_EINVAL;
  }
  if (p->num_iou_thrs < 1 || p->num_iou_thrs > HPD_COCO_MAX_IOU_THRS) {
    set_error("hpd_coco_eval: num_iou_thrs must be in [1,%d] (got %d)", HPD_COCO_MAX_IOU_THRS, p->num_iou_thrs);
    return HPD_EINVAL;
  }
  if (p->num_rec_thrs < 1 || p->num_rec_thrs > HPD_COCO_MAX_REC_THRS) {
    set_error("hpd_coco_eval: num_rec_thrs must be in [1,%d] (got %d)", HPD_COCO_MAX_REC_THRS, p->num_rec_thrs);
    return HPD_EINVAL;
  }
  if (p->num_areas < 1 || p->num_areas > HPD_COCO_MAX_AREAS) {
    set_error("hpd_coco_eval: num_areas must be in [1,%d] (got %d)", HPD_COCO_MAX_AREAS, p->num_areas);
    return HPD_EINVAL;
  }
  if ((long long)p->num_images * p->max_dets > 0x7fffffffLL) {
    set_error("hpd_coco_eval: num_images * max_dets must be < 2^31");
    return HPD_EINVAL;
  }
  return HPD_OK;
}

size_t coco_eval_workspace_bytes(const HpdCocoEvalParams* p, int* rc) {
  CocoWs w;
  *rc = coco_workspace(p, nullptr, &w);
  return *rc ? 0 : w.total;
}

int launch_coco_eval(const HpdCocoEvalParams* p, const HpdCocoDets* dets, const HpdCocoGts* gts,
                     const HpdCocoEvalOutputs* outs, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!dets || !gts || !outs) { set_error("hpd_coco_eval: dets / gts / outs pointer is NULL"); return HPD_EINVAL; }
  if (!dets->base || !dets->row_offset) { set_error("hpd_coco_eval: dets.base / dets.row_offset is NULL"); return HPD_EINVAL; }
  if (dets->person_stride < 3 * p->num_kpts + 1) {
    set_error("hpd_coco_eval: dets.person_stride must be >= 3K+1 = %d (got %d)", 3 * p->num_kpts + 1, dets->person_stride);
    return HPD_EINVAL;
  }
  if (dets->max_per_row < 0 || dets->max_per_row > HPD_COCO_MAX_PER_IMAGE) {
    set_error("hpd_coco_eval: dets.max_per_row must be in [0,%d] (got %d)", HPD_COCO_MAX_PER_IMAGE, dets->max_per_row);
    return HPD_EINVAL;
  }
  if (dets->off_coco < 0 || dets->off_coco % 8 || dets->off_count < 0 || dets->off_count % 4) {
    set_error("hpd_coco_eval: dets.off_coco must be a multiple of 8 and dets.off_count of 4");
    return HPD_EINVAL;
  }
  if (!gts->kpts || !gts->area || !gts->bbox || !gts->iscrowd || !gts->ignore || !gts->n_gt) {
    set_error("hpd_coco_eval: a ground-truth array is NULL");
    return HPD_EINVAL;
  }
  if (!outs->precision || !outs->recall || !outs->scores) {
    set_error("hpd_coco_eval: precision / recall / scores must be given");
    return HPD_EINVAL;
  }
  CocoWs w;
  int rc = coco_workspace(p, (uint8_t*)ws, &w);
  if (rc) return rc;
  if (!ws || ws_bytes < w.total) {
    set_error("hpd_coco_eval: workspace too small (%zu < %zu bytes)", ws_bytes, w.total);
    return HPD_EWORKSPACE;
  }
  if (outs->oks) w.oks = outs->oks;
  if (outs->codes) w.codes = outs->codes;
  const int N = p->num_images * p->max_dets;

  coco_image_kernel<<<p->num_images, kImgThreads, 0, st>>>(*p, *dets, *gts, w);
  count_launch();
  if ((rc = check_launch("coco_image_kernel"))) return rc;
  size_t sort_bytes = w.sort_bytes;
  const cudaError_t e = cub::DeviceRadixSort::SortPairsDescending(w.sort_tmp, sort_bytes, w.keys_in, w.keys_out,
                                                                  w.vals_in, w.vals_out, N, 0, 64, st);
  count_launch();   // one sort, whatever number of passes CUB runs for it
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hpd_coco_eval: radix sort: %s", cudaGetErrorString(e));
    return HPD_ECUDA;
  }
  coco_accumulate_kernel<<<p->num_areas * p->num_iou_thrs, kAccThreads, 0, st>>>(*p, w, *outs);
  count_launch();
  return check_launch("coco_accumulate_kernel");
}

}  // namespace hpd
