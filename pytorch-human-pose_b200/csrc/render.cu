// Drawing decoded poses into frames (include/hpdecode.h: hpd_render_poses).  The NumPy statement of the rule is
// oracle/render_oracle.py.
//
//   render_kernel  one CTA per 64x32-pixel tile of a frame (grid z: the frame within the launch).  It stages the
//                  frame's joints in shared memory (invisible ones as NaN) and each person's box over its visible
//                  joints.  One warp tests the persons' boxes, widened by the larger primitive margin, against the
//                  tile; the primitives of the persons that meet it are culled with their own boxes, in paint order
//                  (per person: limbs in list order, then joints), and the survivors compacted in that order with
//                  their boxes clipped to the tile.  A tile without survivors is a plain copy.  Otherwise the tile is
//                  staged in shared memory, each pixel walks the survivors backwards, skipping those whose box misses
//                  it, and takes the colour of the first that covers it (the last in paint order), and the tile is
//                  written back.  Rows move as 16- or 8-byte words when both frames' tile rows are aligned to them, as
//                  bytes otherwise.
//
// The cull only decides which primitives a pixel tests, never the result: every pixel's test is the header's exact
// float64 rule (no division, no sqrt, no FMA), and the boxes are one pixel wider than the shapes, far more than the
// rounding of those few operations can move a boundary (|coordinates| <= 2^20).
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace hpd {
namespace {

constexpr int kTileW = 64, kTileH = 32, kThreads = 256, kFramesPerLaunch = 32;
constexpr int kTileRowBytes = 3 * kTileW;
constexpr int kMaxJoints = HPD_MAX_PEOPLE * HPD_MAX_KPTS;                          // 1024: 10-bit joint slots
constexpr int kMaxPrims = HPD_MAX_PEOPLE * (HPD_RENDER_MAX_LIMBS + HPD_MAX_KPTS);   // 3072
constexpr double kMaxCoord = 1048576.0;                                            // 2^20
// palette slots: limb_rgb[0..63], track_rgb[64..95], joint_rgb, untracked_rgb
constexpr int kPalTrack = HPD_RENDER_MAX_LIMBS, kPalJoint = kPalTrack + HPD_RENDER_MAX_COLORS;
constexpr int kPalUntracked = kPalJoint + 1, kPalSize = kPalUntracked + 1;
// a surviving primitive: joint slot a (bits 0-9), joint slot b (10-19), disc flag (20), palette slot (21-27)
constexpr uint32_t kDisc = 1u << 20;

struct RenderArgs {
  HpdRenderParams p;
  HpdRenderFrame f[kFramesPerLaunch];
  const uint8_t* records;   // the launch's first frame
  const int32_t* ids;       // [n][M] from the launch's first frame, or NULL
  const double* coords;     // [n][M][K][2] from the launch's first frame, or NULL
  HpdRecordLayout layout;
};

__device__ __forceinline__ double sq_sum(double dx, double dy) { return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)); }

__device__ __forceinline__ bool limb_covers(double X, double Y, double ax, double ay, double bx, double by, double hh) {
  const double ex = __dsub_rn(bx, ax), ey = __dsub_rn(by, ay);
  const double L2 = sq_sum(ex, ey);
  const double px = __dsub_rn(X, ax), py = __dsub_rn(Y, ay);
  const double t = __dadd_rn(__dmul_rn(px, ex), __dmul_rn(py, ey));
  if (t <= 0.0) return sq_sum(px, py) <= hh;
  if (t >= L2) return sq_sum(__dsub_rn(X, bx), __dsub_rn(Y, by)) <= hh;
  const double cr = __dsub_rn(__dmul_rn(px, ey), __dmul_rn(py, ex));
  return __dmul_rn(cr, cr) <= __dmul_rn(hh, L2);
}

// th rows of rb bytes from src to dst, as T-sized elements (rb, both bases and both strides multiples of sizeof(T))
template <typename T>
__device__ __forceinline__ void copy_rows(const uint8_t* src, int64_t src_stride, uint8_t* dst, int64_t dst_stride,
                                          int th, int rb) {
  const int n = rb / (int)sizeof(T);
  for (int i = threadIdx.x; i < th * n; i += kThreads) {
    const int r = i / n, c = i - r * n;
    reinterpret_cast<T*>(dst + r * dst_stride)[c] = reinterpret_cast<const T*>(src + r * src_stride)[c];
  }
}

// align: the largest of 16, 8 and 1 that divides both bases, both strides and rb
__device__ __forceinline__ void move_rows(int align, const uint8_t* src, int64_t src_stride, uint8_t* dst,
                                          int64_t dst_stride, int th, int rb) {
  if (align == 16)
    copy_rows<uint4>(src, src_stride, dst, dst_stride, th, rb);
  else if (align == 8)
    copy_rows<uint64_t>(src, src_stride, dst, dst_stride, th, rb);
  else
    copy_rows<uint8_t>(src, src_stride, dst, dst_stride, th, rb);
}

__device__ __forceinline__ uint32_t rgb_of(const uint8_t* c) { return c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16; }

__global__ void __launch_bounds__(kThreads) render_kernel(const __grid_constant__ RenderArgs a) {
  const HpdRenderFrame& fr = a.f[blockIdx.z];
  const int x0 = blockIdx.x * kTileW, y0 = blockIdx.y * kTileH;
  if (x0 >= fr.w || y0 >= fr.h) return;
  __shared__ double s_x[kMaxJoints], s_y[kMaxJoints];   // s_x NaN: the joint is not visible
  __shared__ uint32_t s_prim[kMaxPrims];
  __shared__ uint32_t s_box[kMaxPrims];                 // the survivor's box in tile pixels: x0, x1, y0, y1 bytes
  __shared__ __align__(16) uint8_t s_tile[kTileH * kTileRowBytes];
  __shared__ uint32_t s_pal[kPalSize];
  __shared__ int s_pcol[HPD_MAX_PEOPLE];                // palette slot of the person's limbs, -1: limb_rgb[l]
  __shared__ int s_warp[kThreads / 32];
  __shared__ double s_pbox[HPD_MAX_PEOPLE][4];         // a person's visible joints: min x, max x, min y, max y
  __shared__ unsigned s_pmask;                         // the persons whose widened box meets the tile
  const HpdRenderParams& P = a.p;
  const int K = P.num_kpts, M = P.max_people, NL = P.num_limbs, tid = threadIdx.x;
  const HpdRecordLayout& L = a.layout;
  const uint8_t* rec = a.records + (size_t)blockIdx.z * L.row_bytes;
  const int flags = *reinterpret_cast<const int32_t*>(rec + L.off_flags);
  const int n = (flags & 1) ? 0 : min(max(*reinterpret_cast<const int32_t*>(rec + L.off_n_person), 0), M);

  for (int i = tid; i < n * K; i += kThreads) {
    const int p = i / K, k = i - p * K;
    const double* c = a.coords ? a.coords + (((size_t)blockIdx.z * M + p) * K + k) * 2
                               : reinterpret_cast<const double*>(rec + L.off_coco) + (size_t)p * L.coco_stride + 3 * k;
    const double x = c[0], y = c[1];
    const float s = reinterpret_cast<const float*>(rec + L.off_poses)[((size_t)p * K + k) * (3 + P.emb) + 2];
    // |v| <= 2^20 is false for NaN and +-inf: the bound is the finiteness test too
    const bool vis = (double)s > P.kpt_thr && fabs(x) <= kMaxCoord && fabs(y) <= kMaxCoord;
    s_x[i] = vis ? x : __longlong_as_double(0x7ff8000000000000LL);
    s_y[i] = y;
  }
  if (tid < n) {
    const int id = a.ids ? a.ids[(size_t)blockIdx.z * M + tid] : 0;
    s_pcol[tid] = !a.ids ? -1 : id >= 0 ? kPalTrack + id % P.num_track_colors : kPalUntracked;
  }
  if (tid < kPalSize) {
    s_pal[tid] = tid < kPalTrack ? rgb_of(P.limb_rgb[tid])
               : tid < kPalJoint ? rgb_of(P.track_rgb[tid - kPalTrack])
               : tid == kPalJoint ? rgb_of(P.joint_rgb) : rgb_of(P.untracked_rgb);
  }
  __syncthreads();
  if (tid < n) {
    double lx = INFINITY, hx = -INFINITY, ly = INFINITY, hy = -INFINITY;
    for (int k = 0; k < K; ++k) {
      const double x = s_x[tid * K + k], y = s_y[tid * K + k];
      if (x == x) { lx = fmin(lx, x); hx = fmax(hx, x); ly = fmin(ly, y); hy = fmax(hy, y); }
    }
    s_pbox[tid][0] = lx; s_pbox[tid][1] = hx; s_pbox[tid][2] = ly; s_pbox[tid][3] = hy;
  }
  __syncthreads();

  const double h = P.thickness / 2, hh = __dmul_rn(h, h), R = P.joint_radius, rr = __dmul_rn(R, R);
  const double hm = h + 1.0, rm = R + 1.0, pm = fmax(hm, rm);   // box margins
  const int tw = min(kTileW, fr.w - x0), per = NL + K;
  const int th = min(kTileH, fr.h - y0);
  const double tx0 = x0, tx1 = x0 + tw - 1, ty0 = y0, ty1 = y0 + th - 1;
  if (tid < 32) {   // n <= 32: one warp tests the persons' boxes, widened by the larger primitive margin
    const bool hit = tid < n && s_pbox[tid][0] - pm <= tx1 && s_pbox[tid][1] + pm >= tx0 &&
                     s_pbox[tid][2] - pm <= ty1 && s_pbox[tid][3] + pm >= ty0;
    const unsigned m = __ballot_sync(kFull, hit);
    if (tid == 0) s_pmask = m;
  }
  __syncthreads();
  const unsigned pmask = s_pmask;
  const int total = __popc(pmask) * per;   // the primitives of those persons, in paint order
  int ns = 0;
  for (int c0 = 0; c0 < total; c0 += kThreads) {   // uniform across the CTA
    const int q = c0 + tid;
    bool keep = false;
    uint32_t code = 0;
    double lx = 0, hx = 0, ly = 0, hy = 0;           // the primitive's box
    if (q < total) {
      const int pi = q / per, j = q - pi * per, p = __fns(pmask, 0, pi + 1);
      if (j < NL) {
        if (h > 0.0) {
          const int ia = p * K + P.limbs[j][0], ib = p * K + P.limbs[j][1];
          const double ax = s_x[ia], ay = s_y[ia], bx = s_x[ib], by = s_y[ib];
          lx = fmin(ax, bx) - hm; hx = fmax(ax, bx) + hm; ly = fmin(ay, by) - hm; hy = fmax(ay, by) + hm;
          keep = ax == ax && bx == bx && lx <= tx1 && hx >= tx0 && ly <= ty1 && hy >= ty0;
          code = (uint32_t)ia | (uint32_t)ib << 10 | (uint32_t)(s_pcol[p] < 0 ? j : s_pcol[p]) << 21;
        }
      } else if (R > 0.0) {
        const int ia = p * K + (j - NL);
        const double x = s_x[ia], y = s_y[ia];
        lx = x - rm; hx = x + rm; ly = y - rm; hy = y + rm;
        keep = x == x && lx <= tx1 && hx >= tx0 && ly <= ty1 && hy >= ty0;
        code = (uint32_t)ia | kDisc | (uint32_t)kPalJoint << 21;
      }
    }
    const unsigned bal = __ballot_sync(kFull, keep);
    if ((tid & 31) == 0) s_warp[tid >> 5] = __popc(bal);
    __syncthreads();
    int before = 0, chunk = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
      const int cnt = s_warp[w];
      before += w < (tid >> 5) ? cnt : 0;
      chunk += cnt;
    }
    if (keep) {
      const int slot = ns + before + __popc(bal & ((1u << (tid & 31)) - 1));
      s_prim[slot] = code;
      const int bx0 = max((int)floor(lx) - x0, 0), bx1 = min((int)ceil(hx) - x0, tw - 1);
      const int by0 = max((int)floor(ly) - y0, 0), by1 = min((int)ceil(hy) - y0, th - 1);
      s_box[slot] = (uint32_t)bx0 | (uint32_t)bx1 << 8 | (uint32_t)by0 << 16 | (uint32_t)by1 << 24;
    }
    ns += chunk;
    __syncthreads();
  }

  const uint8_t* in = fr.in + (size_t)y0 * fr.in_stride_row + 3 * x0;
  uint8_t* out = fr.out + (size_t)y0 * fr.out_stride_row + 3 * x0;
  const int rb = 3 * tw;
  const uintptr_t bits = (uintptr_t)in | (uintptr_t)out | (uintptr_t)fr.in_stride_row | (uintptr_t)fr.out_stride_row |
                         (uintptr_t)rb;
  const int align = bits % 16 == 0 ? 16 : bits % 8 == 0 ? 8 : 1;
  if (ns == 0) {
    move_rows(align, in, fr.in_stride_row, out, fr.out_stride_row, th, rb);
    return;
  }
  move_rows(align, in, fr.in_stride_row, s_tile, kTileRowBytes, th, rb);
  __syncthreads();
  for (int i = tid; i < th * kTileW; i += kThreads) {
    const int r = i / kTileW, c = i % kTileW;
    if (c >= tw) continue;
    const double X = x0 + c, Y = y0 + r;
    int col = -1;
    for (int s = ns - 1; s >= 0; --s) {
      const uint32_t b = s_box[s];
      if (c < (int)(b & 255) || c > (int)((b >> 8) & 255) || r < (int)((b >> 16) & 255) || r > (int)(b >> 24)) continue;
      const uint32_t e = s_prim[s];
      const int ia = e & 1023;
      const bool cov = (e & kDisc) ? sq_sum(__dsub_rn(X, s_x[ia]), __dsub_rn(Y, s_y[ia])) <= rr
                                   : limb_covers(X, Y, s_x[ia], s_y[ia], s_x[(e >> 10) & 1023], s_y[(e >> 10) & 1023], hh);
      if (cov) {
        col = (int)(e >> 21);
        break;
      }
    }
    if (col >= 0) {
      const uint32_t rgb = s_pal[col];
      uint8_t* q = s_tile + r * kTileRowBytes + 3 * c;
      q[0] = (uint8_t)rgb;
      q[1] = (uint8_t)(rgb >> 8);
      q[2] = (uint8_t)(rgb >> 16);
    }
  }
  __syncthreads();
  move_rows(align, s_tile, kTileRowBytes, out, fr.out_stride_row, th, rb);
}

// byte range [lo, hi) a frame's rows span
struct Span {
  uintptr_t lo, hi;
};

Span span_of(const void* ptr, int64_t stride, int h, int w) {
  const uintptr_t lo = (uintptr_t)ptr;
  return {lo, lo + (uintptr_t)(h - 1) * (uintptr_t)stride + 3u * (uintptr_t)w};
}

bool overlap(const Span& a, const Span& b) { return a.lo < b.hi && b.lo < a.hi; }

constexpr int64_t kMaxStride = 1LL << 47;

int validate_render(const HpdRenderParams* p, const HpdRenderFrame* fr, int n, const uint8_t* records,
                    const int32_t* ids, const double* coords) {
  const char* who = "hpd_render_poses";
  if (!p) { set_error("%s: params pointer is NULL", who); return HPD_EINVAL; }
  if (p->num_kpts < 1 || p->num_kpts > HPD_MAX_KPTS) {
    set_error("%s: num_kpts must be in [1,%d] (got %d)", who, HPD_MAX_KPTS, p->num_kpts);
    return HPD_EINVAL;
  }
  if (p->max_people < 1 || p->max_people > HPD_MAX_PEOPLE) {
    set_error("%s: max_people must be in [1,%d] (got %d)", who, HPD_MAX_PEOPLE, p->max_people);
    return HPD_EINVAL;
  }
  if (p->emb < 1 || p->emb > HPD_MAX_EMB) { set_error("%s: emb must be 1 or 2 (got %d)", who, p->emb); return HPD_EINVAL; }
  if (p->num_limbs < 0 || p->num_limbs > HPD_RENDER_MAX_LIMBS) {
    set_error("%s: num_limbs must be in [0,%d] (got %d)", who, HPD_RENDER_MAX_LIMBS, p->num_limbs);
    return HPD_EINVAL;
  }
  for (int l = 0; l < p->num_limbs; ++l) {
    const int a = p->limbs[l][0], b = p->limbs[l][1];
    if (a < 0 || a >= p->num_kpts || b < 0 || b >= p->num_kpts) {
      set_error("%s: limbs[%d] = (%d, %d): joints must be in [0,num_kpts=%d)", who, l, a, b, p->num_kpts);
      return HPD_EINVAL;
    }
    if (a == b) { set_error("%s: limbs[%d] joins joint %d to itself", who, l, a); return HPD_EINVAL; }
  }
  const struct { const char* name; double v; } sizes[] = {{"thickness", p->thickness}, {"joint_radius", p->joint_radius}};
  for (const auto& s : sizes) {
    if (!(isfinite(s.v) && s.v >= 0.0 && s.v <= 1024.0)) {
      set_error("%s: %s must be finite and in [0, 1024] (got %g)", who, s.name, s.v);
      return HPD_EINVAL;
    }
  }
  if (!isfinite(p->kpt_thr)) { set_error("%s: kpt_thr must be finite", who); return HPD_EINVAL; }
  if (p->num_track_colors < 1 || p->num_track_colors > HPD_RENDER_MAX_COLORS) {
    set_error("%s: num_track_colors must be in [1,%d] (got %d)", who, HPD_RENDER_MAX_COLORS, p->num_track_colors);
    return HPD_EINVAL;
  }
  if (n < 1) { set_error("%s: n_frames must be >= 1 (got %d)", who, n); return HPD_EINVAL; }
  if (!fr) { set_error("%s: frames_host is NULL", who); return HPD_EINVAL; }
  if (!records) { set_error("%s: records is NULL", who); return HPD_EINVAL; }
  if ((uintptr_t)records % 8) { set_error("%s: records must be 8-byte aligned", who); return HPD_EINVAL; }
  if ((uintptr_t)ids % 4) { set_error("%s: track_ids must be 4-byte aligned", who); return HPD_EINVAL; }
  if ((uintptr_t)coords % 8) { set_error("%s: coords must be 8-byte aligned", who); return HPD_EINVAL; }
  for (int f = 0; f < n; ++f) {
    const HpdRenderFrame& F = fr[f];
    if (!F.in || !F.out) { set_error("%s: frame %d: in / out is NULL", who, f); return HPD_EINVAL; }
    if (F.h < 1 || F.h > 32767 || F.w < 1 || F.w > 32767) {
      set_error("%s: frame %d: size %dx%d outside 1..32767", who, f, F.h, F.w);
      return HPD_EINVAL;
    }
    if (F.in_stride_row < 3LL * F.w || F.out_stride_row < 3LL * F.w || F.in_stride_row > kMaxStride ||
        F.out_stride_row > kMaxStride) {
      set_error("%s: frame %d: row strides must be in [3*w=%lld, 2^47] (got in %lld, out %lld)", who, f, 3LL * F.w,
                (long long)F.in_stride_row, (long long)F.out_stride_row);
      return HPD_EINVAL;
    }
  }
  for (int f = 0; f < n; ++f) {
    const Span o = span_of(fr[f].out, fr[f].out_stride_row, fr[f].h, fr[f].w);
    for (int g = 0; g < n; ++g) {
      if (overlap(o, span_of(fr[g].in, fr[g].in_stride_row, fr[g].h, fr[g].w))) {
        set_error("%s: frame %d's output overlaps frame %d's input (out of place only)", who, f, g);
        return HPD_EINVAL;
      }
      if (g < f && overlap(o, span_of(fr[g].out, fr[g].out_stride_row, fr[g].h, fr[g].w))) {
        set_error("%s: frame %d's output overlaps frame %d's output", who, f, g);
        return HPD_EINVAL;
      }
    }
  }
  return HPD_OK;
}

}  // namespace

int launch_render_poses(const HpdRenderParams* p, const HpdRenderFrame* frames, int n_frames, const uint8_t* records,
                        const int32_t* track_ids, const double* coords, cudaStream_t st) {
  int rc = validate_render(p, frames, n_frames, records, track_ids, coords);
  if (rc) return rc;
  const int K = p->num_kpts, M = p->max_people;
  const HpdRecordLayout layout = record_layout(K, M, p->emb);
  for (int f0 = 0; f0 < n_frames; f0 += kFramesPerLaunch) {
    const int n = n_frames - f0 < kFramesPerLaunch ? n_frames - f0 : kFramesPerLaunch;
    RenderArgs a;
    memset(&a, 0, sizeof(a));
    a.p = *p;
    int max_h = 0, max_w = 0;
    for (int i = 0; i < n; ++i) {
      a.f[i] = frames[f0 + i];
      max_h = max_h > a.f[i].h ? max_h : a.f[i].h;
      max_w = max_w > a.f[i].w ? max_w : a.f[i].w;
    }
    a.records = records + (size_t)f0 * layout.row_bytes;
    a.ids = track_ids ? track_ids + (size_t)f0 * M : nullptr;
    a.coords = coords ? coords + (size_t)f0 * M * K * 2 : nullptr;
    a.layout = layout;
    const dim3 grid((max_w + kTileW - 1) / kTileW, (max_h + kTileH - 1) / kTileH, n);
    render_kernel<<<grid, kThreads, 0, st>>>(a);
    count_launch();
    if ((rc = check_launch("render_kernel"))) return rc;
  }
  return HPD_OK;
}

}  // namespace hpd
