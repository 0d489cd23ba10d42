// Shared device/host helpers for libhpdecode (sm_100a).  Compiled with -fmad=false: the only
// fused multiply-adds in the library are the explicit fmaf() calls that reproduce torch's CPU
// bilinear kernel (SURVEY.md App. A.2).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/hpdecode.h"

namespace hpd {

constexpr unsigned kFull = 0xffffffffu;

// ---- launch bookkeeping / error reporting (api.cu) --------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_launch(const char* what);
int ensure_dynamic_smem(const void* kernel, size_t bytes, const char* name);

// ---- bilinear taps, torch CPU semantics (results.py:51,59,65; aten UpSampleKernel.cpp) -----
struct Tap {
  int i0, i1;
  float w0, w1;
};

__host__ __device__ __forceinline__ Tap axis_tap(float scale, int o, int in_size, int out_size) {
  Tap t;
  if (in_size == out_size) {
    t.i0 = t.i1 = o;
    t.w0 = 1.f;
    t.w1 = 0.f;
    return t;
  }
  float src = fmaf(scale, (float)o + 0.5f, -0.5f);
  if (src < 0.f) src = 0.f;
  int i0 = (int)src;
  if (i0 > in_size - 1) i0 = in_size - 1;
  float l1 = src - (float)i0;
  l1 = fminf(fmaxf(l1, 0.f), 1.f);
  t.i0 = i0;
  t.i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  t.w1 = l1;
  t.w0 = 1.f - l1;
  return t;
}

#ifdef __CUDACC__
// out = hy0*(wx0*v00 + wx1*v01) + hy1*(wx0*v10 + wx1*v11) with torch's FMA nesting
__device__ __forceinline__ float lerp2(float wx0, float wx1, float hy0, float hy1, float v00, float v01, float v10,
                                       float v11) {
  const float top = fmaf(wx0, v00, __fmul_rn(wx1, v01));
  const float bot = fmaf(wx0, v10, __fmul_rn(wx1, v11));
  return fmaf(hy0, top, __fmul_rn(hy1, bot));
}

// element i of an input plane of dtype code `dtype` (HPD_F32 / HPD_F16 / HPD_BF16); 16-bit values are widened
// exactly (a bfloat16 is the upper half of a float32)
__device__ __forceinline__ float in_elem(const float* base, size_t i, int dtype) {
  if (dtype == HPD_F32) return base[i];
  const unsigned short u = reinterpret_cast<const unsigned short*>(base)[i];
  return dtype == HPD_F16 ? __half2float(__ushort_as_half(u)) : __uint_as_float((unsigned)u << 16);
}
#endif  // __CUDACC__

// ---- tag values at full resolution (results.py:229-230) -----------------------------------------
// Where the tag stages read a tag: the full-resolution map agg_tags [B,K,H,W,E] when the caller keeps one,
// otherwise the tag-scale network outputs, interpolated at the pixel (tag_at).  The map is never read
// densely (top-k winners, detected joints, refine candidates), so interpolating where it is read saves
// writing 4*K*H*W*E bytes per image.
struct TagSource {
  const float* map;                  // [B,K,H,W,E] or NULL: interpolate from tag / tag_f
  const float *tag, *tag_f;          // tag-scale maps (tag_f: flipped run, E == 2); elements of type `dtype`
  long long tag_sb, tag_sc, tagf_sb, tagf_sc;
  int K, H, W, E;
  int th, tw;                        // tag-scale map size
  float s_y, s_x;                    // th / H, tw / W
  int dtype, tags_preflipped;        // dtype: HPD_F32 / HPD_F16 / HPD_BF16
  int flip[HPD_MAX_KPTS];
};

#ifdef __CUDACC__
// The tag vector of output pixel (y, x) of plane (b, k), as aggregate_tags_kernel writes it into the map: bilinear
// taps on both axes (axis_tap, lerp2), the flipped run read at the mirrored column and the flipped joint unless
// tags_preflipped (model.py:93).  t[e] for e >= E is left alone.
__device__ __forceinline__ void tag_at(const TagSource& s, int b, int k, int y, int x, float (&t)[HPD_MAX_EMB]) {
  const Tap tx = axis_tap(s.s_x, x, s.tw, s.W), ty = axis_tap(s.s_y, y, s.th, s.H);
#pragma unroll
  for (int e = 0; e < HPD_MAX_EMB; ++e) {
    if (e >= s.E) break;
    const bool unflip = (e == 1) && !s.tags_preflipped;
    const float* p = (e == 0) ? s.tag : s.tag_f;
    const size_t po = (e == 0) ? (size_t)b * s.tag_sb + (size_t)k * s.tag_sc
                               : (size_t)b * s.tagf_sb + (size_t)(unflip ? s.flip[k] : k) * s.tagf_sc;
    const int c0 = unflip ? s.tw - 1 - tx.i0 : tx.i0, c1 = unflip ? s.tw - 1 - tx.i1 : tx.i1;
    const size_t r0 = po + (size_t)ty.i0 * s.tw, r1 = po + (size_t)ty.i1 * s.tw;
    t[e] = lerp2(tx.w0, tx.w1, ty.w0, ty.w1, in_elem(p, r0 + c0, s.dtype), in_elem(p, r0 + c1, s.dtype),
                 in_elem(p, r1 + c0, s.dtype), in_elem(p, r1 + c1, s.dtype));
  }
}

// tag vector of pixel idx = y*W + x of plane row = b*K + k: from the map if there is one, else tag_at
__device__ __forceinline__ void tag_value(const TagSource& s, int row, int idx, float (&t)[HPD_MAX_EMB]) {
  if (s.map != nullptr) {
    const float* q = s.map + ((size_t)row * s.H * s.W + idx) * s.E;
    t[0] = q[0];
    if (s.E > 1) t[1] = q[1];
  } else {
    tag_at(s, row / s.K, row % s.K, idx / s.W, idx % s.W, t);
  }
}

// order-preserving float -> signed int map (for redux.sync max)
__device__ __forceinline__ int float_order_int(float f) {
  const int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float order_int_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

__device__ __forceinline__ float warp_max_float(float v) {
  return order_int_float(__reduce_max_sync(kFull, float_order_int(v)));
}

// numpy float32 pairwise-8 summation of n <= 128 strided values (np.mean / np.sum inner loop)
__device__ __forceinline__ float np_sum_pairwise8(const float* a, int n, int stride) {
  if (n < 8) {
    float r = -0.0f;
    for (int i = 0; i < n; ++i) r = __fadd_rn(r, a[i * stride]);
    return r;
  }
  float r0 = a[0], r1 = a[stride], r2 = a[2 * stride], r3 = a[3 * stride], r4 = a[4 * stride], r5 = a[5 * stride],
        r6 = a[6 * stride], r7 = a[7 * stride];
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
    r0 = __fadd_rn(r0, a[(i + 0) * stride]);
    r1 = __fadd_rn(r1, a[(i + 1) * stride]);
    r2 = __fadd_rn(r2, a[(i + 2) * stride]);
    r3 = __fadd_rn(r3, a[(i + 3) * stride]);
    r4 = __fadd_rn(r4, a[(i + 4) * stride]);
    r5 = __fadd_rn(r5, a[(i + 5) * stride]);
    r6 = __fadd_rn(r6, a[(i + 6) * stride]);
    r7 = __fadd_rn(r7, a[(i + 7) * stride]);
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r0, r1), __fadd_rn(r2, r3)),
                        __fadd_rn(__fadd_rn(r4, r5), __fadd_rn(r6, r7)));
  for (; i < n; ++i) res = __fadd_rn(res, a[i * stride]);
  return res;
}

// numpy float64 np.sum of n <= 128 terms fed one at a time in index order (its 128-element block): a plain sum below 8
// terms, the pairwise-8 unrolled loop from 8 on.  r0..r7 are NumPy's eight accumulators, rotated after every term so
// that r0 always receives the next one; after a multiple of 8 terms they are back in place.  Exactly n add() calls.
struct NpSumF64 {
  double r0 = 0, r1 = 0, r2 = 0, r3 = 0, r4 = 0, r5 = 0, r6 = 0, r7 = 0;
  double res = -0.0;
  int c = 0, n, n_main;
  __device__ __forceinline__ explicit NpSumF64(int n_) : n(n_), n_main(n_ - n_ % 8) {}
  __device__ __forceinline__ double block8() const {
    return __dadd_rn(__dadd_rn(__dadd_rn(r0, r1), __dadd_rn(r2, r3)), __dadd_rn(__dadd_rn(r4, r5), __dadd_rn(r6, r7)));
  }
  __device__ __forceinline__ void add(double term) {
    if (n < 8) {
      res = __dadd_rn(res, term);
    } else if (c < n_main) {
      const double v = c < 8 ? term : __dadd_rn(r0, term);
      r0 = r1; r1 = r2; r2 = r3; r3 = r4; r4 = r5; r5 = r6; r6 = r7; r7 = v;
    } else {
      if (c == n_main) res = block8();
      res = __dadd_rn(res, term);
    }
    ++c;
  }
  // the reduction starts from add's identity
  __device__ __forceinline__ double sum() const { return __dadd_rn(0.0, n >= 8 && n_main == n ? block8() : res); }
};

// np.mean(list of n float32 vectors of E components, axis=0) (grouping.py:114,213):
// E == 1 reduces a contiguous axis (pairwise-8), E == 2 accumulates row by row (sequential).
__device__ __forceinline__ void np_mean_vectors(const float* v, int n, int E, int row_stride, float* out) {
  if (E == 1) {
    out[0] = __fdiv_rn(__fadd_rn(0.0f, np_sum_pairwise8(v, n, row_stride)), (float)n);
  } else {
    for (int e = 0; e < E; ++e) {
      float s = 0.0f;
      for (int i = 0; i < n; ++i) s = __fadd_rn(s, v[i * row_stride + e]);
      out[e] = __fdiv_rn(s, (float)n);
    }
  }
}
#endif  // __CUDACC__

// ---- per-image result record (include/hpdecode.h: HpdRecordLayout) ------------------------------
__host__ __device__ inline HpdRecordLayout record_layout(int K, int M, int E) {
  HpdRecordLayout L;
  L.coco_stride = 3 * K + 1;
  L.reserved_ = 0;
  long long off = 0;
  L.off_coco = off;          off += 8LL * M * L.coco_stride;
  L.off_poses = off;         off += 4LL * M * K * (3 + E);
  L.off_person_scores = off; off += 4LL * M;
  L.off_n_person = off;      off += 4;
  L.off_flags = off;         off += 4;
  L.row_bytes = (off + 7) / 8 * 8;
  return L;
}

// ---- per-stage launchers (defined in the stage .cu files) -------------------------------------
int launch_aggregate_nms(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, cudaStream_t st);
HpdStageInputs two_stage_inputs(const HpdScaleInputs& s);   // {hm = {hm_lo, hm_hi}, num_stages = 2}
HpdScaleInputs tag_scale_inputs(const HpdStageInputs& s);   // the tag / tag_f maps alone (HpdBuffers.tag_inputs)
int launch_aggregate_tags(const HpdParams* p, const HpdScaleInputs* scales, float* out, cudaStream_t st);
// where the tag stages read tags: buf->agg_tags if set, else buf->tag_inputs (HPD_EINVAL if neither is given)
int make_tag_source(const HpdParams* p, const HpdBuffers* buf, TagSource* s, const char* who);
int launch_nms(const HpdParams* p, const HpdBuffers* buf, float* nms_out, cudaStream_t st);
int launch_topk(const HpdParams* p, const HpdBuffers* buf, cudaStream_t st);
int launch_group(const HpdParams* p, const HpdBuffers* buf, cudaStream_t st);
int launch_adjust_refine(const HpdParams* p, const HpdBuffers* buf, void* ws, size_t ws_bytes, cudaStream_t st);
size_t refine_workspace_bytes(const HpdParams* p);
int launch_resize(const HpdMap* in, int batch, int channels, float* out, int oh, int ow, cudaStream_t st);
int launch_prepare_input(const HpdImage* images, int batch, float* out, int oh, int ow, const float* mean,
                         const float* stdv, cudaStream_t st);
int launch_prepare_inputs(const HpdImage* images, int batch, const HpdPrepareTarget* targets, int n_targets,
                          const float* mean, const float* stdv, cudaStream_t st);
int multi_scale_size(int h, int w, int input_size, double current_scale, double min_scale, int32_t* size_wh,
                     int32_t* center_xy, double* scale_wh);
int affine_transform_matrix(const double* center, const double* scale, const int32_t* out_wh, int inverse, double* m);
int validate_coco_params(const HpdCocoEvalParams* p);
size_t coco_eval_workspace_bytes(const HpdCocoEvalParams* p, int* rc);
int launch_coco_eval(const HpdCocoEvalParams* p, const HpdCocoDets* dets, const HpdCocoGts* gts,
                     const HpdCocoEvalOutputs* outs, void* ws, size_t ws_bytes, cudaStream_t st);
int validate_track_params(const HpdTrackParams* p, const char* who);
size_t track_state_bytes(const HpdTrackParams* p);
int launch_track_reset(const HpdTrackParams* p, void* state, size_t state_bytes, int clear_ids, cudaStream_t st);
int launch_track(const HpdTrackParams* p, const uint8_t* records, int n_frames, void* state, size_t state_bytes,
                 int32_t* track_ids, cudaStream_t st);
size_t track_smooth_state_bytes(const HpdTrackParams* p);
int launch_track_smooth(const HpdTrackParams* p, const HpdSmoothParams* sp, const uint8_t* records, int n_frames,
                        void* state, size_t state_bytes, int32_t* track_ids, double* coords, cudaStream_t st);
int launch_render_poses(const HpdRenderParams* p, const HpdRenderFrame* frames, int n_frames, const uint8_t* records,
                        const int32_t* track_ids, const double* coords, cudaStream_t st);

}  // namespace hpd
