// C ABI of libhpdecode.so (include/hpdecode.h): argument validation, error strings, launch
// accounting and the whole-path entry point.  No allocation, no synchronisation.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

namespace hpd {

namespace {
thread_local char g_err[512] = "";
thread_local int g_launches = 0;
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(int n) { g_launches += n; }

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();   // consumes the error: a failed launch must not poison later calls
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return HPD_ECUDA;
  }
  return HPD_OK;
}

// Kernels that need more than 48 KB of dynamic shared memory opt in once per (kernel, device): the
// attribute is sticky, so it is not set again on every launch, and a refusal is reported.
int ensure_dynamic_smem(const void* kernel, size_t bytes, const char* name) {
  if (bytes <= 48 * 1024) return HPD_OK;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: no current CUDA device", name);
    return HPD_ECUDA;
  }
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> granted;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = granted[std::make_pair(kernel, dev)];
  if (have >= bytes) return HPD_OK;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: cannot opt in to %zu bytes of shared memory: %s", name, bytes, cudaGetErrorString(e));
    return HPD_ECUDA;
  }
  have = bytes;
  return HPD_OK;
}

static int validate(const HpdParams* p, const HpdBuffers* buf) {
  if (!p || !buf) { set_error("params / buffers pointer is NULL"); return HPD_EINVAL; }
  if (p->batch < 1) { set_error("batch must be >= 1 (got %d)", p->batch); return HPD_EINVAL; }
  if (p->num_kpts < 1 || p->num_kpts > HPD_MAX_KPTS) { set_error("num_kpts must be in [1,%d] (got %d)", HPD_MAX_KPTS, p->num_kpts); return HPD_EINVAL; }
  if (p->max_people < 1 || p->max_people > HPD_MAX_PEOPLE) { set_error("max_people must be in [1,%d] (got %d)", HPD_MAX_PEOPLE, p->max_people); return HPD_EINVAL; }
  if (p->emb < 1 || p->emb > HPD_MAX_EMB) { set_error("emb must be 1 or 2 (got %d)", p->emb); return HPD_EINVAL; }
  if (p->out_h < 1 || p->out_w < 1) { set_error("bad output size %dx%d", p->out_h, p->out_w); return HPD_EINVAL; }
  if ((long long)p->out_h * p->out_w < 64LL * p->max_people) {
    // torch's CPU topk switches to nth_element+sort (other tie order) below this size
    set_error("H*W must be >= 64*max_people (got %dx%d, M=%d)", p->out_h, p->out_w, p->max_people);
    return HPD_EINVAL;
  }
  if ((long long)p->out_h * p->out_w >= (1LL << 31)) { set_error("map too large"); return HPD_EINVAL; }
  if ((long long)p->batch * p->num_kpts > 65535) { set_error("batch*num_kpts must be <= 65535"); return HPD_EINVAL; }
  if (p->num_scales < 1 || p->num_scales > HPD_MAX_SCALES) { set_error("num_scales must be in [1,%d]", HPD_MAX_SCALES); return HPD_EINVAL; }
  if (p->tag_scale < 0 || p->tag_scale >= p->num_scales) { set_error("tag_scale out of range"); return HPD_EINVAL; }
  for (int k = 0; k < p->num_kpts; ++k) {
    if (p->flip_index[k] < 0 || p->flip_index[k] >= p->num_kpts || p->joints_order[k] < 0 || p->joints_order[k] >= p->num_kpts) {
      set_error("flip_index / joints_order entry %d out of range", k);
      return HPD_EINVAL;
    }
  }
  return HPD_OK;
}

// The two-stage HpdScaleInputs of the older entry points as HpdStageInputs (NULL stays NULL); n <= HPD_MAX_SCALES.
static const HpdStageInputs* as_stages(const HpdScaleInputs* scales, int n, HpdStageInputs* out) {
  if (!scales) return nullptr;
  for (int s = 0; s < n; ++s) out[s] = two_stage_inputs(scales[s]);
  return out;
}

static int decode_validated(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, void* workspace,
                            size_t workspace_bytes, cudaStream_t st);

}  // namespace hpd

using namespace hpd;

extern "C" {

int hpd_abi_version(void) { return HPD_ABI_VERSION; }

const char* hpd_last_error_string(void) { return g_err; }

int hpd_last_launch_count(void) { return g_launches; }

int hpd_workspace_bytes(const HpdParams* p, size_t* out_bytes) {
  if (!p || !out_bytes) { set_error("NULL argument"); return HPD_EINVAL; }
  *out_bytes = refine_workspace_bytes(p);
  return HPD_OK;
}

int hpd_aggregate_nms_stages(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return launch_aggregate_nms(p, scales, buf, (cudaStream_t)stream);
}

int hpd_aggregate_nms(const HpdParams* p, const HpdScaleInputs* scales, const HpdBuffers* buf, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  HpdStageInputs st[HPD_MAX_SCALES];
  return launch_aggregate_nms(p, as_stages(scales, p->num_scales, st), buf, (cudaStream_t)stream);
}

int hpd_aggregate_tags(const HpdParams* p, const HpdScaleInputs* scales, float* out, void* stream) {
  g_launches = 0;
  const HpdBuffers none = {};
  int rc = validate(p, &none);
  if (rc) return rc;
  return launch_aggregate_tags(p, scales, out, (cudaStream_t)stream);
}

int hpd_nms(const HpdParams* p, const HpdBuffers* buf, float* nms_out, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return launch_nms(p, buf, nms_out, (cudaStream_t)stream);
}

int hpd_topk(const HpdParams* p, const HpdBuffers* buf, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return launch_topk(p, buf, (cudaStream_t)stream);
}

int hpd_group(const HpdParams* p, const HpdBuffers* buf, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return launch_group(p, buf, (cudaStream_t)stream);
}

int hpd_adjust_refine(const HpdParams* p, const HpdBuffers* buf, void* workspace, size_t workspace_bytes,
                      void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return launch_adjust_refine(p, buf, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hpd_resize_bilinear(const HpdMap* in, int batch, int channels, float* out, int out_h, int out_w, void* stream) {
  g_launches = 0;
  return launch_resize(in, batch, channels, out, out_h, out_w, (cudaStream_t)stream);
}

int hpd_record_layout(const HpdParams* p, HpdRecordLayout* out) {
  if (!p || !out) { set_error("NULL argument"); return HPD_EINVAL; }
  if (p->num_kpts < 1 || p->num_kpts > HPD_MAX_KPTS || p->max_people < 1 || p->max_people > HPD_MAX_PEOPLE || p->emb < 1 ||
      p->emb > HPD_MAX_EMB) {
    set_error("hpd_record_layout: num_kpts / max_people / emb out of range");
    return HPD_EINVAL;
  }
  *out = record_layout(p->num_kpts, p->max_people, p->emb);
  return HPD_OK;
}

int hpd_multi_scale_size(int img_h, int img_w, int input_size, double current_scale, double min_scale,
                         int32_t size_resized_wh[2], int32_t center_xy[2], double scale_wh[2]) {
  return multi_scale_size(img_h, img_w, input_size, current_scale, min_scale, size_resized_wh, center_xy, scale_wh);
}

int hpd_get_affine_transform(const double center_xy[2], const double scale_wh[2], const int32_t output_size_wh[2],
                             int inverse, double m_out[6]) {
  return affine_transform_matrix(center_xy, scale_wh, output_size_wh, inverse, m_out);
}

int hpd_prepare_geometry(int n, const int32_t* img_h, const int32_t* img_w, int input_size, double current_scale,
                         double min_scale, int32_t* size_resized_wh, int32_t* center_xy, double* scale_wh, double* m_forward,
                         double* m_inverse) {
  if (n < 1 || !img_h || !img_w || !size_resized_wh || !center_xy || !scale_wh || !m_forward || !m_inverse) {
    set_error("hpd_prepare_geometry: bad arguments");
    return HPD_EINVAL;
  }
  for (int i = 0; i < n; ++i) {
    int rc = multi_scale_size(img_h[i], img_w[i], input_size, current_scale, min_scale, size_resized_wh + 2 * i,
                              center_xy + 2 * i, scale_wh + 2 * i);
    if (rc) return rc;
    const double c[2] = {(double)center_xy[2 * i], (double)center_xy[2 * i + 1]};
    if ((rc = affine_transform_matrix(c, scale_wh + 2 * i, size_resized_wh + 2 * i, 0, m_forward + 6 * i))) return rc;
    if ((rc = affine_transform_matrix(c, scale_wh + 2 * i, size_resized_wh + 2 * i, 1, m_inverse + 6 * i))) return rc;
  }
  return HPD_OK;
}

int hpd_prepare_input(const HpdImage* images_host, int batch, float* out, int out_h, int out_w, const float mean[3],
                      const float std_[3], void* stream) {
  g_launches = 0;
  return launch_prepare_input(images_host, batch, out, out_h, out_w, mean, std_, (cudaStream_t)stream);
}

int hpd_prepare_inputs(const HpdImage* images_host, int batch, const HpdPrepareTarget* targets_host, int n_targets,
                       const float mean[3], const float std_[3], void* stream) {
  g_launches = 0;
  return launch_prepare_inputs(images_host, batch, targets_host, n_targets, mean, std_, (cudaStream_t)stream);
}

int hpd_coco_eval_workspace_bytes(const HpdCocoEvalParams* p, size_t* out_bytes) {
  if (!out_bytes) { set_error("NULL argument"); return HPD_EINVAL; }
  int rc = validate_coco_params(p);
  if (rc) return rc;
  *out_bytes = coco_eval_workspace_bytes(p, &rc);
  return rc;
}

int hpd_coco_eval(const HpdCocoEvalParams* p, const HpdCocoDets* dets, const HpdCocoGts* gts,
                  const HpdCocoEvalOutputs* outs, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = validate_coco_params(p);
  if (rc) return rc;
  return launch_coco_eval(p, dets, gts, outs, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hpd_track_state_bytes(const HpdTrackParams* p, size_t* out_bytes) {
  g_launches = 0;
  int rc = validate_track_params(p, "hpd_track_state_bytes");
  if (rc) return rc;
  if (!out_bytes) { set_error("hpd_track_state_bytes: out_bytes is NULL"); return HPD_EINVAL; }
  *out_bytes = track_state_bytes(p);
  return HPD_OK;
}

int hpd_track_reset(const HpdTrackParams* p, void* state, size_t state_bytes, int clear_ids, void* stream) {
  g_launches = 0;
  int rc = validate_track_params(p, "hpd_track_reset");
  if (rc) return rc;
  return launch_track_reset(p, state, state_bytes, clear_ids, (cudaStream_t)stream);
}

int hpd_track(const HpdTrackParams* p, const uint8_t* records, int n_frames, void* state, size_t state_bytes,
              int32_t* track_ids, void* stream) {
  g_launches = 0;
  int rc = validate_track_params(p, "hpd_track");
  if (rc) return rc;
  return launch_track(p, records, n_frames, state, state_bytes, track_ids, (cudaStream_t)stream);
}

int hpd_track_smooth_state_bytes(const HpdTrackParams* p, size_t* out_bytes) {
  g_launches = 0;
  int rc = validate_track_params(p, "hpd_track_smooth_state_bytes");
  if (rc) return rc;
  if (!out_bytes) { set_error("hpd_track_smooth_state_bytes: out_bytes is NULL"); return HPD_EINVAL; }
  *out_bytes = track_smooth_state_bytes(p);
  return HPD_OK;
}

int hpd_track_smooth(const HpdTrackParams* p, const HpdSmoothParams* sp, const uint8_t* records, int n_frames,
                     void* state, size_t state_bytes, int32_t* track_ids, double* coords, void* stream) {
  g_launches = 0;
  int rc = validate_track_params(p, "hpd_track_smooth");
  if (rc) return rc;
  return launch_track_smooth(p, sp, records, n_frames, state, state_bytes, track_ids, coords, (cudaStream_t)stream);
}

int hpd_render_poses(const HpdRenderParams* p, const HpdRenderFrame* frames_host, int n_frames, const uint8_t* records,
                     const int32_t* track_ids, const double* coords, void* stream) {
  g_launches = 0;
  return launch_render_poses(p, frames_host, n_frames, records, track_ids, coords, (cudaStream_t)stream);
}

int hpd_decode(const HpdParams* p, const HpdScaleInputs* scales, const HpdBuffers* buf, void* workspace,
               size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  HpdStageInputs st[HPD_MAX_SCALES];
  return decode_validated(p, as_stages(scales, p->num_scales, st), buf, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hpd_decode_stages(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, void* workspace,
                      size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = validate(p, buf);
  if (rc) return rc;
  return decode_validated(p, scales, buf, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"

namespace hpd {

// hpd_decode / hpd_decode_stages after validate()
static int decode_validated(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, void* workspace,
                            size_t workspace_bytes, cudaStream_t st) {
  int rc;
  HpdBuffers b = *buf;
  if (scales) {
    rc = launch_aggregate_nms(p, scales, &b, st);
    b.tag_inputs = tag_scale_inputs(scales[p->tag_scale]);   // the tag stages interpolate from these when agg_tags is NULL
  } else {
    rc = launch_nms(p, &b, nullptr, st);
  }
  if (rc) return rc;
  if ((rc = launch_topk(p, &b, st))) return rc;
  if ((rc = launch_group(p, &b, st))) return rc;
  return launch_adjust_refine(p, &b, workspace, workspace_bytes, st);
}

}  // namespace hpd
