// Input side of the inference path (SURVEY.md 8(f)-4): InferenceKeypointsModel.prepare_input
// (/root/reference/src/keypoints/model.py:70-76) = resize_align_multi_scale
// (/root/reference/src/base/transforms/utils.py:60-97) + T.ToTensor + T.Normalize (model.py:45-50).
//
// Host side (float64 like the reference, no device work):
//   hpd_multi_scale_size      get_multi_scale_size       utils.py:60-87
//   hpd_get_affine_transform  get_affine_transform       utils.py:25-57 (rot = 0, shift = 0: the only call shapes on
//                             this path, utils.py:95 and results.py:166) with cv2.getAffineTransform's solver replayed
// Device side:
//   warp_normalise_kernel     cv2.warpAffine(image, trans, size) with INTER_LINEAR / BORDER_CONSTANT(0) in OpenCV's
//                             fixed-point arithmetic, then x/255, (x-mean)/std in float32, HWC uint8 -> CHW float32.
// Both were pinned bit-for-bit against OpenCV 4.13 / torchvision 0.26 in the build container (oracle/input_oracle.py,
// tests/test_oracle_input.py, goldens in tests/golden/input_*.npz).
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace hpd {

namespace {

// ---- host geometry -----------------------------------------------------------------------------------------------
// Python's float floor division  a // b  (CPython floatobject.c: float_divmod)
double py_floordiv(double vx, double wx) {
  double mod = fmod(vx, wx);
  double div = (vx - mod) / wx;
  if (mod != 0.0 && ((wx < 0) != (mod < 0))) div -= 1.0;
  if (div == 0.0) return copysign(0.0, vx / wx);
  double fl = floor(div);
  if (div - fl > 0.5) fl += 1.0;
  return fl;
}

// cv::hal::LU64f as cv::solve(A, b, x, DECOMP_LU) runs it for getAffineTransform's 6x6 system: partial pivoting,
// rows scaled by -1/pivot, back substitution; plain float64 multiply/add in this order.
bool lu_solve6(double A[6][6], double b[6]) {
  const int m = 6;
  for (int i = 0; i < m; ++i) {
    int k = i;
    for (int j = i + 1; j < m; ++j)
      if (fabs(A[j][i]) > fabs(A[k][i])) k = j;
    if (fabs(A[k][i]) < 2.220446049250313e-16 * 100) return false;   // DBL_EPSILON*100, OpenCV's singularity test
    if (k != i) {
      for (int j = i; j < m; ++j) { const double t = A[i][j]; A[i][j] = A[k][j]; A[k][j] = t; }
      const double t = b[i]; b[i] = b[k]; b[k] = t;
    }
    const double d = -1 / A[i][i];
    for (int j = i + 1; j < m; ++j) {
      const double alpha = A[j][i] * d;
      for (int c = i + 1; c < m; ++c) A[j][c] += alpha * A[i][c];
      b[j] += alpha * b[i];
    }
  }
  for (int i = m - 1; i >= 0; --i) {
    double s = b[i];
    for (int c = i + 1; c < m; ++c) s -= A[i][c] * b[c];
    b[i] = s / A[i][i];
  }
  return true;
}

// ---- device warp ---------------------------------------------------------------------------------------------------
constexpr int kImagesPerLaunch = 32;
constexpr int kAbBits = 10, kInterBits = 5, kCoefBits = 15;   // OpenCV: AB_BITS, INTER_BITS, INTER_REMAP_COEF_BITS

struct WarpImage {
  const uint8_t* ptr;
  long long stride_row;
  int h, w;
  double im[6];   // inverse map (destination -> source), cv::warpAffine's own inversion of M
};

struct WarpArgs {
  WarpImage img[kImagesPerLaunch];
  float mean[3], stdv[3];
  float* out;     // [n,3,oh,ow] of this launch
  int oh, ow;
};

// hpd_prepare_inputs: one (target, image) pair per entry, each with its own output size and optional mirrored output
struct WarpEntry {
  WarpImage img;
  float* out;            // [3,oh,ow] of this image at this target
  float* out_flipped;    // [3,oh,ow] mirrored in x, or nullptr
  int oh, ow;
};

struct WarpTargetsArgs {
  WarpEntry e[kImagesPerLaunch];
  float mean[3], stdv[3];
};

__device__ __forceinline__ int cv_round_sat(double v) {   // saturate_cast<int>(double) = cvRound, half to even
  if (v >= 2147483647.0) return 2147483647;
  if (v <= -2147483648.0) return (-2147483647 - 1);
  return __double2int_rn(v);
}

constexpr int kWarpRows = 16;   // output rows per block

// Block = 256 output columns x kWarpRows rows of one image.  The float64 parts of OpenCV's coordinate arithmetic
// depend on the row alone (X0, Y0) or on the column alone (adelta, bdelta): the first are computed once per block row
// by 16 threads and shared, the second once per thread, so the per-pixel work is integer arithmetic, four 3-byte taps
// and three table look-ups (the first version redid eight float64 operations per pixel and was issue-bound at 0.43 TB/s).
// Both input kernels run this body, so their outputs agree bit for bit.  kFlip: every value is also stored at column
// ow-1-x of out_flipped (torch.flip(x, [3]) of the same tensor, without reading it back).
template <bool kFlip>
__device__ __forceinline__ void warp_normalise_block(const WarpImage& I, const float* mean, const float* stdv, float* out,
                                                     float* out_flipped, int oh, int ow) {
  __shared__ float lut[3][256];
  __shared__ int s_x0[kWarpRows], s_y0[kWarpRows];
  constexpr int AB_SCALE = 1 << kAbBits, ROUND_DELTA = AB_SCALE / (1 << kInterBits) / 2;
  const int y_first = blockIdx.y * kWarpRows;
  for (int i = threadIdx.x; i < 768; i += blockDim.x) {
    const int c = i >> 8, v = i & 255;
    // to_tensor: uint8 -> float32, div(255); normalize: sub_(mean).div_(std)
    lut[c][v] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, 255.0f), mean[c]), stdv[c]);
  }
  if (threadIdx.x < kWarpRows) {
    const double y = (double)(y_first + threadIdx.x);
    s_x0[threadIdx.x] = cv_round_sat(__dmul_rn(__dadd_rn(__dmul_rn(I.im[1], y), I.im[2]), (double)AB_SCALE)) + ROUND_DELTA;
    s_y0[threadIdx.x] = cv_round_sat(__dmul_rn(__dadd_rn(__dmul_rn(I.im[4], y), I.im[5]), (double)AB_SCALE)) + ROUND_DELTA;
  }
  __syncthreads();
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= ow) return;
  const int adelta = cv_round_sat(__dmul_rn(__dmul_rn(I.im[0], (double)x), (double)AB_SCALE));
  const int bdelta = cv_round_sat(__dmul_rn(__dmul_rn(I.im[3], (double)x), (double)AB_SCALE));
  const size_t plane = (size_t)oh * ow;
  float* o = out + (size_t)y_first * ow + x;
  float* of = kFlip ? out_flipped + (size_t)y_first * ow + (ow - 1 - x) : nullptr;
  const int rows = min(kWarpRows, oh - y_first);
#pragma unroll 4
  for (int r = 0; r < rows; ++r, o += ow) {
    const int X = (s_x0[r] + adelta) >> (kAbBits - kInterBits), Y = (s_y0[r] + bdelta) >> (kAbBits - kInterBits);
    const int sx = min(max(X >> kInterBits, -32768), 32767), sy = min(max(Y >> kInterBits, -32768), 32767);
    const int ax = X & 31, ay = Y & 31;
    // the bilinear table entries (1-fx)(1-fy), fx(1-fy), (1-fx)fy, fx*fy scaled by 2^15 are exact integers
    const int w00 = (32 - ax) * (32 - ay) * 32, w01 = ax * (32 - ay) * 32, w10 = (32 - ax) * ay * 32, w11 = ax * ay * 32;
    const bool x0in = sx >= 0 && sx < I.w, x1in = sx + 1 >= 0 && sx + 1 < I.w;
    const bool y0in = sy >= 0 && sy < I.h, y1in = sy + 1 >= 0 && sy + 1 < I.h;
    const uint8_t* r0 = I.ptr + (long long)sy * I.stride_row + (long long)sx * 3;
    const uint8_t* r1 = r0 + I.stride_row;
    if (x0in && x1in && y0in && y1in) {      // all four taps inside the image (nearly always): no per-tap tests
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int acc = (int)r0[c] * w00 + (int)r0[3 + c] * w01 + (int)r1[c] * w10 + (int)r1[3 + c] * w11;
        const float v = lut[c][(acc + (1 << (kCoefBits - 1))) >> kCoefBits];     // weights sum to 2^15: in 0..255
        o[(size_t)c * plane] = v;
        if (kFlip) of[(size_t)c * plane] = v;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int v00 = (y0in && x0in) ? r0[c] : 0, v01 = (y0in && x1in) ? r0[3 + c] : 0;
        const int v10 = (y1in && x0in) ? r1[c] : 0, v11 = (y1in && x1in) ? r1[3 + c] : 0;
        const int acc = v00 * w00 + v01 * w01 + v10 * w10 + v11 * w11;
        const int px = min(max((acc + (1 << (kCoefBits - 1))) >> kCoefBits, 0), 255);
        const float v = lut[c][px];
        o[(size_t)c * plane] = v;
        if (kFlip) of[(size_t)c * plane] = v;
      }
    }
    if (kFlip) of += ow;
  }
}

__global__ void __launch_bounds__(256) warp_normalise_kernel(const __grid_constant__ WarpArgs a) {
  const int n = blockIdx.z;
  warp_normalise_block<false>(a.img[n], a.mean, a.stdv, a.out + (size_t)n * 3 * a.oh * a.ow, nullptr, a.oh, a.ow);
}

// Grid (x, y) covers the largest target of the launch; blocks past their own entry's size leave at once.
__global__ void __launch_bounds__(256) warp_normalise_targets_kernel(const __grid_constant__ WarpTargetsArgs a) {
  const WarpEntry& e = a.e[blockIdx.z];
  if ((int)(blockIdx.x * blockDim.x) >= e.ow || (int)blockIdx.y * kWarpRows >= e.oh) return;
  if (e.out_flipped)
    warp_normalise_block<true>(e.img, a.mean, a.stdv, e.out, e.out_flipped, e.oh, e.ow);
  else
    warp_normalise_block<false>(e.img, a.mean, a.stdv, e.out, nullptr, e.oh, e.ow);
}

// cv::warpAffine without WARP_INVERSE_MAP inverts M itself, in this order
void invert_like_warp_affine(const double* m, double* im) {
  double M[6];
  memcpy(M, m, sizeof(M));
  double D = M[0] * M[4] - M[1] * M[3];
  D = D != 0 ? 1. / D : 0;
  const double A11 = M[4] * D, A22 = M[0] * D;
  M[0] = A11; M[1] *= -D;
  M[3] *= -D; M[4] = A22;
  const double b1 = -M[0] * M[2] - M[1] * M[5];
  const double b2 = -M[3] * M[2] - M[4] * M[5];
  M[2] = b1; M[5] = b2;
  memcpy(im, M, sizeof(M));
}

bool bad_image(const HpdImage& im) {
  return !im.ptr || im.h < 1 || im.w < 1 || im.h > 32767 || im.w > 32767 || im.stride_row < 3LL * im.w;
}

}  // namespace

int launch_prepare_input(const HpdImage* images, int batch, float* out, int oh, int ow, const float* mean,
                         const float* stdv, cudaStream_t st) {
  if (!images || !out || !mean || !stdv || batch < 1 || oh < 1 || ow < 1 || oh > 65535 * kWarpRows) {
    set_error("hpd_prepare_input: bad arguments");
    return HPD_EINVAL;
  }
  for (int b0 = 0; b0 < batch; b0 += kImagesPerLaunch) {
    const int n = batch - b0 < kImagesPerLaunch ? batch - b0 : kImagesPerLaunch;
    WarpArgs a;
    memset(&a, 0, sizeof(a));
    for (int i = 0; i < n; ++i) {
      const HpdImage& im = images[b0 + i];
      if (bad_image(im)) {
        set_error("hpd_prepare_input: image %d: bad pointer / size / stride", b0 + i);
        return HPD_EINVAL;
      }
      a.img[i].ptr = im.ptr; a.img[i].stride_row = im.stride_row; a.img[i].h = im.h; a.img[i].w = im.w;
      invert_like_warp_affine(im.m, a.img[i].im);
    }
    for (int c = 0; c < 3; ++c) { a.mean[c] = mean[c]; a.stdv[c] = stdv[c]; }
    a.out = out + (size_t)b0 * 3 * oh * ow;
    a.oh = oh; a.ow = ow;
    const dim3 grid((ow + 255) / 256, (oh + kWarpRows - 1) / kWarpRows, n);
    warp_normalise_kernel<<<grid, 256, 0, st>>>(a);
    count_launch();
    if (int rc = check_launch("warp_normalise_kernel")) return rc;
  }
  return HPD_OK;
}

int launch_prepare_inputs(const HpdImage* images, int batch, const HpdPrepareTarget* targets, int n_targets,
                          const float* mean, const float* stdv, cudaStream_t st) {
  if (!images || !targets || !mean || !stdv || batch < 1 || n_targets < 1 || n_targets > HPD_MAX_SCALES) {
    set_error("hpd_prepare_inputs: bad arguments (batch >= 1, 1 <= n_targets <= %d, non-NULL arrays)", HPD_MAX_SCALES);
    return HPD_EINVAL;
  }
  // everything is checked before the first launch: a rejected call enqueues nothing
  for (int t = 0; t < n_targets; ++t) {
    const HpdPrepareTarget& T = targets[t];
    if (!T.out || T.out_h < 1 || T.out_w < 1 || T.out_h > 65535 * kWarpRows) {
      set_error("hpd_prepare_inputs: target %d: bad output pointer / size", t);
      return HPD_EINVAL;
    }
    if (T.out_flipped == T.out) {
      set_error("hpd_prepare_inputs: target %d: out_flipped must not be out", t);
      return HPD_EINVAL;
    }
    for (int b = 0; b < batch; ++b) {
      if (bad_image(images[(size_t)t * batch + b])) {
        set_error("hpd_prepare_inputs: target %d image %d: bad pointer / size / stride", t, b);
        return HPD_EINVAL;
      }
    }
  }
  const long long total = (long long)n_targets * batch;
  for (long long e0 = 0; e0 < total; e0 += kImagesPerLaunch) {
    const int n = total - e0 < kImagesPerLaunch ? (int)(total - e0) : kImagesPerLaunch;
    WarpTargetsArgs a;
    memset(&a, 0, sizeof(a));
    int max_h = 0, max_w = 0;
    for (int i = 0; i < n; ++i) {
      const long long e = e0 + i;          // entry e = image b of target t, images_host's order
      const int t = (int)(e / batch), b = (int)(e % batch);
      const HpdImage& im = images[e];
      const HpdPrepareTarget& T = targets[t];
      const size_t img_elems = (size_t)3 * T.out_h * T.out_w;
      WarpEntry& E = a.e[i];
      E.img.ptr = im.ptr; E.img.stride_row = im.stride_row; E.img.h = im.h; E.img.w = im.w;
      invert_like_warp_affine(im.m, E.img.im);
      E.out = T.out + (size_t)b * img_elems;
      E.out_flipped = T.out_flipped ? T.out_flipped + (size_t)b * img_elems : nullptr;
      E.oh = T.out_h; E.ow = T.out_w;
      max_h = max_h > T.out_h ? max_h : T.out_h;
      max_w = max_w > T.out_w ? max_w : T.out_w;
    }
    for (int c = 0; c < 3; ++c) { a.mean[c] = mean[c]; a.stdv[c] = stdv[c]; }
    const dim3 grid((max_w + 255) / 256, (max_h + kWarpRows - 1) / kWarpRows, n);
    warp_normalise_targets_kernel<<<grid, 256, 0, st>>>(a);
    count_launch();
    if (int rc = check_launch("warp_normalise_targets_kernel")) return rc;
  }
  return HPD_OK;
}

int multi_scale_size(int h, int w, int input_size, double current_scale, double min_scale, int32_t* size_wh,
                     int32_t* center_xy, double* scale_wh) {
  if (h < 1 || w < 1 || input_size < 1 || !(current_scale > 0) || !(min_scale > 0) || !size_wh || !center_xy || !scale_wh) {
    set_error("hpd_multi_scale_size: bad arguments");
    return HPD_EINVAL;
  }
  center_xy[0] = (int32_t)(w / 2.0 + 0.5);
  center_xy[1] = (int32_t)(h / 2.0 + 0.5);
  const long long min_input = (long long)(py_floordiv(min_scale * input_size + 63, 64) * 64);
  if (w < h) {
    const int wr = (int)((double)min_input * current_scale / min_scale);
    const long long hr64 = (long long)(py_floordiv((double)min_input / w * h + 63, 64) * 64);
    const int hr = (int)((double)hr64 * current_scale / min_scale);
    size_wh[0] = wr; size_wh[1] = hr;
    scale_wh[0] = (double)w;
    scale_wh[1] = (double)hr / wr * w;
  } else {
    const int hr = (int)((double)min_input * current_scale / min_scale);
    const long long wr64 = (long long)(py_floordiv((double)min_input / h * w + 63, 64) * 64);
    const int wr = (int)((double)wr64 * current_scale / min_scale);
    size_wh[0] = wr; size_wh[1] = hr;
    scale_wh[1] = (double)h;
    scale_wh[0] = (double)wr / hr * h;
  }
  return HPD_OK;
}

int affine_transform_matrix(const double* center, const double* scale, const int32_t* out_wh, int inverse, double* m) {
  if (!center || !scale || !out_wh || !m) {
    set_error("hpd_get_affine_transform: NULL argument");
    return HPD_EINVAL;
  }
  const double dst_w = out_wh[0], dst_h = out_wh[1];
  float src[3][2], dst[3][2];
  // rot = 0: src_dir = (0*1 - (-w/2)*0, 0*0 + (-w/2)*1); shift = 0 adds +0.0 terms
  const double dir_x = 0.0 * 1.0 - (-scale[0] / 2) * 0.0, dir_y = 0.0 * 0.0 + (-scale[0] / 2) * 1.0;
  src[0][0] = (float)(center[0] + scale[0] * 0.0);
  src[0][1] = (float)(center[1] + scale[1] * 0.0);
  src[1][0] = (float)(center[0] + dir_x + scale[0] * 0.0);
  src[1][1] = (float)(center[1] + dir_y + scale[1] * 0.0);
  const float dst_dir_y = (float)(-dst_w / 2);
  dst[0][0] = (float)(dst_w * 0.5);
  dst[0][1] = (float)(dst_h * 0.5);
  dst[1][0] = (float)(dst_w * 0.5 + (double)0.0f);
  dst[1][1] = (float)(dst_h * 0.5 + (double)dst_dir_y);
  auto third = [](const float a[2], const float b[2], float out[2]) {   // b + (-(a-b).y, (a-b).x), float32
    const float dx = a[0] - b[0], dy = a[1] - b[1];
    out[0] = b[0] + (-dy);
    out[1] = b[1] + dx;
  };
  third(src[0], src[1], src[2]);
  third(dst[0], dst[1], dst[2]);
  const float(*from)[2] = inverse ? dst : src;
  const float(*to)[2] = inverse ? src : dst;
  double A[6][6], b[6];
  memset(A, 0, sizeof(A));
  for (int i = 0; i < 3; ++i) {
    A[2 * i][0] = A[2 * i + 1][3] = from[i][0];
    A[2 * i][1] = A[2 * i + 1][4] = from[i][1];
    A[2 * i][2] = A[2 * i + 1][5] = 1;
    b[2 * i] = to[i][0];
    b[2 * i + 1] = to[i][1];
  }
  if (!lu_solve6(A, b)) memset(b, 0, sizeof(b));   // cv::solve leaves zeros for a singular system
  memcpy(m, b, 6 * sizeof(double));
  return HPD_OK;
}

}  // namespace hpd
