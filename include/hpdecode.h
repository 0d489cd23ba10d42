/* hpdecode -- B200 (sm_100a) bottom-up keypoint decode: C ABI of libhpdecode.so
 *
 * Drop-in boundary for the HigherHRNet decode path of thawro/pytorch-human-pose.  The
 * reference has no FFI layer (it is pure Python); each entry point below is the device twin
 * of one reference method, cited as /root/reference-relative file:line.  INTEGRATION.md shows
 * the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer unless the name ends in _host.  The caller owns every
 *    buffer; the library allocates nothing, never synchronises, and enqueues all work on the
 *    given stream (a cudaStream_t passed as void*; NULL = the legacy default stream).
 *  - All maps the library writes are float32.  Network outputs are float32, float16 or bfloat16 NCHW views with explicit batch / channel
 *    strides in ELEMENTS and contiguous rows (HigherHRNet's hm_lo / tag are channel slices of
 *    one 34-channel tensor: src/keypoints/architectures/higher_hrnet.py:78-79).
 *  - Return value: 0 on success, an HPD_E* code otherwise; hpd_last_error_string() gives the
 *    message of the calling thread's last failure.  No C++ exception crosses the ABI.
 *  - Re-entrant: one workspace per in-flight call; safe from one host thread per GPU.
 *  - Inputs must be finite (NaN ordering of torch.topk / MaxPool2d is not reproduced).  hpd_group alone returns on
 *    any top-k tensors: costs it cannot solve on are guarded and reported in flags bit 1.
 */
#ifndef HPDECODE_H_
#define HPDECODE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HPD_EXPORT __attribute__((visibility("default")))
#else
#define HPD_EXPORT
#endif

#define HPD_ABI_VERSION 6
#define HPD_MAX_KPTS 32     /* joints per person (COCO: 17) */
#define HPD_MAX_PEOPLE 32   /* max_num_people == top-k; the warp-wide Hungarian handles n <= 32 */
#define HPD_MAX_EMB 2       /* tag embedding dims: 1 (no flip test) or 2 (flip test) */
#define HPD_MAX_SCALES 4    /* test scales averaged into one heatmap */
#define HPD_COCO_MAX_IOU_THRS 16    /* COCO keypoint evaluation: OKS thresholds (pycocotools: 10) */
#define HPD_COCO_MAX_REC_THRS 128   /* recall thresholds (pycocotools: 101) */
#define HPD_COCO_MAX_AREAS 4        /* area ranges (pycocotools keypoints: all, medium, large) */
#define HPD_COCO_MAX_PER_IMAGE 1024 /* detections, and ground-truth annotations, per image */

enum {
  HPD_OK = 0,
  HPD_EINVAL = 1,       /* bad argument / unsupported shape */
  HPD_EWORKSPACE = 2,   /* workspace too small */
  HPD_ECUDA = 3         /* a CUDA call failed (launch configuration, etc.) */
};

enum {
  HPD_F32 = 0,          /* float32 maps (inference path, model.py:78-111) */
  HPD_F16 = 1,          /* IEEE half maps: the validation-time caller runs the net under autocast
                         * (module.py:78,100-110); values are widened on load, all arithmetic stays float32 */
  HPD_BF16 = 2          /* bfloat16 maps (the net under bf16 autocast): widened exactly on load like HPD_F16 */
};

/* One NCHW tensor view. */
typedef struct HpdMap {
  const void* ptr;    /* NULL = absent */
  int64_t stride_b;   /* elements between images */
  int64_t stride_c;   /* elements between channels; rows are contiguous (stride_y == w) */
  int32_t h, w;
  int32_t dtype;      /* HPD_F32, HPD_F16 or HPD_BF16; all maps of one call share it (hpd_resize_bilinear: HPD_F32) */
  int32_t reserved_;
} HpdMap;

/* Raw network outputs for one test scale: the un-flipped forward and, when the flip test is on,
 * the forward of the horizontally flipped image (model.py:83-86). */
typedef struct HpdScaleInputs {
  HpdMap hm_lo, hm_hi, tag;         /* stage-1 heatmaps (S/4), stage-2 heatmaps (S/2), tags (S/4) */
  HpdMap hm_lo_f, hm_hi_f, tag_f;   /* flipped run; ptr == NULL when flip test is off */
} HpdScaleInputs;

/* Raw network outputs for one test scale, for a head with 1 to HPD_MAX_STAGES heatmap stages (results.py:46-54,226
 * take them as a list): HRNet with the associative-embedding head and no deconvolution gives one stage at S/4,
 * HigherHRNet two (S/4, S/2), HigherHRNet with two deconvolution modules three (S/4, S/2, S).  Every stage is flip
 * averaged, stages 0..n-2 are resized to the last stage's size, and their mean ((U_0 + U_1) + ...) / n is taken
 * there.  HpdScaleInputs is the two-stage case: {hm = {hm_lo, hm_hi}, num_stages = 2}. */
#define HPD_MAX_STAGES 4
typedef struct HpdStageInputs {
  HpdMap hm[HPD_MAX_STAGES];    /* heatmap stages in the network's order; the mean is taken at hm[num_stages-1]'s size */
  HpdMap hm_f[HPD_MAX_STAGES];  /* flipped run; ptr NULL when the flip test is off */
  HpdMap tag, tag_f;            /* as in HpdScaleInputs */
  int32_t num_stages;           /* 1..HPD_MAX_STAGES */
  int32_t reserved_;
} HpdStageInputs;

typedef struct HpdParams {
  int32_t batch;        /* B images per call */
  int32_t num_kpts;     /* K <= HPD_MAX_KPTS */
  int32_t out_h, out_w; /* H, W of the aggregated maps == network input size (results.py:219) */
  int32_t emb;          /* E: 1 or 2 (2 iff flip inputs are given to the aggregate stage) */
  int32_t max_people;   /* M = max_num_people = top-k (grouping.py:70,153); H*W >= 64*M required */
  int32_t num_scales;   /* heatmaps are averaged over this many scales (1 in the reference) */
  int32_t tag_scale;    /* index of the scale whose tag maps are used */
  int32_t do_adjust;    /* grouping.py:274 */
  int32_t do_refine;    /* grouping.py:278 */
  int32_t tags_preflipped; /* 1: tag_f is already un-flipped and joint-permuted, i.e. it is the second entry of
                            * the reference's tags_heatmaps list (model.py:91-94) as from_preds receives it */
  int32_t force_generic; /* testing only, 0 in production.  bit 0: generic aggregation kernel instead of the specialised
                          * ones, and in top-k the literal libstdc++ heap code (one lane, shared memory) over the whole
                          * row instead of the floor mode / warp-wide heap; bit 1: one warp per row in top-k even for
                          * small batches; bit 2: rows with ties are streamed by that one warp instead of being handed
                          * to the second (8 warps per row) launch.  All variants are bit-identical (tests). */
  int32_t batches_in_flight; /* hint, 0 or 1 = unknown / latency matters: small batches (<= 512 rows) give every top-k row eight
                          * warps; >= 8: the caller keeps that many batches in flight (DecodePipeline), so the row gets one
                          * warp and the batches overlap instead (+5 % throughput at 8-16 images per batch).  Same results. */
  int32_t reserved_;
  double det_thr;       /* grouping.py:71,100  (compared in float64) */
  double tag_thr;       /* grouping.py:72,135  (compared in float64) */
  int32_t flip_index[HPD_MAX_KPTS];   /* COCO_FLIP_INDEX (transforms.py:11) */
  int32_t joints_order[HPD_MAX_KPTS]; /* MPPEHeatmapParser.joints_order (grouping.py:63-65) */
} HpdParams;

/* Device buffers written by the stages.  WPR = (W + 31) / 32 words per image row.
 * Every field but agg_tags / tag_inputs is required by hpd_decode; single-stage calls document what they touch. */
typedef struct HpdBuffers {
  float* agg_hm;        /* [B,K,H,W]      aggregated heatmaps (results.py:227)                  */
  float* agg_tags;      /* [B,K,H,W,E]    resized tags, E innermost (results.py:229-230).  May be NULL: the
                         * tag stages then interpolate the tags they read from tag_inputs (bit-identical), and
                         * hpd_aggregate_tags writes the map on demand                                          */
  uint32_t* nms_mask;   /* [B,K,H,WPR]    bit x%32 of word (y, x/32): pixel survives NMS         */
  float* nms_wmax;      /* [B,K,H,WPR]    max of the NMS'd values of the word's pixels           */
  float* hm_wmax;       /* [B,K,H,WPR]    max of the raw aggregated values of the word's pixels  */
  float* scores_k;      /* [B,K,M]        top-k values, torch CPU order (grouping.py:153)        */
  int32_t* idx_k;       /* [B,K,M]        flat indices y*W+x                                     */
  int32_t* coords_k;    /* [B,K,M,2]      (x, y) (grouping.py:163-165)                           */
  float* tags_k;        /* [B,K,M,E]      (grouping.py:158-161)                                  */
  float* poses;         /* [B,M,K,3+E]    grouped joints [x,y,score,tag..]; zero-filled rows     */
  float* person_scores; /* [B,M]          grouping.py:276                                        */
  int32_t* n_person;    /* [B]            persons returned (<= M)                                */
  int32_t* flags;       /* [B]            bit0: empty-scene fallback fired (grouping.py:262-269);
                         * bit1: grouping guarded a cost the reference's munkres never returns on -- NaN, +-inf or
                         * |cost| >= 2^63 (from NaN / inf tags or scores, or tags ~1e17 apart) was replaced by 1e10
                         * (grouping.py:126-128's "cannot match" value), or a solve reached its step-6 cap and left
                         * that joint's detections unmatched.  Never set on finite inputs of the reference's range. */
  float* tag_bmin;      /* [B,K,HB,WPR]   HB = (H+3)/4: lower / upper bound of the first tag component over     */
  float* tag_bmax;      /* [B,K,HB,WPR]   4 image rows x one 32-pixel word (refine prefilter; -inf/+inf = none) */
  uint8_t* records;     /* [B][row_bytes] optional (NULL = not written): one result record per image, laid out as
                         * hpd_record_layout() says; written by the epilogue of hpd_adjust_refine / hpd_decode     */
  const double* inv_affine; /* [B][6] optional: per-image 2x3 matrix (row major) that maps network-input pixels back
                         * to the raw image, i.e. get_affine_transform(center, scale, 0, (W, H), inverse=True)
                         * (results.py:158-171, base/transforms/utils.py:25-57).  NULL = identity              */
  HpdScaleInputs tag_inputs; /* read only when agg_tags is NULL: the tag-scale network outputs (tag, and tag_f when
                         * E == 2; the other maps are ignored) the tag stages interpolate from.  hpd_decode fills it
                         * from scales[tag_scale] itself; hpd_topk / hpd_adjust_refine need it from the caller */
} HpdBuffers;

/* Layout of one result record (all offsets in bytes from the start of the image's row; row_bytes % 8 == 0).
 * The record is everything the reference's callers read after a decode, ready for ONE device->host copy:
 *   coco          f64 [M][3K+1]  per person (x, y, 1) * K then the person score: the "keypoints" list and "score"
 *                                of evaluate_dataset's COCO record (bin/eval.py:31-47) with x, y back-projected to
 *                                the raw image (results.py:158-171,189-201,244).  Persons >= n_person: zeros.
 *                                Like the reference, back-projected coordinates are rounded to float32 (they are
 *                                written into a float32 array, results.py:165-170) -- except in the empty-scene
 *                                fallback, whose pseudo-person is float64 throughout (grouping.py:262-269).
 *   poses         f32 [M][K][3+E] grouped joints in network-input pixels (x, y, score, tags), grouping.py:283
 *   person_scores f32 [M]        grouping.py:276
 *   n_person      i32            persons returned
 *   flags         i32            bit 0: empty-scene fallback fired; bit 1: grouping guarded a cost (HpdBuffers)  */
typedef struct HpdRecordLayout {
  int64_t row_bytes;
  int64_t off_coco, off_poses, off_person_scores, off_n_person, off_flags;
  int32_t coco_stride;  /* doubles per person: 3K + 1 */
  int32_t reserved_;
} HpdRecordLayout;

/* One raw image for hpd_prepare_input: uint8, HWC, 3 channels, resident on the device. */
typedef struct HpdImage {
  const uint8_t* ptr;
  int64_t stride_row;   /* bytes between rows (>= 3*w) */
  int32_t h, w;
  double m[6];          /* the forward 2x3 matrix cv2.warpAffine receives (base/transforms/utils.py:95-96) */
} HpdImage;

/* ---- COCO keypoint evaluation (pycocotools COCOeval, iouType "keypoints": evaluate + accumulate) ------------
 * One category (person).  Images are given in ascending image-id order (COCOeval's p.imgIds), so image index order is
 * the order accumulate concatenates them in.  Everything that decides a result is float64. */
typedef struct HpdCocoEvalParams {
  int32_t num_images;   /* I */
  int32_t num_kpts;     /* K <= HPD_MAX_KPTS */
  int32_t max_dets;     /* maxDets[-1] <= HPD_MAX_PEOPLE: detections kept per image, by score */
  int32_t max_gts;      /* G <= HPD_COCO_MAX_PER_IMAGE: ground-truth slots per image in HpdCocoGts */
  int32_t num_iou_thrs; /* T <= HPD_COCO_MAX_IOU_THRS */
  int32_t num_rec_thrs; /* R <= HPD_COCO_MAX_REC_THRS */
  int32_t num_areas;    /* A <= HPD_COCO_MAX_AREAS */
  int32_t reserved_;
  double iou_thrs[HPD_COCO_MAX_IOU_THRS];   /* p.iouThrs, as NumPy computed them (np.linspace) */
  double rec_thrs[HPD_COCO_MAX_REC_THRS];   /* p.recThrs */
  double area_rng[HPD_COCO_MAX_AREAS][2];   /* p.areaRng: [lo, hi], inclusive */
  double kpt_vars[HPD_MAX_KPTS];            /* (p.kpt_oks_sigmas * 2) ** 2, as NumPy computed them */
} HpdCocoEvalParams;

/* Detections, read in place: image i's row starts at base + row_offset[i] bytes (row_offset[i] < 0: the image has no
 * detections).  A row holds an int32 count n at +off_count and n persons of [x, y, v] * K + score (float64) at
 * +off_coco, person_stride doubles apart -- the COCO section of decode result records (HpdRecordLayout: off_coco,
 * off_n_person, coco_stride), or rows packed from result dicts.  Persons are in the order of the results list: score
 * ties are broken by it.  Counts are read as min(max(n, 0), max_per_row).  Scores must not be NaN. */
typedef struct HpdCocoDets {
  const uint8_t* base;
  const int64_t* row_offset;  /* [I] device */
  int64_t off_coco;           /* multiple of 8 (base + row_offset[i] must be 8-byte aligned too) */
  int64_t off_count;          /* multiple of 4 */
  int32_t person_stride;      /* doubles between persons, >= 3K + 1 */
  int32_t max_per_row;        /* D <= HPD_COCO_MAX_PER_IMAGE */
} HpdCocoDets;

/* Ground truth, padded to G = params.max_gts per image, annotations of an image in dataset order. */
typedef struct HpdCocoGts {
  const double* kpts;       /* [I][G][K][3] x, y, v */
  const double* area;       /* [I][G] the annotation's area */
  const double* bbox;       /* [I][G][4] x, y, w, h */
  const uint8_t* iscrowd;   /* [I][G] */
  const uint8_t* ignore;    /* [I][G] iscrowd || num_keypoints == 0 (COCOeval._prepare) */
  const int32_t* n_gt;      /* [I] annotations of the image (<= G) */
} HpdCocoGts;

enum { HPD_COCO_ABSENT = 0, HPD_COCO_TP = 1, HPD_COCO_FP = 2, HPD_COCO_IGNORED = 3 };

/* accumulate's arrays for the one category and the one maxDets entry, -1 where no gt is non-ignored (npig == 0). */
typedef struct HpdCocoEvalOutputs {
  double* precision;  /* [T][R][A] */
  double* recall;     /* [T][A] */
  double* scores;     /* [T][R][A] */
  double* oks;        /* optional [I][max_dets][G]: computeOks per image (score rank x gt), 0 outside n_dets x n_gt */
  uint8_t* codes;     /* optional [A][T][I][max_dets]: HPD_COCO_* of each (area, threshold, image, score rank) */
  int64_t* npig;      /* optional [A]: non-ignored gts per area range */
} HpdCocoEvalOutputs;

HPD_EXPORT int hpd_abi_version(void);
HPD_EXPORT const char* hpd_last_error_string(void);

/* Bytes of scratch hpd_decode / hpd_adjust_refine need for these params. */
HPD_EXPORT int hpd_workspace_bytes(const HpdParams* p, size_t* out_bytes);

/* (a)+(b) fused aggregation + NMS: model.py:85-96, results.py:46-67,225-230, grouping.py:80-83.
 * Reads scales[0..num_scales); writes agg_hm, nms_mask, nms_wmax, hm_wmax, tag_bmin, tag_bmax in one kernel, and
 * agg_tags unless it is NULL: the tag map is written by a second kernel on the same stream, the one
 * hpd_aggregate_tags launches (hpd_last_launch_count() is then one higher). */
HPD_EXPORT int hpd_aggregate_nms(const HpdParams* p, const HpdScaleInputs* scales, const HpdBuffers* buf, void* stream);

/* hpd_aggregate_nms for heads with 1..HPD_MAX_STAGES heatmap stages per scale (HpdStageInputs).  hpd_aggregate_nms is
 * this call with two stages.  Flipped maps are given for every stage of every scale or for none, each with its stage's
 * shape; all maps share one dtype.  Everything is checked before the first launch. */
HPD_EXPORT int hpd_aggregate_nms_stages(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf,
                                        void* stream);

/* The tag half of hpd_aggregate_nms alone (results.py:229-230), for callers that decoded with agg_tags == NULL and
 * want the map after all: reads the tag / tag_f maps of scales[tag_scale]; writes out [B,K,H,W,E].  It is the one
 * producer of the map: hpd_aggregate_nms and hpd_decode fill agg_tags with the same kernel. */
HPD_EXPORT int hpd_aggregate_tags(const HpdParams* p, const HpdScaleInputs* scales, float* out, void* stream);

/* Standalone bilinear resize with torch's CPU arithmetic (BaseKeypointsResult.match_heatmaps_size,
 * resize_heatmaps_list, resize_heatmaps: results.py:46-67).  in: [batch,channels,h,w] view;
 * out: contiguous [batch,channels,out_h,out_w]. */
HPD_EXPORT int hpd_resize_bilinear(const HpdMap* in, int batch, int channels, float* out, int out_h, int out_w,
                                   void* stream);

/* (b) alone, for callers that hand in aggregated maps (MPPEHeatmapParser.parse/top_k/nms,
 * grouping.py:80-83,150): reads agg_hm; writes nms_mask, nms_wmax, hm_wmax, tag_bmin/bmax (= no bound) and, if nms_out is
 * not NULL, the float NMS'd map [B,K,H,W] exactly as the reference's nms() returns it. */
HPD_EXPORT int hpd_nms(const HpdParams* p, const HpdBuffers* buf, float* nms_out, void* stream);

/* (c) per-joint top-k with torch-CPU (std::partial_sort) tie order: grouping.py:147-170.
 * Reads agg_hm, agg_tags (or tag_inputs), nms_mask, nms_wmax; writes scores_k, idx_k, coords_k, tags_k. */
HPD_EXPORT int hpd_topk(const HpdParams* p, const HpdBuffers* buf, void* stream);

/* (d) associative-embedding grouping: grouping.py:85-145 + py_max_match :55-59 + fallback :262-269.
 * Reads scores_k, coords_k, tags_k; writes poses, n_person, flags.  Returns on every input: see flags bit 1. */
HPD_EXPORT int hpd_group(const HpdParams* p, const HpdBuffers* buf, void* stream);

/* (e) adjust + person score + refine: grouping.py:172-191, :276, :193-250.
 * Reads agg_hm, agg_tags (or tag_inputs), hm_wmax, tag_bmin, tag_bmax, idx_k, scores_k, tags_k (refine: the tags at idx_k, as
 * hpd_topk writes them), n_person, flags; updates poses in place;
 * writes person_scores and, if buf->records is given, the per-image result records (back-projection through
 * buf->inv_affine + COCO layout, results.py:158-201,240-244, bin/eval.py:31-47) in the epilogue of its last kernel. */
HPD_EXPORT int hpd_adjust_refine(const HpdParams* p, const HpdBuffers* buf, void* workspace, size_t workspace_bytes,
                      void* stream);

/* Whole path: hpd_aggregate_nms -> hpd_topk -> hpd_group -> hpd_adjust_refine on one stream.
 * If scales == NULL the aggregation is skipped and buf->agg_hm / agg_tags are taken as inputs
 * (the MPPEHeatmapParser.parse entry, grouping.py:252).  With scales and agg_tags == NULL the tag stages read
 * scales[tag_scale] (buf->tag_inputs is ignored); the network outputs must then stay unchanged until the call's
 * work has run.  With scales and a non-NULL agg_tags the map is written as hpd_aggregate_nms writes it (one launch
 * more) and the tag stages read it. */
HPD_EXPORT int hpd_decode(const HpdParams* p, const HpdScaleInputs* scales, const HpdBuffers* buf, void* workspace,
               size_t workspace_bytes, void* stream);

/* hpd_decode over HpdStageInputs (1..HPD_MAX_STAGES heatmap stages per scale); hpd_decode is this call with two
 * stages.  The tag stages read the tag / tag_f maps of scales[tag_scale] as hpd_decode's do. */
HPD_EXPORT int hpd_decode_stages(const HpdParams* p, const HpdStageInputs* scales, const HpdBuffers* buf, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* Offsets and size of the per-image result record for these params (num_kpts, max_people, emb). */
HPD_EXPORT int hpd_record_layout(const HpdParams* p, HpdRecordLayout* out);

/* ---- input side (SURVEY 8(f)-4): InferenceKeypointsModel.prepare_input, model.py:70-76 ---------------------
 * Host-side geometry, float64 like the reference (no device work, no stream):
 * get_multi_scale_size (base/transforms/utils.py:60-87): resized (w, h), center, scale of an img_h x img_w image. */
HPD_EXPORT int hpd_multi_scale_size(int img_h, int img_w, int input_size, double current_scale, double min_scale,
                                    int32_t size_resized_wh[2], int32_t center_xy[2], double scale_wh[2]);

/* get_affine_transform(center, scale, rot=0, output_size, inverse) (base/transforms/utils.py:25-57): float32 point
 * triples, then cv2.getAffineTransform's 6x6 LU solve replayed in float64 (bit-identical to OpenCV 4.x). */
HPD_EXPORT int hpd_get_affine_transform(const double center_xy[2], const double scale_wh[2], const int32_t output_size_wh[2],
                                        int inverse, double m_out[6]);

/* Both of the above for n images in one call (the batched evaluation loop): per image i the resized size, center, scale,
 * the forward matrix (for hpd_prepare_input) and the inverse one (for HpdBuffers.inv_affine). */
HPD_EXPORT int hpd_prepare_geometry(int n, const int32_t* img_h, const int32_t* img_w, int input_size, double current_scale,
                                    double min_scale, int32_t* size_resized_wh /*[n][2]*/, int32_t* center_xy /*[n][2]*/,
                                    double* scale_wh /*[n][2]*/, double* m_forward /*[n][6]*/, double* m_inverse /*[n][6]*/);

/* resize_align_multi_scale's cv2.warpAffine (INTER_LINEAR, BORDER_CONSTANT 0; base/transforms/utils.py:96) followed by
 * T.ToTensor + T.Normalize (model.py:45-50): images_host[b] (uint8 HWC on the device, descriptors on the host) ->
 * out [batch,3,out_h,out_w] float32.  The warp replays OpenCV's fixed-point arithmetic (10-bit coordinates, 5-bit
 * sub-pixel positions, 15-bit weights) and the normalisation torch's float32 sequence, so out is bit-identical to
 * the reference's tensor.  mean / std: 3 floats each (host). */
HPD_EXPORT int hpd_prepare_input(const HpdImage* images_host, int batch, float* out, int out_h, int out_w,
                                 const float mean[3], const float std_[3], void* stream);

/* One output of hpd_prepare_inputs: a test scale's network input [batch,3,out_h,out_w] float32 and, optionally, its
 * horizontally mirrored copy (the flip-test input, model.py:86), same shape. */
typedef struct HpdPrepareTarget {
  float* out;
  float* out_flipped;   /* NULL = none; must not equal out */
  int32_t out_h, out_w;
} HpdPrepareTarget;

/* hpd_prepare_input for every test scale of a batch in one pass: images_host[t*batch + b] is image b with the forward
 * matrix of target t (the same image pointer for every t, normally).  targets_host[t].out receives exactly what
 * hpd_prepare_input writes for those descriptors, and out_flipped[b][c][y][out_w-1-x] = out[b][c][y][x] (a second store
 * of the same value: bit-identical to torch.flip(out, [3]), no extra read).  n_targets <= HPD_MAX_SCALES.  Up to 32
 * (target, image) pairs go in one launch; larger calls are split (hpd_last_launch_count).  Every argument is checked
 * before the first launch. */
HPD_EXPORT int hpd_prepare_inputs(const HpdImage* images_host, int batch, const HpdPrepareTarget* targets_host,
                                  int n_targets, const float mean[3], const float std_[3], void* stream);

/* Bytes of scratch hpd_coco_eval needs for these params. */
HPD_EXPORT int hpd_coco_eval_workspace_bytes(const HpdCocoEvalParams* p, size_t* out_bytes);

/* COCOeval(gt, dt, "keypoints").evaluate() + accumulate() (pycocotools cocoeval.py): OKS per image, the greedy
 * matching of every (area range, threshold), a stable global score order, and the precision / recall / score arrays.
 * The summary statistics are a mean over these arrays, left to the host (hpdecode.cocoeval). */
HPD_EXPORT int hpd_coco_eval(const HpdCocoEvalParams* p, const HpdCocoDets* dets, const HpdCocoGts* gts,
                             const HpdCocoEvalOutputs* outs, void* workspace, size_t workspace_bytes, void* stream);

/* ---- person tracking across frames (greedy OKS matching, the tracker of mmpose's video demos) ------------------
 * Frames are result records (HpdRecordLayout for num_kpts, max_people, emb) in time order.  Per frame, its persons
 * are visited in descending person score (ties: lower index).  Each takes the live track, not yet claimed in this
 * frame, with the highest OKS against the pose that last matched it (ties: smaller id), if that OKS is > oks_thr;
 * otherwise it starts a new track (ids 0, 1, ... never reused) if it has >= min_keypoints visible joints, or gets -1.
 * Tracks started in a frame are not candidates in that frame.  Unclaimed tracks age by one per frame and are dropped
 * at age max_age.  OKS: over the joints visible in both poses (poses[.][k][2] > 0; none: 0), with the COCO-section
 * coordinates, s = the mean of the two poses' areas (bounding box of the visible joints; 0 below two) and
 *   e_k = (dx*dx + dy*dy) / kpt_vars[k] / (s + 2^-52) / 2,  OKS = np.sum(exp(-e)) / |J|   (float64, NumPy's order).
 * A frame whose flags bit 0 is set (the empty-scene fallback) has no persons.  Person scores must not be NaN. */
typedef struct HpdTrackParams {
  int32_t num_kpts;       /* K <= HPD_MAX_KPTS */
  int32_t max_people;     /* M <= HPD_MAX_PEOPLE: persons per record */
  int32_t emb;            /* E of the records: 1 or 2 */
  int32_t max_age;        /* 1..HPD_TRACK_MAX_AGE: a track unclaimed for max_age frames is dropped */
  int32_t min_keypoints;  /* 0..K visible joints a person needs to start a track */
  int32_t reserved_;
  double oks_thr;         /* a match needs OKS > oks_thr (finite) */
  double kpt_vars[HPD_MAX_KPTS];   /* (2 sigma_k)^2, finite and > 0: cocoeval's kpt_vars for COCO's sigmas */
} HpdTrackParams;
#define HPD_TRACK_MAX_AGE 8

/* Bytes of the tracker state for these params (room for max_people * max_age tracks).  The layout is private. */
HPD_EXPORT int hpd_track_state_bytes(const HpdTrackParams* p, size_t* out_bytes);

/* Drops every track of the state (with a smoothing state, their filters too).  clear_ids = 1 also restarts the ids at
 * 0: a new state must be reset so once before its first hpd_track or hpd_track_smooth.  One memset on the stream, no
 * kernel launch. */
HPD_EXPORT int hpd_track_reset(const HpdTrackParams* p, void* state, size_t state_bytes, int clear_ids, void* stream);

/* Tracks n_frames >= 1 consecutive records (records + f * row_bytes, read in place) in one kernel launch, continuing
 * from the state and updating it.  track_ids [n_frames][max_people] int32: the id of each person, -1 for persons
 * that start no track and for slots >= n_person.  Every argument is checked before the launch. */
HPD_EXPORT int hpd_track(const HpdTrackParams* p, const uint8_t* records, int n_frames, void* state, size_t state_bytes,
                         int32_t* track_ids, void* stream);

/* ---- smoothing of tracked joints across frames (the 1-Euro filter: Casiez, Roussel, Vogel, CHI 2012) -------------
 * hpd_track_smooth tracks exactly as hpd_track (same ids; OKS uses the last raw pose) and also filters the COCO-section
 * coordinates of every tracked person's visible joints, x and y independently, with state per (track, joint) that
 * lives and dies with the track.  Frames are numbered consecutively across calls, fallback frames included.  For
 * person p < n_person of frame f with id >= 0 and joint k visible (poses[p][k][2] > 0), with the raw coordinate x:
 *   the first time joint k of the track is visible:  x^ = x, dx^ = 0, output x, last = f;
 *   otherwise, with g = f - last >= 1, each step one correctly rounded float64 operation (no FMA), in this order,
 *   TWO_PI = the float64 2 * pi, products and sums grouped left to right as written:
 *     te  = (double)g / fps
 *     rd  = (TWO_PI * d_cutoff) * te;  ad = rd / (rd + 1)
 *     dx  = (x - x^) / te
 *     dx^' = ad * dx + (1 - ad) * dx^
 *     c   = min_cutoff + beta * |dx^'|
 *     r   = (TWO_PI * c) * te;         a  = r / (r + 1)
 *     x^' = a * x + (1 - a) * x^
 *   output x^', store x^', dx^', last = f.
 * Invisible joints (their state untouched) and persons with id -1 (the empty-scene fallback's pseudo-person included)
 * are written raw; rows p >= n_person are 0.  A dropped track's filters are gone; a new track starts unseeded. */
typedef struct HpdSmoothParams {
  double min_cutoff;   /* Hz, in (0, 1e6] */
  double beta;         /* speed coefficient, in [0, 1e6] */
  double d_cutoff;     /* Hz, cutoff of the speed estimate, in (0, 1e6] */
  double fps;          /* the video's constant frame rate, in [1e-3, 1e6].  Not just > 0: with a subnormal fps,
                        * te = g / fps overflows to inf and rd / (rd + 1) is inf / inf = NaN.  With these bounds no
                        * step overflows for coordinates below 1e280 in magnitude. */
} HpdSmoothParams;

/* Bytes of a smoothing tracker state: the hpd_track state plus the filters of max_people * max_age tracks.  A state is
 * used with either hpd_track or hpd_track_smooth, never both; hpd_track_reset works on either kind. */
HPD_EXPORT int hpd_track_smooth_state_bytes(const HpdTrackParams* p, size_t* out_bytes);

/* hpd_track plus smoothing, in one kernel launch: track_ids as hpd_track's, coords [n_frames][max_people][num_kpts][2]
 * float64 (8-byte aligned).  Every argument is checked before the launch. */
HPD_EXPORT int hpd_track_smooth(const HpdTrackParams* p, const HpdSmoothParams* sp, const uint8_t* records,
                                int n_frames, void* state, size_t state_bytes, int32_t* track_ids, double* coords,
                                void* stream);

/* ---- drawing decoded poses into frames (skeletons and joints, for video overlays) -------------------------------
 * For frame f with record R (HpdRecordLayout for num_kpts, max_people, emb), optional ids[f][M] and optional
 * coords[f][M][K][2]:
 *  - Persons drawn: none when R's flags bit 0 is set (the empty-scene fallback's pseudo-person is not a person);
 *    otherwise p < clamp(n_person, 0, M), in ascending p.
 *  - Joint position: coords[f][p][k] when coords are given, else the COCO-section (x, y) of R (float64, raw-frame
 *    pixels).  Joint visible: (double)poses[p][k][2] > kpt_thr, and both coordinates finite with |x|, |y| <= 2^20
 *    (32 times the largest frame side: every product below stays finite).
 *  - Pixel (c, r) has its centre at X = c, Y = r: cv2.warpAffine's convention, which the input side reproduces, so
 *    the convention of the records' coordinates.
 *  - All float64, each step one correctly rounded operation, no FMA, grouped left to right as written.
 *    Joint disc of radius Rj at (jx, jy): covered iff (X-jx)*(X-jx) + (Y-jy)*(Y-jy) <= Rj*Rj.
 *    Limb (a, b), both joints visible, h = thickness / 2: ex = bx-ax, ey = by-ay, L2 = ex*ex + ey*ey, px = X-ax,
 *    py = Y-ay, t = px*ex + py*ey; then
 *      t <= 0  (a zero-length limb lands here):  covered iff px*px + py*py <= h*h;
 *      t >= L2:                                   covered iff (X-bx)*(X-bx) + (Y-by)*(Y-by) <= h*h;
 *      else, with cr = px*ey - py*ex:             covered iff cr*cr <= (h*h)*L2.
 *  - Paint order: per person p, its limbs in list order, then its joints 0..K-1.  A covered pixel takes the colour
 *    of the LAST primitive that covers it; uncovered pixels are copied from the input; row padding past 3w bytes of
 *    the output is not written.  No blending, no anti-aliasing.  thickness 0 draws no limbs, joint_radius 0 no joints.
 *  - Colours are three bytes in the frame's own channel order.  Without ids limb l takes limb_rgb[l]; with ids a
 *    person with id >= 0 takes track_rgb[id % num_track_colors] for all its limbs, one with id < 0 untracked_rgb.
 *    Joints always take joint_rgb. */
#define HPD_RENDER_MAX_LIMBS 64
#define HPD_RENDER_MAX_COLORS 32
typedef struct HpdRenderParams {
  int32_t num_kpts;       /* K <= HPD_MAX_KPTS */
  int32_t max_people;     /* M <= HPD_MAX_PEOPLE: persons per record */
  int32_t emb;            /* E of the records: 1 or 2 */
  int32_t num_limbs;      /* 0..HPD_RENDER_MAX_LIMBS */
  int32_t limbs[HPD_RENDER_MAX_LIMBS][2];       /* joint indices in [0, K), distinct within a limb */
  uint8_t limb_rgb[HPD_RENDER_MAX_LIMBS][3];
  uint8_t joint_rgb[3];
  uint8_t untracked_rgb[3];
  uint8_t reserved0_[2];
  int32_t num_track_colors;                     /* 1..HPD_RENDER_MAX_COLORS */
  int32_t reserved1_;
  uint8_t track_rgb[HPD_RENDER_MAX_COLORS][3];
  double thickness;       /* limb width in pixels, finite, in [0, 1024] */
  double joint_radius;    /* finite, in [0, 1024] */
  double kpt_thr;         /* finite */
} HpdRenderParams;

/* One frame: uint8 HWC, 3 channels, on the device.  out must not overlap any frame's input or another output. */
typedef struct HpdRenderFrame {
  const uint8_t* in;
  uint8_t* out;
  int64_t in_stride_row, out_stride_row;   /* bytes between rows, >= 3*w */
  int32_t h, w;                            /* 1..32767 */
} HpdRenderFrame;

/* Draws frames_host[f] (descriptors on the host) with the persons of records + f * row_bytes (read in place, 8-byte
 * aligned), track_ids [n_frames][max_people] int32 (NULL: no ids) and coords [n_frames][max_people][num_kpts][2]
 * float64 (NULL: the records' COCO section; 8-byte aligned).  Out of place only.  One launch per 32 frames; no
 * allocation, no workspace.  Every argument is checked before the first launch. */
HPD_EXPORT int hpd_render_poses(const HpdRenderParams* p, const HpdRenderFrame* frames_host, int n_frames,
                                const uint8_t* records, const int32_t* track_ids, const double* coords, void* stream);

/* Number of kernel launches the previous call on this thread enqueued (for bench accounting). */
HPD_EXPORT int hpd_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* HPDECODE_H_ */
