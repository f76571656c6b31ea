/* frcnn_b200 -- C ABI of the B200 (sm_100a) Faster R-CNN inference path.
 *
 * Drop-in boundary for endernewton/tf-faster-rcnn's `Network.test_image()` / `im_detect()` / `nms()`
 * hot path.  The reference's only native interface on this path is
 *     void _nms(int* keep_out, int* num_out, const float* boxes_host, int boxes_num,
 *               int boxes_dim, float nms_overlap_thresh, int device_id);      (lib/nms/gpu_nms.hpp:1-2)
 * reached through lib/nms/gpu_nms.pyx:16-31 and lib/model/nms_wrapper.py:15-23; everything else on the
 * path is TensorFlow graph ops called from Python (lib/nets/network.py).  This header therefore exports
 *   (1) frcnn_nms_host      -- argument-compatible superset of `_nms` (same order + `flags`),
 *   (2) one entry point per device stage of the TEST-mode graph, so the Python host code that mirrors
 *       lib/nets/{vgg16,resnet_v1,mobilenet_v1}.py can enqueue the graph on a CUDA stream (and capture it into a CUDA graph).
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative frcnn_status; the message of
 *     the last failure on the calling thread is read with frcnn_last_error().  Nothing is printed
 *     (the reference's CUDA_CHECK prints and continues, lib/nms/nms_kernel.cu:12-19).
 *   - pointers named *_dev are device pointers owned by the caller (PyTorch tensors' data_ptr());
 *     `stream` is a cudaStream_t passed as void*; all device entry points are asynchronous on it.
 *   - activations: NHWC fp32, dense.  conv weights: packed by frcnn_pack_conv_weights.
 *   - a handle/plan is single-stream and not re-entrant; one per GPU/rank.
 */
#ifndef FRCNN_B200_H_
#define FRCNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  FRCNN_OK = 0,
  FRCNN_ERR_CUDA = -1,         /* a CUDA runtime/driver call failed (text in frcnn_last_error) */
  FRCNN_ERR_ARG = -2,          /* invalid argument */
  FRCNN_ERR_NO_DEVICE = -3,    /* no usable sm_100 device */
  FRCNN_ERR_DRIVER_ENTRY = -4, /* cuTensorMapEncodeTiled not obtainable from the driver */
  FRCNN_ERR_CAPACITY = -5      /* problem larger than the compiled-in capacity */
} frcnn_status;

/* NMS predicate flags (SURVEY.md 8(a) row N). */
#define FRCNN_NMS_PLUS_ONE 1u        /* '+1' pixel areas (cpu_nms.pyx / nms_kernel.cu); else continuous (TF) */
#define FRCNN_NMS_INCLUSIVE 2u       /* suppress when ovr >= thr (cpu_nms.pyx:65); else ovr > thr */
#define FRCNN_NMS_SKIP_DEGENERATE 4u /* IoU := 0 when either area <= 0 (tf.image.non_max_suppression) */
#define FRCNN_NMS_MODE_CPU_NMS (FRCNN_NMS_PLUS_ONE | FRCNN_NMS_INCLUSIVE)
#define FRCNN_NMS_MODE_GPU_NMS (FRCNN_NMS_PLUS_ONE)
#define FRCNN_NMS_MODE_TF (FRCNN_NMS_SKIP_DEGENERATE)

/* activation applied by conv/depthwise epilogues */
#define FRCNN_ACT_NONE 0
#define FRCNN_ACT_RELU 1
#define FRCNN_ACT_RELU6 2

int frcnn_version(void);
/* copies the calling thread's last error text into buf (NUL terminated); returns its length */
int frcnn_last_error(char* buf, size_t buflen);
/* 0 when device `device_id` exists and is compute capability 10.x */
int frcnn_check_device(int device_id);
/* cudaMemsetAsync(dev_ptr, 0, bytes) on `stream`: lets a host layer clear buffers (detection records) without a framework fill kernel */
int frcnn_zero_async(void* dev_ptr, size_t bytes, void* stream);

/* CUDA-graph capture of a sequence of the stage calls below (one image or batch = one replay): begin on a NON-default stream,
 * enqueue the stages on that stream, end -> an executable graph; launch it on any stream.  No allocation or synchronisation
 * happens inside the stages, so the whole TEST-mode path is capturable. */
typedef struct frcnn_graph frcnn_graph;
int frcnn_graph_begin(void* stream);
int frcnn_graph_end(void* stream, frcnn_graph** out);
int frcnn_graph_launch(const frcnn_graph* g, void* stream);
void frcnn_graph_destroy(frcnn_graph* g);

/* ---- (1) NMS, host buffers: replaces `_nms` (lib/nms/gpu_nms.hpp:1-2, nms_kernel.cu:91-144) ----------
 * boxes_host: [boxes_num, boxes_dim>=4] rows (x1,y1,x2,y2,...), ALREADY sorted by descending score, as the
 * reference's Cython wrapper guarantees (gpu_nms.pyx:25-28).  keep_out: capacity boxes_num; receives
 * indices into the sorted input in ascending order.  Synchronous.  device_id < 0 selects the calling thread's current
 * device; the caller's current device is restored before returning (the reference's _nms leaves it switched). */
int frcnn_nms_host(int* keep_out, int* num_out, const float* boxes_host, int boxes_num, int boxes_dim,
                   float nms_overlap_thresh, int device_id, unsigned flags);

/* Same greedy NMS, device buffers, no sort: boxes_dev [n,4] in priority order.  keep_dev: capacity
 * max_out (int32 indices into boxes_dev), num_dev: int32 count.  Early exit at max_out kept. */
int frcnn_nms_sorted_dev(const float* boxes_dev, int n, float thresh, unsigned flags, int max_out,
                         int* keep_dev, int* num_dev, void* stream);

/* ---- (2) dense stages: conv / FC as implicit GEMM on tcgen05 (FP16x3 operand split, fp32 accumulate in TMEM) -
 * Replaces slim.conv2d / slim.fully_connected (+ folded bias or BatchNorm scale/shift, ReLU/ReLU6,
 * residual add) as used by lib/nets/{vgg16,resnet_v1,mobilenet_v1}.py and network.py:323-378.
 *   out[n,ho,wo,co] = act( (sum_{r,s,ci} in[n, ho*stride+r-pad_t, wo*stride+s-pad_l, ci] * w[co,r,s,ci])
 *                          * scale[co] + shift[co] (+ residual[n,ho,wo,co]) )
 * Requirements: cin % 32 == 0.  w_hi/w_lo from frcnn_pack_conv_weights.  scale may be NULL (=1). */
typedef struct frcnn_conv_plan frcnn_conv_plan;
#define FRCNN_CONV_F16X3 0   /* fp16 hi/lo split of both operands, 3 x tcgen05.mma.kind::f16, fp32 accumulate.  Activation range:
                              * fp32-grade for |x| < 65520; an activation of larger magnitude (like an Inf or NaN) makes every
                              * output whose window reads it Inf or NaN, and leaves all other outputs unaffected. */
#define FRCNN_CONV_TF32X3 1  /* tf32 hi/lo split, 3 x kind::tf32 (same 22-bit products, twice the tensor time) */
#define FRCNN_CONV_F16X1 2   /* THROUGHPUT mode, not fp32-grade: plain fp16 operands (the hi planes only), 1 MMA per product, fp32
                              * accumulate; ~3e-4 of the output range per layer instead of ~4e-7.  Same packed weights as F16X3. */

typedef struct {
  const float* in_dev;       /* [n, h, w, cin] */
  const void* w_hi_dev;      /* [cout, kh*kw*cin] hi plane from frcnn_pack_conv_weights (fp16) / _tf32 (fp32) */
  const void* w_lo_dev;      /* [cout, kh*kw*cin] lo plane (residual of the hi rounding) */
  const float* scale_dev;    /* [cout] or NULL */
  const float* shift_dev;    /* [cout] or NULL */
  const float* residual_dev; /* [n, ho, wo, cout] or NULL */
  float* out_dev;            /* [n, ho, wo, cout] */
  int n, h, w, cin;
  int cout, kh, kw, stride;
  int pad_t, pad_l;          /* zero padding before the first row / column */
  int ho, wo;
  int act;                   /* FRCNN_ACT_* */
  int block_n;               /* 0 = choose; else 64/128 */
  int kb_per_chunk;          /* 0 = default (8): 32-wide k-blocks summed in TMEM before promotion to registers */
  int split_k;               /* 0 = choose; 1 = never; n = split the K loop over n CTAs + deterministic reduce pass */
  int impl;                  /* FRCNN_CONV_F16X3 (0, default) | FRCNN_CONV_TF32X3 (r01 kernel, kept for A/B measurements) | FRCNN_CONV_F16X1 */
  float out_mult;            /* F16X3: 2^-wexp of frcnn_pack_conv_weights (0 is read as 1) */
} frcnn_conv_desc;

int frcnn_conv_plan_create(frcnn_conv_plan** out, const frcnn_conv_desc* d);
int frcnn_conv_plan_run(const frcnn_conv_plan* p, void* stream);
/* Host-only (no CUDA call): the work decomposition frcnn_conv_plan_create would choose on a GPU with sm_count SMs.  Device
 * pointers in *d are ignored.  out16 = {block_n, tile_n, tile_h, tile_w, m_tiles, n_tiles, tiles, split_tiles, splits,
 * k_blocks_per_split, work_units, grid, k_blocks, k_blocks_per_chunk, tiles_h, tiles_w}. */
int frcnn_conv_plan_geometry(const frcnn_conv_desc* d, int sm_count, int* out16);
int frcnn_conv_plan_info(const frcnn_conv_plan* p, int* block_n, int* tile_n, int* tile_h, int* tile_w,
                         int* grid_m, int* grid_n, int* splits, int* smem_bytes);
/* debug aid: trace_dev (int64[64*8], device) receives clock64() stamps of the pipeline hand-offs of CTA (0,0)
 * for its first 64 k-blocks: [kb][0]=producer saw slot free, [1]=TMA issued, [2]=splitter saw data, [6]=split done,
 * [3]=splitter arrived, [4]=MMA saw operands, [5]=MMAs issued+committed, [chunk][7]=epilogue saw TMEM chunk. NULL disables. */
int frcnn_conv_plan_set_trace(frcnn_conv_plan* p, long long* trace_dev);
void frcnn_conv_plan_destroy(frcnn_conv_plan* p);
/* development aid: in the watchdog build (libfrcnn_b200_wd.so, -DFRCNN_WATCHDOG) a barrier wait of the dense kernel that
 * lasts > ~0.2 s aborts the kernel instead of hanging the GPU; out16 = {aborted, waits_timed_out, block, thread, wait_tag,
 * parity, aux, ...}.  In the normal build out16[15] = 0xffffffff and the rest is zero. */
int frcnn_debug_watchdog(unsigned int* out16, int reset);

/* HWIO [kh,kw,cin,cout] (TF layout) -> K-major [cout][kh][kw][cin] fp16 planes:
 *   hi = RN_f16(w * 2^wexp), lo = RN_f16((w * 2^wexp - hi) * 2^11).  The caller picks wexp so that max|w| * 2^wexp lies in
 * [2^13, 2^14) and passes out_mult = 2^-wexp in the conv descriptor. */
int frcnn_pack_conv_weights(const float* w_hwio_dev, void* w_hi_dev, void* w_lo_dev, int kh, int kw,
                            int cin, int cout, int wexp, void* stream);
/* same layout, fp32 planes of tf32-rounded values (hi = RN_tf32(w), lo = RN_tf32(w - hi)) for FRCNN_CONV_TF32X3 */
int frcnn_pack_conv_weights_tf32(const float* w_hwio_dev, float* w_hi_dev, float* w_lo_dev, int kh, int kw,
                                 int cin, int cout, void* stream);

/* ---- (3) bandwidth stages (SIMT, fp32, no FMA contraction where the oracle has separate roundings) ---- */
/* first-layer convolution for cin==3 (vgg conv1_1, resnet conv1 7x7/2, mobilenet Conv2d_0 3x3/2):
 * direct fp32 FFMA conv, w HWIO [k,k,3,cout], y = act(conv*scale + shift) */
int frcnn_conv_first(const float* in_dev, const float* w_hwio_dev, const float* scale_dev,
                     const float* shift_dev, float* out_dev, int n, int h, int w, int cout, int k,
                     int stride, int pad_t, int pad_l, int ho, int wo, int act, void* stream);
/* depthwise 3x3 (slim.separable_conv2d with num_outputs=None, mobilenet_v1.py:21-49):
 * w [3,3,c] ; y = act(dw*scale + shift) */
int frcnn_depthwise3x3(const float* in_dev, const float* w_dev, const float* scale_dev,
                       const float* shift_dev, float* out_dev, int n, int h, int w, int c, int stride,
                       int pad_t, int pad_l, int ho, int wo, int act, void* stream);
/* max pool k x k / stride; padded cells are skipped when pad_is_neg_inf != 0 (TF 'SAME'),
 * or count as zeros (tf.pad + 'VALID', resnet_v1.py:83-84) */
int frcnn_max_pool(const float* in_dev, float* out_dev, int n, int h, int w, int c, int k, int stride,
                   int pad_t, int pad_l, int ho, int wo, int pad_is_neg_inf, void* stream);
/* mean over the spatial positions: [r, hw, c] -> [r, c]  (tf.reduce_mean axis=[1,2]) */
int frcnn_spatial_mean(const float* in_dev, float* out_dev, int r, int hw, int c, void* stream);

/* image -> network blob on the device (lib/model/test.py:26-58 for one scale): blob[y,x,c] = bilinear resize, with OpenCV's
 * INTER_LINEAR float arithmetic, of (float32(img) - means) ; img_dev uint8 BGR [h0,w0,3]; blob_dev fp32 [H,W,3] with
 * H = cvRound(h0*fy), W = cvRound(w0*fx) computed by the caller.  means3 is a HOST pointer. */
int frcnn_preprocess(const unsigned char* img_dev, int h0, int w0, const double* means3, double fx, double fy,
                     float* blob_dev, int H, int W, void* stream);

/* ---- (4) proposal / detection stages.  Every stage takes `batch` images of one blob shape (the reference is batch 1,
 * lib/nets/network.py:388; batch > 1 is the throughput extension of SURVEY.md 8(f) rank 4): per-image arrays are
 * concatenated image-major, RoI rows carry their image index in column 0 exactly like crop_and_resize's box_ind. ---- */

/* RPN: 2-way softmax (fg prob), anchor generation, bbox_transform_inv, clip -- proposal_layer.py:62-69.
 * rpn_out_dev: [batch*hw, ld] rows with the 2A class logits at column 0 and the 4A deltas at column delta_col
 * (delta_col % 4 == 0, ld % 4 == 0: the fused 1x1 RPN head writes both).
 * base_anchors_dev [A,4].  scores_dev [batch*hw*A], props_dev [batch*hw*A,4] in (image,h,w,a) order. */
int frcnn_rpn_decode(const float* rpn_out_dev, int ld, int delta_col, const float* base_anchors_dev, int num_anchors,
                     int batch, int fh, int fw, int feat_stride, float im_h, float im_w, float* scores_dev,
                     float* props_dev, void* stream);
/* stable descending sort of `batch` segments of n fp32 keys each (ties: lower index first) -> order_dev int32[batch*n],
 * indices LOCAL to the segment; one thread-block cluster per segment, n <= 90 112.  The workspace arguments are kept
 * from the r01 (CUB based) signature and may be NULL / 0. */
size_t frcnn_sort_workspace_bytes(int n);
int frcnn_sort_desc(const float* keys_dev, int n, int batch, int* order_dev, float* sorted_keys_dev, void* workspace_dev,
                    size_t workspace_bytes, void* stream);
/* proposal selection (proposal_layer_tf / proposal_layer / proposal_top_layer), per image: walk `order`, greedy NMS
 * with `flags` over the first `pre_nms_top_n` (<=0: all) candidates, stop at post_nms_top_n.  thresh < 0
 * means no NMS (TEST.MODE='top').  props/scores/order: [batch][n].  rois_dev [batch*post_nms_top_n,5] =
 * (image,x1,y1,x2,y2), zero padded per image; roi_scores_dev [batch*post_nms_top_n]; keep_dev int32 segment-local
 * indices into props; num_dev int32[batch] counts. */
int frcnn_proposals(const float* props_dev, const float* scores_dev, const int* order_dev, int n, int batch,
                    int pre_nms_top_n, int post_nms_top_n, float thresh, unsigned flags, float* rois_dev,
                    float* roi_scores_dev, int* keep_dev, int* num_dev, void* stream);
/* tf.image.crop_and_resize on the stride-16 feature map + optional 2x2 max pool (network.py:141-157,
 * resnet_v1.py:55-76).  feat_dev [batch,fh,fw,c]; rois_dev [r,5] = (image index, blob-scale pixels).  pooled = 7;
 * pre_pool 0: direct 7x7, 1: 14x14 then 2x2/2 max.  out [r,7,7,c] */
int frcnn_crop_pool(const float* feat_dev, int batch, int fh, int fw, int c, const float* rois_dev, int r, int pooled,
                    int pre_pool, float* out_dev, void* stream);
/* split the fused [r, ld] head GEMM output (cls logits at col 0, 4C deltas at col C):
 * cls_score [r,C], cls_prob = softmax, bbox_pred = delta*stds + means (network.py:361-378,428-432) */
int frcnn_cls_finish(const float* head_out_dev, int ld, int r, int num_classes, const float* stds4,
                     const float* means4, float* cls_score_dev, float* cls_prob_dev, float* bbox_pred_dev,
                     void* stream);
/* im_detect tail: boxes = rois[:,1:5]/scale; bbox_transform_inv; one-sided clip to the ORIGINAL image
 * (lib/model/test.py:95-102,67-77).  im_meta_dev [batch,3] fp32 = (im_scale, orig_h, orig_w) per image, read on the
 * device (the launch is CUDA-graph capturable: the host only rewrites the 12 bytes).  pred_boxes_dev [r,4C] */
int frcnn_bbox_decode(const float* rois_dev, const float* bbox_pred_dev, int r, int num_classes, int batch,
                      const float* im_meta_dev, float* pred_boxes_dev, void* stream);
/* test_net tail (lib/model/test.py:162-180), per image: per class j>=1: score > thresh, NMS(flags, nms_thresh), then the
 * max_per_image cap over all classes.  r = RoI rows per image (<= 8192; above 1024 -- TEST.MODE='top' with
 * RPN_TOP_N=5000 -- the kept sets live in `workspace_dev`, frcnn_detect_post_workspace_bytes(r, C, batch) bytes, else the
 * workspace may be NULL).  num_rois_dev: int32[batch] valid-row counts.  det_dev [batch,max_det,6] =
 * (x1,y1,x2,y2,score,class) sorted by (class, descending score); ndet_dev int32[batch] = the number of detections of
 * the image, which EXCEEDS max_det when the records did not fit (the caller must treat that as an error).
 * record_stride (4-byte words; 0 = dense): distance between consecutive images in BOTH det_dev and ndet_dev, so that a
 * caller can interleave count and rows into one fixed-size record per image (the multi-GPU all-gather payload).
 * keep_dev [batch,C,r] int32 roi indices per class (after the cap), keep_cnt_dev [batch,C]; keep_score_dev [batch,C,r]. */
size_t frcnn_detect_post_workspace_bytes(int r, int num_classes, int batch);
int frcnn_detect_post(const float* cls_prob_dev, const float* pred_boxes_dev, const int* num_rois_dev, int r, int batch,
                      int num_classes, float score_thresh, float nms_thresh, unsigned flags,
                      int max_per_image, int max_det, float* det_dev, int* ndet_dev, int record_stride, int* keep_dev,
                      int* keep_cnt_dev, float* keep_score_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRCNN_B200_H_ */
