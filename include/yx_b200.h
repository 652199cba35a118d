/*
 * yx_b200.h — C-ABI of the B200-native (sm_100a) YOLOX detection hot path.
 *
 * Every entry point is `extern "C"`, takes plain device pointers + sizes + a
 * `cudaStream_t` passed as `void*`, returns 0 on success or a negative
 * `yx_status` code, never throws and never synchronises the host (all work is
 * enqueued on `stream`, so the calls are CUDA-graph capturable).  There are no
 * torch types in any signature; PyTorch only owns the memory the pointers refer
 * to.  All activations are NHWC ("channels-last"), 16-bit (bf16/fp16) on the
 * tensor-core path or fp32 on the verification path; channel counts and channel
 * offsets are multiples of 8 elements so that every pixel row is 16-byte aligned.
 *
 * The reference (yhenon/pixeltable-yolox, a pure-PyTorch library) has no FFI of
 * its own; each entry point below names the reference function (file:line under
 * /root/reference) whose arithmetic it replaces.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 */
#ifndef YX_B200_H_
#define YX_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YX_VERSION 100 /* 0.1.0 */

typedef enum yx_status {
  YX_OK = 0,
  YX_ERR_INVALID_ARG = -1,   /* bad shape / alignment / null pointer              */
  YX_ERR_UNSUPPORTED = -2,   /* shape outside what the sm_100a kernels implement  */
  YX_ERR_CUDA = -3,          /* a CUDA runtime/driver call failed (see yx_last_error) */
  YX_ERR_NO_DEVICE = -4,     /* no sm_100 device visible: there is NO CPU fallback */
  YX_ERR_CAPACITY = -5       /* a caller-provided workspace/output is too small   */
} yx_status;

typedef enum yx_dtype { YX_BF16 = 0, YX_FP16 = 1, YX_FP32 = 2, YX_U8 = 3 } yx_dtype;
typedef enum yx_act { YX_ACT_NONE = 0, YX_ACT_SILU = 1, YX_ACT_RELU = 2, YX_ACT_LRELU = 3 } yx_act;

/* Epilogue of the implicit-GEMM conv. */
typedef enum yx_epilogue {
  YX_EPI_STORE = 0, /* y = act(acc + bias) (+ residual) -> NHWC activation, dtype of the input */
  YX_EPI_HEAD = 1   /* YOLOX head: acc+bias -> [B, A, 5+nc] fp32 with decode/sigmoid fused
                       (yolox/models/yolo_head.py:185-187,205-207,233-251)                     */
} yx_epilogue;

const char* yx_strerror(int code);
/* Last error message of the calling thread (CUDA error string, failed check ...). */
const char* yx_last_error(void);
int yx_version(void);
/* 0 when device `dev` is an sm_100 part and the kernels can run, else YX_ERR_NO_DEVICE. */
int yx_device_check(int dev);

/* ------------------------------------------------------------------------------------------
 * Dense conv + folded BN + activation as one implicit GEMM
 *   replaces BaseConv.forward  (yolox/models/network_blocks.py:27-52, act(bn(conv(x))))
 *   and the biased 1x1 prediction convs of YoloxHead (yolox/models/yolo_head.py:94-120).
 *   BN folding follows fuse_conv_and_bn (yolox/utils/model_utils.py:33-75).
 *
 * GEMM view: M = batch*out_h*out_w pixels, N = out_c, K = ksize*ksize*in_c.
 *   in  : NHWC, `in_c` channels read starting at `in` with a per-pixel stride of `in_ld`
 *         elements (so a channel slice of a wider concat buffer is a valid input);
 *   w   : [out_c][ksize*ksize][in_c] (K-major), BN scale folded in, same dtype as `in`;
 *   bias: [out_c] fp32 (folded BN shift, or the pred-conv bias);
 *   out : NHWC slice, per-pixel stride `out_ld`; `res` (optional) is added AFTER the
 *         activation (Bottleneck shortcut, network_blocks.py:95-99);
 *   ups : optional second destination that receives the result replicated 2x2
 *         (nn.Upsample(scale_factor=2, "nearest") fused into the producer:
 *         yolox/models/yolo_pafpn.py:97-99,102-104); its spatial size is 2*out_h x 2*out_w.
 * Constraints: ksize in {1,3}; stride in {1,2}; pad = (ksize-1)/2; in_c % 16 == 0;
 *   out_c % 16 == 0; all *_ld % 8 == 0; pointers 16-byte aligned.
 * ------------------------------------------------------------------------------------------ */
typedef struct yx_conv_desc {
  int32_t batch, in_h, in_w, in_c;
  int32_t out_h, out_w, out_c;
  int32_t ksize, stride;
  int32_t dtype;    /* yx_dtype of in/w/out/res: YX_BF16 | YX_FP16 (tcgen05) | YX_FP32 (SIMT) */
  int32_t act;      /* yx_act */
  int32_t epilogue; /* yx_epilogue */
  const void* in;   int64_t in_ld;
  const void* w;
  const float* bias;
  void* out;        int64_t out_ld;
  const void* res;  int64_t res_ld;
  void* ups;        int64_t ups_ld;
  /* YX_EPI_HEAD only: out_c (>= 5+nc, padded) accumulators per pixel are written as fp32 rows
   * head_out[(b*head_anchors + head_anchor_off + y*out_w + x)*(5+head_nc) + c], c < 5+nc.
   * head_decode is a bit set:  bit0 = box decode: c<2 -> (v + grid)*head_stride,
   * c in {2,3} -> exp(v)*head_stride;  bit1 = sigmoid on c >= 4 (obj, cls).
   *   3 = eval with decode_in_inference (yolo_head.py:185-187, 233-251)
   *   2 = eval with decode_in_inference=False (yolo_head.py:208-211)
   *   1 = training branch: decoded boxes, raw logits (yolo_head.py:161-166, 213-231)
   *   0 = raw prediction-conv outputs */
  float* head_out;
  int32_t head_anchors, head_anchor_off, head_nc, head_decode;
  float head_stride;
  /* optional second destination (YX_EPI_STORE): output channels >= out2_begin (a multiple of 16) are written
   * to out2[pixel*out2_ld + (c - out2_begin)] instead of `out`; lets one stacked GEMM (CspLayer conv1 | conv2,
   * network_blocks.py:176-177) feed two dense buffers. out2 == NULL disables it. */
  int32_t out2_begin;
  void* out2;       int64_t out2_ld;
  /* YX_EPI_HEAD with head_decode == 3 on the tcgen05 path: stage 1 of yx_postprocess fused into the epilogue
   * (the thread that decodes an anchor row still holds it in registers). When head_cand != NULL every anchor with
   * score >= head_conf_thre writes its candidate row head_cand[(b*head_anchors + a)*8] =
   * (x1,y1,x2,y2,obj,class_conf,class,score) (rows of the other anchors are left untouched: stage 2 never reads
   * them) and appends its 64-bit sort key to head_keys[b*head_anchors + ...] (count in
   * head_counts[b], which the caller zeroes first: yx_postprocess_begin) -- exactly what filter_kernel computes from
   * the fp32 rows (boxes.py:32-50), so yx_nms_prefiltered can follow without re-reading the prediction tensor.
   * head_xyxy != 0 additionally stores corners instead of (cx,cy,w,h) in head_out, the in-place conversion of
   * boxes.py:32-37. The three pointers come from yx_postprocess_workspace_ptrs. */
  float* head_cand;
  uint64_t* head_keys;
  int32_t* head_counts;
  float head_conf_thre;
  int32_t head_xyxy;
  /* YX_EPI_STORE on the tcgen05 path, depth-to-space store (0 = off): out_c == 4 * shuffle2_c, `out` is an NHWC buffer of
   * spatial size 2*out_h x 2*out_w, and channel c of output pixel (b, y, x) is written to pixel (b, 2y + (q >> 1), 2x + (q & 1)),
   * channel c - q * shuffle2_c, q = c / shuffle2_c. With the sub-pixel weights of yx_pack_train_weights(subpixel = 1) this
   * makes the dgrad of a 3x3 stride-2 conv ONE stride-1 conv over dy. No res / ups / out2. */
  int32_t shuffle2_c;
} yx_conv_desc;

/* tcgen05/TMEM/TMA implicit GEMM for bf16/fp16; routes YX_FP32 to the SIMT kernel. */
int yx_conv_bn_act_fwd(const yx_conv_desc* d, void* stream);
/* Runs the launch selection of yx_conv_bn_act_fwd for `d` without launching (needs a device: it encodes the tensor
 * maps). Fills up to `capacity` ints and returns the count, or a negative yx_status:
 *   mode (0 per-tap ring, 1 halo, 2 stride-2 planes), flat, b_resident, G, ctas_per_sm, epi_groups, acc_stages, a_slots,
 *   stages, BN, n_tiles, m_tiles, num_tiles, grid, tw, th.
 * CTA i of the halo / planes modes owns the units [num_tiles*i/grid, num_tiles*(i+1)/grid); the per-tap ring hands
 * tile t to CTA t % grid. */
int yx_conv_schedule(const yx_conv_desc* d, int32_t* info, int32_t capacity);
/* ------------------------------------------------------------------------------------------
 * Fused Bottleneck: y = [x +] act(bn2(conv3x3(act(bn1(conv1x1(x))))))  in one kernel
 *   replaces Bottleneck.forward (yolox/models/network_blocks.py:77-99: conv1 1x1, conv2 3x3,
 *   `y + x` when use_add) with hidden == in == out channels (CspLayer passes expansion = 1.0,
 *   network_blocks.py:169-172). The hidden tensor stays in shared memory / TMEM.
 *   x   : NHWC slice, c channels, per-pixel stride x_ld;  out: NHWC slice (out_ld), MUST NOT alias x
 *   w1  : [c][1][c], w2: [c][9][c] packed like yx_conv_desc.w (BN folded); bias1/bias2 fp32 [c]
 * Constraints: c in {16, 32, 64, 128}; dtype bf16/fp16; x_ld, out_ld multiples of 16; x/out 32-byte aligned.
 * ------------------------------------------------------------------------------------------ */
typedef struct yx_bneck_desc {
  int32_t batch, h, w, c;
  int32_t dtype;    /* YX_BF16 | YX_FP16 */
  int32_t act;      /* yx_act of both convs */
  int32_t use_add;  /* 1: shortcut (network_blocks.py:97-98) */
  const void* x;    int64_t x_ld;
  const void* w1;   const float* bias1;
  const void* w2;   const float* bias2;
  void* out;        int64_t out_ld;
} yx_bneck_desc;
int yx_bottleneck_fwd(const yx_bneck_desc* d, void* stream);
/* 1 when yx_bottleneck_fwd supports this shape (callers fall back to two yx_conv_bn_act_fwd). */
int yx_bottleneck_supported(const yx_bneck_desc* d);

/* CUDA-core (FFMA, fp32 accumulate in K order) implementation of the same contract for every
 * dtype: the fp32 verification mode and the on-device cross-check of the tensor-core kernel. */
int yx_conv_bn_act_fwd_simt(const yx_conv_desc* d, void* stream);

/* Depthwise 3x3 conv + folded BN + act (DWConv.dconv, network_blocks.py:55-67), NHWC.
 *   w: [9][c] (tap-major) in `dtype`, bias [c] fp32. stride in {1,2}, pad 1. */
int yx_dwconv3x3_bn_act_fwd(const void* in, int64_t in_ld, const void* w, const float* bias,
                            void* out, int64_t out_ld, int32_t batch, int32_t in_h, int32_t in_w,
                            int32_t c, int32_t stride, int32_t act, int32_t dtype, void* stream);

/* SPP max pools (SPPBottleneck, network_blocks.py:120-142): reads c channels at `buf`
 * (pixel stride ld) and writes maxpool5/9/13 (stride 1, -inf padding) to channel offsets
 * c, 2c, 3c of the same buffer, i.e. completes cat[x, m5(x), m9(x), m13(x)] in place. */
int yx_spp_maxpool(void* buf, int64_t ld, int32_t batch, int32_t h, int32_t w, int32_t c,
                   int32_t dtype, void* stream);

/* Focus space-to-depth (network_blocks.py:193-208): NCHW image [B,3,H,W] (fp32 or uint8,
 * raw 0..255) -> NHWC [B,H/2,W/2,out_ld] with channels (TL,BL,TR,BR) x (c0,c1,c2) = 12 real
 * channels, the rest zero. */
int yx_focus_s2d(const void* img, int32_t img_dtype, void* out, int64_t out_ld, int32_t out_dtype,
                 int32_t batch, int32_t h, int32_t w, void* stream);

/* Fused Focus + stem conv + folded BN + act on the tensor cores (network_blocks.py:186-208 + 27-52):
 * reads the raw NCHW image (fp32 or uint8) once and writes the NHWC 16-bit stem output once.
 * The 3x3 conv runs on the space-to-depth grid, one K = 16 GEMM step per filter tap:
 *   w    : [out_c][9][16] in `dtype`: tap = 3*r + s, k = 2*(2*c + py) + px for image channel c and pixel parity
 *          (py, px) = Wfocus[o, 3*(2*px+py)+c, r, s] * bn_scale (Focus order TL, BL, TR, BR), k = 12..15 zero.
 *          For dtype fp16 the kernel feeds pixels as x/256: pack 256 * W.
 *   bias : [out_c] fp32; out: [B, h/2, w/2, out_ld] NHWC.  out_c % 16 == 0, out_c <= 128. */
int yx_focus_conv_bn_act_fwd(const void* img, int32_t img_dtype, const void* w, const float* bias,
                             void* out, int64_t out_ld, int32_t batch, int32_t h, int32_t wd,
                             int32_t out_c, int32_t act, int32_t dtype, void* stream);

/* Fold BN into a conv and repack it for yx_conv_bn_act_fwd (model_utils.py:33-75):
 *   src    : [o][i][kh][kw] fp32 (nn.Conv2d.weight); gamma/beta/mean/var [o] fp32 or NULL
 *            (plain conv); conv_bias [o] fp32 or NULL;
 *   dst_w  : packed [dst_o_total][kh*kw][dst_i_total]; rows o land at dst_o_off + o, columns i
 *            at dst_i_off + i (everything else is left untouched: zero the buffer first);
 *   dst_b  : fp32 [dst_o_total], written at dst_o_off + o.
 * depthwise != 0 packs [c][1][3][3] -> [9][dst_i_total] (tap-major) instead. */
int yx_pack_weights(const float* src, const float* gamma, const float* beta, const float* mean,
                    const float* var, const float* conv_bias, float eps, int32_t o, int32_t i,
                    int32_t kh, int32_t kw, void* dst_w, int32_t dst_dtype, int32_t dst_o_off,
                    int32_t dst_i_off, int32_t dst_i_total, float* dst_b, int32_t depthwise,
                    void* stream);

/* Standalone decode of an undecoded [B, A, 5+nc] fp32 tensor in place
 * (YoloxHead.decode_outputs, yolo_head.py:233-251). hw: 2*n_levels ints (h,w per level). */
int yx_head_decode(float* pred, int32_t batch, int32_t anchors, int32_t nc, const int32_t* hw,
                   const int32_t* strides, int32_t n_levels, void* stream);

/* ------------------------------------------------------------------------------------------
 * postprocess: score filter + class-aware NMS  (yolox/utils/boxes.py:31-75 and the
 * third-party torchvision.ops.batched_nms it calls, boxes.py:62-67).
 *   pred      : [B, A, 5+nc] fp32 (cx,cy,w,h,obj,cls...). When `inplace_xyxy` != 0 the first
 *               four columns are overwritten with (x1,y1,x2,y2) exactly like boxes.py:32-37.
 *   dets      : [B, max_det, 7] fp32 rows (x1,y1,x2,y2,obj,class_conf,class_pred) in
 *               descending-score order; det_idx [B, max_det] int64 anchor index of each kept
 *               row; det_count [B] int32.
 *   nms_variant: 0 = coordinate-offset trick (torchvision CUDA path for <= 100k coordinates),
 *               1 = per-class ("vanilla", torchvision CPU path above 4000 coordinates),
 *               2 = class-agnostic (boxes.py:55-60),
 *               3 / 4 = what torchvision itself picks per image on CUDA / on CPU:
 *               the offset trick unless 4*n_candidates > 100000 (CUDA, torchvision >= 0.19; 0.26 is installed and
 *               generated the goldens) / 4000 (CPU), else per-class.
 *               5 = the CUDA rule of torchvision 0.17.2, the version the reference pins (poetry.lock:2084-2085):
 *               per-class above 20000 coordinates.
 *   workspace : yx_postprocess_workspace_bytes(B, A) bytes of device scratch.
 * ------------------------------------------------------------------------------------------ */
int64_t yx_postprocess_workspace_bytes(int32_t batch, int32_t anchors);
int yx_postprocess(float* pred, int32_t batch, int32_t anchors, int32_t nc, float conf_thre,
                   double nms_thre, int32_t nms_variant, int32_t inplace_xyxy, float* dets,
                   int64_t* det_idx, int32_t* det_count, int32_t max_det, void* workspace,
                   int64_t workspace_bytes, void* stream);

/* yx_postprocess with stage 1 (score filter) already done by the head epilogues (yx_conv_desc.head_cand):
 *   yx_postprocess_workspace_ptrs : where the candidate rows / sort keys / per-image counters live inside a
 *                                   workspace of yx_postprocess_workspace_bytes(batch, anchors) bytes
 *   yx_postprocess_begin          : zeroes the per-image candidate counters (before the head GEMMs run)
 *   yx_nms_prefiltered            : stage 2 (sort + class-aware NMS + detection rows), same outputs as yx_postprocess */
int yx_postprocess_workspace_ptrs(void* workspace, int32_t batch, int32_t anchors, float** cand, uint64_t** keys,
                                  int32_t** counts);
int yx_postprocess_begin(void* workspace, int32_t batch, int32_t anchors, void* stream);
int yx_nms_prefiltered(int32_t batch, int32_t anchors, double nms_thre, int32_t nms_variant, float* dets,
                       int64_t* det_idx, int32_t* det_count, int32_t max_det, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* The two stages of yx_postprocess on their own (parity tests, SURVEY 8b export list); both use
 * a workspace of yx_postprocess_workspace_bytes(batch, anchors | n_max) bytes.
 * conf_thre is compared in fp32 (torch casts the Python scalar to the tensor dtype, boxes.py:48);
 * nms_thre is a double because torchvision's CPU kernel compares the fp32 IoU with a double.
 * yx_score_filter_compact: candidates in ascending anchor order: cand [B, A, 8] fp32 rows
 *   (x1,y1,x2,y2,obj,class_conf,class_pred,score), cand_idx [B, A] int32, cand_count [B].
 * yx_batched_nms: boxes [B, n_max, 4] xyxy, scores [B, n_max], cls [B, n_max] (int32),
 *   counts [B]; keep [B, n_max] int32 indices (into the per-image candidate list) in
 *   descending score order, keep_count [B]. */
int yx_score_filter_compact(const float* pred, int32_t batch, int32_t anchors, int32_t nc,
                            float conf_thre, float* cand, int32_t* cand_idx, int32_t* cand_count,
                            void* workspace, int64_t workspace_bytes, void* stream);
int yx_batched_nms(const float* boxes, const float* scores, const int32_t* cls,
                   const int32_t* counts, int32_t batch, int32_t n_max, double nms_thre,
                   int32_t nms_variant, int32_t* keep, int32_t* keep_count, void* workspace,
                   int64_t workspace_bytes, void* stream);

/* Pairwise IoU (yolox/utils/boxes.py:78-101): a [n,4], b [m,4] fp32 -> out [n,m]. */
int yx_bboxes_iou(const float* a, int32_t n, const float* b, int32_t m, int32_t xyxy, float* out,
                  void* stream);

/* ------------------------------------------------------------------------------------------
 * SimOTA label assignment (YoloxHead.get_assignments / get_geometry_constraint /
 * simota_matching, yolox/models/yolo_head.py:420-574), batched over images, no host sync.
 *   pred   : [B, A, 5+nc] fp32 training-branch head output (decoded boxes, raw obj/cls logits)
 *   labels : [B, max_gt, 5] fp32 rows (cls, cx, cy, w, h), zero padded (data_augment.py:200-208)
 *   anchor grid: x_shift[A], y_shift[A], stride[A] fp32 (yolo_head.py:213-231)
 * outputs (dense over anchors):
 *   fg_mask [B, A] uint8, matched_gt [B, A] int32 (-1 when not foreground),
 *   matched_iou [B, A] fp32, matched_cls [B, A] int32, num_fg [B] int32, num_gt [B] int32.
 *   status [B] int32 (may be NULL): 0, or YX_SIMOTA_CAPACITY (more in-centre anchors than 9*levels*max_gt: the
 *   anchor grid is not one unit-spaced grid per stride level; the surplus was dropped), or YX_SIMOTA_BAD_CLASS (a label
 *   class outside [0, nc): F.one_hot raises in the reference; clamped here). Written by the kernel, no host sync.
 *   levels: number of distinct strides in stride_per_anchor (3 for every named config).
 *   max_gt: label rows per image, 1..512 (the reference pads to 120, data_augment.py:200-208).
 *   workspace: yx_simota_workspace_bytes(B, A, max_gt, levels) bytes.
 * One thread-block cluster per image (up to 8 CTAs): see csrc/yx_simota.cu.
 * ------------------------------------------------------------------------------------------ */
#define YX_SIMOTA_CAPACITY 1
#define YX_SIMOTA_BAD_CLASS 2
int64_t yx_simota_workspace_bytes(int32_t batch, int32_t anchors, int32_t max_gt, int32_t levels);
int yx_simota_assign(const float* pred, const float* labels, const float* x_shift,
                     const float* y_shift, const float* stride_per_anchor, int32_t batch,
                     int32_t anchors, int32_t nc, int32_t max_gt, int32_t levels, uint8_t* fg_mask,
                     int32_t* matched_gt, float* matched_iou, int32_t* matched_cls,
                     int32_t* num_fg, int32_t* num_gt, int32_t* status, void* workspace,
                     int64_t workspace_bytes, void* stream);
/* simota_matching alone (yolo_head.py:542-574) on a given cost / IoU matrix [G, n] fp32
 * (row stride ld): match_gt [n] int32 (-1 = not matched), match_iou [n] fp32, num_fg[1]. */
int yx_simota_matching(const float* cost, const float* ious, int32_t num_gt, int32_t n,
                       int64_t ld, int32_t* match_gt, float* match_iou, int32_t* num_fg,
                       void* stream);

/* ------------------------------------------------------------------------------------------
 * Head losses, forward and gradient in one pass (YoloxHead.get_losses, yolox/models/yolo_head.py:354-418;
 * IOUloss, yolox/models/losses.py:7-51; BCEWithLogits on objectness of every anchor and on the classes of
 * the foreground anchors with target one_hot(matched class) * matched IoU; L1 on the raw regression outputs).
 *   pred / labels / fg_mask / matched_* : as for yx_simota_assign (its outputs are this call's inputs)
 *   origin   : [B, A, 4] fp32 raw regression outputs or NULL (use_l1 off); x_shift/y_shift/stride: [A]
 *   giou     : 0 = loss_type "iou" (1 - iou^2), 1 = "giou"
 *   sums     : [4] fp64 = sum of the iou / obj / cls / l1 terms, NOT divided by num_fg
 *   grad     : [B, A, 5+nc] fp32 = d(reg_weight*iou_sum + obj_sum + cls_sum)/d pred
 *   grad_origin : [B, A, 4] fp32 = d(l1_sum)/d origin (when origin != NULL)
 * The caller divides by max(num_fg, 1) (yolo_head.py:382). No host synchronisation.
 * ------------------------------------------------------------------------------------------ */
int yx_head_losses(const float* pred, const float* labels, int32_t max_gt, const uint8_t* fg_mask,
                   const int32_t* matched_gt, const float* matched_iou, const int32_t* matched_cls,
                   const float* origin, const float* x_shift, const float* y_shift, const float* stride,
                   int32_t batch, int32_t anchors, int32_t nc, int32_t giou, float reg_weight, double* sums,
                   float* grad, float* grad_origin, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training branch of YoloxHead.forward for ONE level (yolox/models/yolo_head.py:161-201, get_output_and_grid :213-231):
 * reg [B,4,h,w], obj [B,1,h,w], cls [B,nc,h,w] contiguous NCHW conv outputs (dtype: YX_FP32 / YX_BF16 / YX_FP16) ->
 * rows [anchor_off, anchor_off + h*w) of out [B, anchors, 5+nc] fp32: xy = (xy + grid) * stride, wh = exp(wh) * stride,
 * raw obj / cls logits; origin (may be NULL): [B, anchors, 4] fp32 raw regression rows (`origin_preds`, :190-200).
 * _bwd: grad_out [B, anchors, 5+nc] fp32 (+ grad_origin or NULL) and the forward's `out` -> gradients of reg / obj / cls
 * in their own layout and dtype.
 * ------------------------------------------------------------------------------------------ */
int yx_head_train_decode(const void* reg, const void* obj, const void* cls, int32_t dtype, int32_t batch, int32_t nc,
                         int32_t h, int32_t w, float stride, int32_t anchors, int32_t anchor_off, float* out,
                         float* origin, void* stream);
int yx_head_train_decode_bwd(const float* grad_out, const float* out, const float* grad_origin, int32_t dtype,
                             int32_t batch, int32_t nc, int32_t h, int32_t w, float stride, int32_t anchors,
                             int32_t anchor_off, void* grad_reg, void* grad_obj, void* grad_cls, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer step + EMA update of every tensor in one launch: torch.optim.SGD(momentum, nesterov, per-group weight decay)
 * as built by yolox/config.py:307-333, and ModelEMA.update (yolox/utils/ema.py:46-58).
 *   table  : device int64 [n_tensors, 6] rows = param ptr | grad ptr (0: EMA only, e.g. BN running statistics) |
 *            momentum-buffer ptr | ema ptr (0: none) | numel | weight decay (fp32 bits in the low word); fp32 tensors
 *   chunks : device int32 [n_chunks, 2] rows = (tensor index, first element); one CTA per chunk of chunk_elems elements
 *   first_step != 0: momentum buffers are initialised with the gradient (torch's first step)
 *   ema_decay d and ema_rest = (float)(1.0 - d) with d = decay * (1 - exp(-updates / 2000)) evaluated by the caller.
 *   hyper (device fp32[3], may be NULL): {lr, ema_decay, ema_rest} read by the kernel INSTEAD of the arguments, so that a
 *   CUDA graph holding this launch follows the schedule (the caller updates the three floats before each replay).
 * ------------------------------------------------------------------------------------------ */
int yx_sgd_ema_step(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, float lr,
                    float momentum, int32_t nesterov, int32_t first_step, float ema_decay, float ema_rest,
                    const float* hyper, void* stream);

/* ------------------------------------------------------------------------------------------
 * Gradient all-reduce + yx_sgd_ema_step as ONE kernel over NVLink peer memory: the data-parallel exchange of the training step
 * (DDP's ncclAllReduce, yolox/core/trainer.py:169) fused with the optimizer step and the EMA update that follow it
 * (core/trainer.py:119-124). Every rank's gradients live in one flat fp32 buffer of `flat_elems` elements allocated as symmetric
 * memory; peer_grad_ptrs[q] (HOST array of `world` addresses) is rank q's buffer as mapped into THIS process, peer_flag_ptrs[q] a
 * zero-initialised symmetric uint32[world] array of rank q (barrier flags). The table's grad pointers must point into the local
 * buffer. Reduce-scatter in rank order (deterministic) -> barrier -> all-gather fused with the update; three node-wide
 * barriers per call. `state`: local device uint32[4], zero-initialised once, owned by the kernel. hyper: device {lr, ema_decay,
 * 1 - ema_decay} (required). Every rank must make the same sequence of calls. world <= 16.
 * ------------------------------------------------------------------------------------------ */
int yx_allreduce_sgd_ema_step(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, float momentum,
                              int32_t nesterov, int32_t first_step, const float* hyper, const int64_t* peer_grad_ptrs,
                              const int64_t* peer_flag_ptrs, int64_t flat_elems, int32_t rank, int32_t world, uint32_t* state,
                              void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-mode BatchNorm2d + activation of a BaseConv (yolox/models/network_blocks.py:27-52 with the BN in train mode;
 * eps / momentum as set by yolox/config.py:165-176), forward and backward, on the conv output x [N, C, H*W] (contiguous
 * NCHW; YX_FP32 / YX_BF16 / YX_FP16), statistics and affine parameters in fp32.
 *   fwd: batch mean / biased variance per channel -> save_mean, save_invstd [C]; running_mean / running_var (may be NULL)
 *        updated with `momentum` and the UNBIASED variance like F.batch_norm; y = act(x_hat * gamma + beta), same dtype as x.
 *   bwd: dy = gradient w.r.t. y -> dx (dtype of x), dgamma, dbeta [C] fp32. x_hat and the pre-activation are recomputed
 *        from x and the saved statistics, nothing else is kept from the forward.
 *   channels_last != 0: x / y / dy / dx are [N*H*W][C] (torch.channels_last, C % 8 == 0), else [N][C][H*W].
 *   dy_ld (channels_last only; 0 = C): per-pixel stride of dy in elements, so that a channel slice of a wider gradient
 *   tensor (the backward of torch.cat) is read in place.
 *   acc_dgamma / acc_dbeta (may be NULL): fp32 [C] buffers the backward ALSO adds dgamma / dbeta to (the parameters' .grad).
 *   num_batches_tracked (may be NULL): nn.BatchNorm2d's int64 call counter, incremented by the forward.
 *   act: YX_ACT_SILU / YX_ACT_RELU / YX_ACT_LRELU / YX_ACT_NONE.  workspace: yx_bn_act_workspace_bytes(N, C, H*W).
 * ------------------------------------------------------------------------------------------ */
int64_t yx_bn_act_workspace_bytes(int32_t n, int32_t c, int32_t hw);
int yx_bn_act_train_fwd(const void* x, int32_t dtype, int32_t channels_last, int32_t n, int32_t c, int32_t hw,
                        const float* gamma,
                        const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                        int64_t* num_batches_tracked, int32_t act, void* y, float* save_mean, float* save_invstd, void* workspace,
                        int64_t workspace_bytes, void* stream);
int yx_bn_act_train_bwd(const void* x, const void* dy, int32_t dtype, int32_t channels_last, int32_t n, int32_t c,
                        int32_t hw,
                        const float* gamma, const float* beta, const float* save_mean, const float* save_invstd,
                        int32_t act, void* dx, float* dgamma, float* dbeta, float* acc_dgamma, float* acc_dbeta, int64_t dy_ld,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training conv stack on the tensor cores: what torch autograd / cuDNN computes for BaseConv.conv and the prediction
 * convs inside Trainer.train_one_iter (yolox/core/trainer.py:96-129: forward, loss.backward()), for the modules of
 * yolox/models/network_blocks.py:27-52 and yolox/models/yolo_head.py:94-120.
 *   forward : yx_conv_bn_act_fwd with w = w_fwd, a zero (or the conv's) bias and YX_ACT_NONE; BatchNorm + activation
 *             follow as yx_bn_act_train_fwd.
 *   dgrad   : the same kernel with w = w_dgrad (weights rotated by 180 degrees, in/out channels swapped) on dy (stride 1)
 *             or on its zero-stuffed copy (stride 2: yx_dilate2 writes z[b, 2*oy, 2*ox] = dy[b, oy, ox], zeros elsewhere;
 *             z has the conv INPUT's spatial size zh x zw).
 *   wgrad   : yx_conv_wgrad, dW[o][tap][i] = sum over output pixels of dy[p][o] * x[p shifted by tap][i]: a tcgen05 GEMM with
 *             both operands MN-major straight from the NHWC tensors (TMA: tap shift, zero padding, stride), the pixel
 *             dimension split over CTAs and reduced in a fixed order. dw: fp32, element (o, i, tap) at
 *             o*dw_stride_o + i*dw_stride_i + tap*dw_stride_tap (tap = 3*kh + kw), so NCHW-contiguous and channels_last
 *             weight gradients are both written in place; only o < out_c_real, i < in_c_real are written (x / dy carry
 *             channel counts padded to multiples of 16: in_c, out_c). accumulate != 0: dw += (gradient accumulation straight
 *             into the parameter's .grad, what autograd's AccumulateGrad would do with one more launch per parameter).
 *   yx_pack_train_weights: fp32 weight (same stride convention) -> w_fwd [o_pad][taps][i_pad] and
 *             w_dgrad [i_pad][taps][o_pad] in `dtype` (either may be NULL), zero padded. subpixel != 0 (3x3 stride-2 convs with
 *             an even input size): w_dgrad is instead [4 * i_pad][9][o_pad], the four sub-pixel phases of the transposed conv as
 *             one stride-1 3x3 conv over dy (phase q = 2 * (row parity) + column parity of the dx pixel; tap (r', s') reads
 *             dy[a + r' - 1, b + s' - 1]; only the positions that carry a weight are written: zero the buffer once), to be run
 *             with yx_conv_desc.shuffle2_c = i_pad -- no zero-stuffed copy, a quarter of the pixels.
 * x, dy: NHWC, 16-bit, per-pixel strides x_ld / dy_ld (multiples of 8), 16-byte aligned. ksize 1 | 3, stride 1 | 2.
 * ------------------------------------------------------------------------------------------ */
int64_t yx_conv_wgrad_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, int32_t in_c, int32_t out_h, int32_t out_w,
                                      int32_t out_c, int32_t ksize, int32_t stride);
int yx_conv_wgrad(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, int32_t dtype, int32_t batch, int32_t in_h,
                  int32_t in_w, int32_t in_c, int32_t out_h, int32_t out_w, int32_t out_c, int32_t ksize, int32_t stride,
                  int32_t in_c_real, int32_t out_c_real, float* dw, int64_t dw_stride_o, int64_t dw_stride_i, int64_t dw_stride_tap,
                  int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream);
int yx_pack_train_weights(const float* w, int64_t stride_o, int64_t stride_i, int64_t stride_tap, int32_t o, int32_t i, int32_t taps,
                          int32_t o_pad, int32_t i_pad, void* w_fwd, void* w_dgrad, int32_t subpixel, int32_t dtype, void* stream);
/* yx_pack_train_weights for every conv of a model in one launch. table: device int64 [n, 12] rows = w ptr | stride_o |
 * stride_i | stride_tap | o | i | taps | o_pad | i_pad | w_fwd ptr | w_dgrad ptr (0: skip) | subpixel; chunks: device int32 [n_chunks, 2]
 * rows = (tensor index, first element of its [o_pad][taps][i_pad] index space), one CTA per chunk of chunk_elems elements. */
int yx_pack_train_weights_multi(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, int32_t dtype,
                                void* stream);
int yx_dilate2(const void* dy, void* z, int32_t batch, int32_t oh, int32_t ow, int32_t zh, int32_t zw, int32_t c, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training depthwise conv (the depthwise BaseConv of DWConv, yolox/models/network_blocks.py:55-74, inside the training step):
 * 3x3, pad 1, no bias, stride 1 | 2, groups = channels = c. Output size oh = (in_h - 1) / stride + 1, ow likewise.
 *   forward : yx_dwconv3x3_train_fwd, y[b, p, c] = sum over taps of x[b, p*stride + tap - 1, c] * w16[c, tap]
 *   dgrad   : yx_dwconv3x3_dgrad, dx[b, q, c] = sum over the taps where (q + 1 - tap) / stride is exact and inside dy of
 *             dy[b, (q + 1 - tap) / stride, c] * w16[c, tap] (a gather: no atomics, no zero-stuffed copy)
 *   wgrad   : yx_dwconv3x3_wgrad, dW[c, tap] = sum over b and output pixels p of dy[b, p, c] * x[b, p*stride + tap - 1, c]: the
 *             pixels split over CTAs (the split depends on the shape and the device only), fp32 partials [split][9][c] in the
 *             caller's workspace (yx_dwconv3x3_wgrad_workspace_bytes; -1 for a bad shape), summed in split order by a second
 *             launch: deterministic. accumulate != 0: dw += (straight into the parameter's .grad).
 * w / dw: the fp32 parameter [c, 1, 3, 3], element (c, tap = 3*kh + kw) at c*w_stride_c + tap*w_stride_tap, so NCHW-contiguous and
 * channels_last weights both work. The forward and the dgrad round w to `dtype` as they read it (autocast's weight cast).
 * x, y, dy, dx: NHWC, dtype YX_BF16 | YX_FP16, per-pixel strides *_ld in elements (multiples of 8, >= c), 16-byte aligned;
 * c % 8 == 0. fp32 accumulation. A bad shape or pointer returns a negative yx_status (message: yx_last_error()).
 * ------------------------------------------------------------------------------------------ */
int yx_dwconv3x3_train_fwd(const void* x, int64_t x_ld, const float* w, int64_t w_stride_c, int64_t w_stride_tap, void* y,
                           int64_t y_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride, int32_t dtype,
                           void* stream);
int yx_dwconv3x3_dgrad(const void* dy, int64_t dy_ld, const float* w, int64_t w_stride_c, int64_t w_stride_tap, void* dx,
                       int64_t dx_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride, int32_t dtype,
                       void* stream);
int64_t yx_dwconv3x3_wgrad_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride);
int yx_dwconv3x3_wgrad(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, int32_t dtype, int32_t batch, int32_t in_h,
                       int32_t in_w, int32_t c, int32_t stride, float* dw, int64_t dw_stride_c, int64_t dw_stride_tap,
                       int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream);

/* Backward of the SPP pools (SPPBottleneck, network_blocks.py:120-142; forward = yx_spp_maxpool on the concat buffer):
 * cat: NHWC buffer whose channels [0, c) hold the pools' input x (pixel stride ld); dout: NHWC gradient of the 4c-channel
 * concat (pixel stride dout_ld); dx32: dense fp32 [B, h, w, c] that the CALLER pre-loads with dout[..., :c] (the identity
 * segment); the gradient of every pooled value is added at the first maximum of its window (torch's tie rule). */
int yx_spp_maxpool_bwd(const void* cat, int64_t ld, const void* dout, int64_t dout_ld, float* dx32, int32_t batch, int32_t h,
                       int32_t w, int32_t c, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Test-time preprocessing on the device (`preproc`, yolox/data/data_augment.py:140-156; YoloxProcessor.__call__,
 * yolox/models/processor.py:30-37): aspect-preserving cv2.resize(INTER_LINEAR) of each decoded HWC uint8 image into the
 * top-left corner of a 114-grey H x W canvas, HWC -> CHW. Bit-exact with OpenCV's 8-bit fixed-point bilinear.
 *   images : device array of `batch` yx_letterbox_image records; out: [batch, channels, H, W] YX_U8 or YX_FP32 (0..255)
 * ------------------------------------------------------------------------------------------ */
typedef struct yx_letterbox_image {
  const uint8_t* src;   /* device pointer, HWC uint8 */
  int32_t h, w;         /* source height / width */
  int64_t pitch;        /* bytes per source row */
} yx_letterbox_image;
int yx_letterbox_u8(const yx_letterbox_image* images, int32_t batch, int32_t channels, int32_t H, int32_t W,
                    void* out, int32_t out_dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Evaluator result rows (CocoEvaluator.convert_to_coco_format, yolox/evaluators/coco_evaluator.py:205-251) from the
 * detections of yx_postprocess / yx_nms_prefiltered: for image b and kept row k < min(det_count[b], max_det):
 * bbox = xyxy / scale[b] -> (x, y, w, h); score = obj * class_conf; category = class_ids[cls] (class_ids may be NULL);
 * rows of all images compacted in image order. Outputs sized batch * max_det rows; total[0] = number written.
 * ------------------------------------------------------------------------------------------ */
int yx_coco_rows(const float* dets, const int32_t* det_count, int32_t batch, int32_t max_det, const float* scale,
                 const int64_t* image_ids, const int32_t* class_ids, int32_t n_class_ids, float* bbox, float* score,
                 int32_t* category, int64_t* image_id, int32_t* total, void* stream);

/* ------------------------------------------------------------------------------------------
 * Plan: the native runtime.  A plan is an ordered list of the launches of one forward pass
 * (YoloxModule.forward eval branch, yolox/models/yolox.py:72-92) over pre-allocated buffers.
 * Tensor maps are encoded once at add time; yx_plan_run enqueues every launch on `stream`
 * from C++ (one FFI call per forward) and can replay them as one CUDA graph.
 * ------------------------------------------------------------------------------------------ */
typedef struct yx_plan yx_plan;
yx_plan* yx_plan_create(void);
void yx_plan_destroy(yx_plan* p);
int yx_plan_add_conv(yx_plan* p, const yx_conv_desc* d);
int yx_plan_add_bottleneck(yx_plan* p, const yx_bneck_desc* d);
int yx_plan_add_dwconv(yx_plan* p, const void* in, int64_t in_ld, const void* w, const float* bias,
                       void* out, int64_t out_ld, int32_t batch, int32_t in_h, int32_t in_w,
                       int32_t c, int32_t stride, int32_t act, int32_t dtype);
int yx_plan_add_spp(yx_plan* p, void* buf, int64_t ld, int32_t batch, int32_t h, int32_t w,
                    int32_t c, int32_t dtype);
int yx_plan_add_focus(yx_plan* p, const void* img, int32_t img_dtype, void* out, int64_t out_ld,
                      int32_t out_dtype, int32_t batch, int32_t h, int32_t w);
int yx_plan_add_focus_conv(yx_plan* p, const void* img, int32_t img_dtype, const void* w,
                           const float* bias, void* out, int64_t out_ld, int32_t batch, int32_t h,
                           int32_t wd, int32_t out_c, int32_t act, int32_t dtype);
int yx_plan_add_postprocess(yx_plan* p, float* pred, int32_t batch, int32_t anchors, int32_t nc,
                            float conf_thre, double nms_thre, int32_t nms_variant,
                            int32_t inplace_xyxy, float* dets, int64_t* det_idx,
                            int32_t* det_count, int32_t max_det, void* workspace,
                            int64_t workspace_bytes);
/* fused-filter variant: yx_plan_add_postprocess_begin goes before the head GEMMs (first op of the plan),
 * yx_plan_add_nms_prefiltered after them */
int yx_plan_add_postprocess_begin(yx_plan* p, void* workspace, int32_t batch, int32_t anchors);
int yx_plan_add_nms_prefiltered(yx_plan* p, int32_t batch, int32_t anchors, double nms_thre, int32_t nms_variant,
                                float* dets, int64_t* det_idx, int32_t* det_count, int32_t max_det,
                                void* workspace, int64_t workspace_bytes);
/* Independent branches. Ops added between yx_plan_begin_lane(lane, after_op) and yx_plan_end_lane belong to side
 * lane `lane` (1..8): in graph mode they run on their own stream, ordered only after main-lane op `after_op`
 * (an index < yx_plan_num_ops, -1 = everything added so far). yx_plan_join_lanes makes the next main-lane op (or
 * the end of the plan) wait for all lanes. Eager runs and yx_plan_profile execute the ops in the order they were
 * added, which must therefore be a valid serial order. Used for the three levels of YoloxHead.forward
 * (yolox/models/yolo_head.py:140-160: the per-level loop has no cross-level dependency). */
int yx_plan_begin_lane(yx_plan* p, int32_t lane, int32_t after_op);
int yx_plan_end_lane(yx_plan* p);
int yx_plan_join_lanes(yx_plan* p);
int yx_plan_num_launches(const yx_plan* p);
int yx_plan_num_ops(const yx_plan* p);
/* Measurement aid: runs the ops one by one (no graph) with a CUDA event between consecutive ops on
 * `stream` and returns each op's device time in milliseconds (ms[i], i < yx_plan_num_ops) and its
 * kind (0 tcgen05 conv, 1 SIMT conv, 2 depthwise, 3 SPP, 4 focus, 5 postprocess, 6 fused focus+stem conv). Synchronises. */
int yx_plan_profile(yx_plan* p, void* stream, float* ms, int32_t* kinds, int32_t capacity);
/* use_graph != 0: capture on first use, replay afterwards. */
int yx_plan_run(yx_plan* p, void* stream, int32_t use_graph);

#ifdef __cplusplus
}
#endif
#endif /* YX_B200_H_ */
