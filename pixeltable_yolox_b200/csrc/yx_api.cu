// C-ABI (include/yx_b200.h) and the plan runtime: an ordered list of pre-encoded launches for
// one YoloxModule.forward (yolox/models/yolox.py:72-92) + postprocess (utils/boxes.py:31-75),
// enqueued from C++ in one FFI call and replayable as a CUDA graph.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "yx_epilogue.cuh"

namespace yx {

// ---- implemented in the kernel translation units ----
struct ConvTcParams;
struct ConvTcLaunch;
int conv_tc_prepare(const yx_conv_desc* d, ConvTcLaunch* L);
int conv_tc_launch(const ConvTcLaunch* L, cudaStream_t stream);
int conv_tc_schedule(const yx_conv_desc* d, int32_t* info, int capacity);
int conv_simt_launch(const yx_conv_desc* d, cudaStream_t stream);
int focus_launch(const void* img, int img_dtype, void* out, long long out_ld, int out_dtype, int batch, int h, int w, cudaStream_t s);
int spp_launch(void* buf, long long ld, int batch, int h, int w, int c, int dtype, cudaStream_t s);
int dwconv_launch(const void* in, long long in_ld, const void* w, const float* bias, void* out, long long out_ld,
                  int batch, int in_h, int in_w, int c, int stride, int act, int dtype, cudaStream_t s);
int pack_launch(const float* src, const float* gamma, const float* beta, const float* mean, const float* var,
                const float* conv_bias, float eps, int o, int i, int kh, int kw, void* dst_w, int dst_dtype,
                int dst_o_off, int dst_i_off, int dst_i_total, float* dst_b, int depthwise, cudaStream_t s);
int decode_launch(float* pred, int batch, int anchors, int nc, const int* hw, const int* strides, int n_levels, cudaStream_t s);
int iou_launch(const float* a, int n, const float* b, int m, int xyxy, float* out, cudaStream_t s);
long long postprocess_ws_bytes(int batch, int anchors);
int postprocess_launch(float* pred, int batch, int anchors, int nc, float conf_thre, double nms_thre, int nms_variant,
                       int inplace_xyxy, float* dets, long long* det_idx, int* det_count, int max_det, void* ws,
                       long long ws_bytes, cudaStream_t s);
int head_loss_launch(const float* pred, const float* labels, int max_gt, const unsigned char* fg_mask, const int* matched_gt,
                     const float* matched_iou, const int* matched_cls, const float* origin, const float* x_shift,
                     const float* y_shift, const float* stride, int batch, int anchors, int nc, int giou, float reg_weight,
                     double* sums, float* grad, float* grad_origin, cudaStream_t s);
int postprocess_ws_ptrs(void* ws, int batch, int anchors, float** cand, unsigned long long** keys, int** counts);
int postprocess_begin_launch(void* ws, int batch, int anchors, cudaStream_t s);
int nms_prefiltered_launch(int batch, int anchors, double nms_thre, int nms_variant, float* dets, long long* det_idx,
                           int* det_count, int max_det, void* ws, long long ws_bytes, cudaStream_t s);
int filter_compact_launch(const float* pred, int batch, int anchors, int nc, float conf_thre, float* cand,
                          int* cand_idx, int* cand_count, void* ws, long long ws_bytes, cudaStream_t s);
int batched_nms_launch(const float* boxes, const float* scores, const int* cls, const int* counts, int batch,
                       int n_max, double nms_thre, int nms_variant, int* keep, int* keep_count, void* ws,
                       long long ws_bytes, cudaStream_t s);
long long simota_ws_bytes(int batch, int anchors, int max_gt, int levels);
int simota_assign_launch(const float* pred, const float* labels, const float* xs, const float* ys, const float* st,
                         int batch, int anchors, int nc, int max_gt, int levels, unsigned char* fg_mask, int* matched_gt,
                         float* matched_iou, int* matched_cls, int* num_fg, int* num_gt, int* status, void* ws,
                         long long ws_bytes, cudaStream_t s);
int simota_matching_launch(const float* cost, const float* ious, int G, int n, long long ld, int* match_gt,
                           float* match_iou, int* num_fg, cudaStream_t s);
int head_train_decode_launch(const void* reg, const void* obj, const void* cls, int dtype, int batch, int nc, int h, int w,
                             float stride, int anchors, int anchor_off, float* out, float* origin, cudaStream_t s);
int head_train_decode_bwd_launch(const float* gout, const float* out, const float* gorigin, int dtype, int batch, int nc, int h,
                                 int w, float stride, int anchors, int anchor_off, void* greg, void* gobj, void* gcls,
                                 cudaStream_t s);
int sgd_ema_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, float lr, float momentum,
                   int nesterov, int first_step, float ema_decay, float ema_rest, const float* hyper, cudaStream_t s);
int letterbox_launch(const void* images_dev, int batch, int channels, int H, int W, void* out, int out_dtype, cudaStream_t s);
int coco_rows_launch(const float* dets, const int* det_count, int batch, int max_det, const float* scale,
                     const long long* image_ids, const int* class_ids, int n_class_ids, float* bbox, float* score,
                     int* category, long long* image_id, int* total, cudaStream_t s);
long long bn_act_ws_bytes(int n, int c, int hw);
int bn_act_train_fwd_launch(const void* x, int dtype, int nhwc, int n, int c, int hw, const float* gamma, const float* beta, float eps,
                            float momentum, float* running_mean, float* running_var, long long* nbt, int act, void* y, float* save_mean,
                            float* save_invstd, void* ws, long long ws_bytes, cudaStream_t s);
int bn_act_train_bwd_launch(const void* x, const void* dy, int dtype, int nhwc, int n, int c, int hw, const float* gamma, const float* beta,
                            const float* save_mean, const float* save_invstd, int act, void* dx, float* dgamma, float* dbeta,
                            float* acc_dgamma, float* acc_dbeta, long long dy_ld, void* ws, long long ws_bytes, cudaStream_t s);
long long wgrad_ws_bytes(int batch, int in_h, int in_w, int in_c, int out_h, int out_w, int out_c, int ksize, int stride);
int wgrad_launch(const void* x, long long x_ld, const void* dy, long long dy_ld, int dtype, int batch, int in_h, int in_w, int in_c,
                 int out_h, int out_w, int out_c, int ksize, int stride, int in_c_real, int out_c_real, float* dw, long long dw_so,
                 long long dw_si, long long dw_st, int accumulate, void* ws, long long ws_bytes, cudaStream_t stream);
int pack_train_weights_launch(const float* w, long long so, long long si, long long st, int o, int i, int taps, int o_pad, int i_pad,
                              void* wf, void* wd, int subpixel, int dtype, cudaStream_t stream);
int dilate2_launch(const void* dy, void* z, int batch, int oh, int ow, int zh, int zw, int c, cudaStream_t stream);
int dw_train_fwd_launch(const void* x, long long x_ld, const float* w, long long w_sc, long long w_st, void* y, long long y_ld,
                        int batch, int in_h, int in_w, int c, int stride, int dtype, cudaStream_t stream);
int dw_dgrad_launch(const void* dy, long long dy_ld, const float* w, long long w_sc, long long w_st, void* dx, long long dx_ld,
                    int batch, int in_h, int in_w, int c, int stride, int dtype, cudaStream_t stream);
long long dw_wgrad_ws_bytes(int batch, int in_h, int in_w, int c, int stride);
int dw_wgrad_launch(const void* x, long long x_ld, const void* dy, long long dy_ld, int dtype, int batch, int in_h, int in_w, int c,
                    int stride, float* dw, long long dw_sc, long long dw_st, int accumulate, void* ws, long long ws_bytes,
                    cudaStream_t stream);
int pack_train_weights_multi_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, int dtype, cudaStream_t stream);
int spp_bwd_launch(const void* cat, long long ld, const void* dout, long long dld, float* dx32, int batch, int h, int w, int c,
                   int dtype, cudaStream_t s);
int allreduce_sgd_ema_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, float momentum, int nesterov,
                             int first_step, const float* hyper, const long long* peer_grad, const long long* peer_flag,
                             long long flat_elems, int rank, int world, unsigned* state, cudaStream_t s);
struct StemLaunch;
StemLaunch* stem_alloc();
void stem_free(StemLaunch*);
int stem_prepare(const void* img, int img_dtype, const void* w, const float* bias, void* out, long long out_ld,
                 int batch, int h, int wd, int out_c, int act, int dtype, StemLaunch* L);
int stem_launch(const StemLaunch* L, cudaStream_t stream);
ConvTcLaunch* conv_tc_alloc();
void conv_tc_free(ConvTcLaunch*);
struct BneckLaunch;
BneckLaunch* bneck_alloc();
void bneck_free(BneckLaunch*);
bool bneck_supported(const yx_bneck_desc* d);
int bneck_prepare(const yx_bneck_desc* d, BneckLaunch* L);
int bneck_launch(const BneckLaunch* L, cudaStream_t stream);

// ---- error plumbing ----
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return YX_ERR_NO_DEVICE;
  return YX_ERR_CUDA;
}

int num_sms() {
  static int cached_dev[kMaxDevices] = {};     // per device: one process may drive several GPUs
  int& cached = cached_dev[current_device_slot()];
  if (!cached) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      cached = 148;
  }
  return cached;
}

int max_smem_optin() {
  static int cached_dev[kMaxDevices] = {};
  int& cached = cached_dev[current_device_slot()];
  if (!cached) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess && n > 0)
      cached = n;
  }
  return cached;
}

int encode_tma(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
               const cuuint64_t* byte_strides, const cuuint32_t* box, const cuuint32_t* elem_strides,
               CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what) {
  // a driver entry point: resolved through the runtime, so the library loads without libcuda
  static const auto encode = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess;
    return reinterpret_cast<decltype(&cuTensorMapEncodeTiled)>(ok ? p : nullptr);
  }();
  YX_REQUIRE(encode != nullptr, YX_ERR_NO_DEVICE, "cuTensorMapEncodeTiled unavailable (no CUDA driver)");
  static const cuuint32_t ones[5] = {1, 1, 1, 1, 1};
  const CUresult r = encode(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, byte_strides, box,
                            elem_strides ? elem_strides : ones, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char shape[192];   // rank <= 5: " size/box" fits 32 characters per dimension
    int n = 0;
    for (int i = 0; i < rank; ++i) n += snprintf(shape + n, sizeof(shape) - n, " %llu/%u", (unsigned long long)dims[i], box[i]);
    set_error("cuTensorMapEncodeTiled(%s) failed: %d (size/box per dimension:%s; row pitch %llu bytes)", what, (int)r, shape,
              rank > 1 ? (unsigned long long)byte_strides[0] : 0ull);
    return YX_ERR_CUDA;
  }
  return YX_OK;
}

static int require_device() {
  static int ok_dev[kMaxDevices] = {};         // checked once per device, not once per process
  int& ok = ok_dev[current_device_slot()];
  if (ok) return YX_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice", __FILE__, __LINE__);
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute", __FILE__, __LINE__);
  YX_REQUIRE(major == 10, YX_ERR_NO_DEVICE,
             "device %d has compute capability %d.x; these kernels are built for sm_100a only (no fallback)", dev, major);
  ok = 1;
  return YX_OK;
}

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
enum OpKind { OP_CONV_TC, OP_CONV_SIMT, OP_DWCONV, OP_SPP, OP_FOCUS, OP_POST, OP_STEM, OP_BNECK, OP_POST_BEGIN, OP_NMS };

struct Op {
  OpKind kind;
  int lane;        // 0 = main stream; > 0: side lane (independent branch)
  int after;       // side lanes: index of the main-lane op whose completion the lane's first op waits for (-1: none)
  bool join;       // before this main-lane op, main waits for every side lane
  ConvTcLaunch* tc;  // OP_CONV_TC
  StemLaunch* stem;  // OP_STEM
  BneckLaunch* bneck;  // OP_BNECK
  yx_conv_desc conv;  // OP_CONV_SIMT
  struct { const void* in; long long in_ld; const void* w; const float* bias; void* out; long long out_ld;
           int batch, in_h, in_w, c, stride, act, dtype; } dw;
  struct { void* buf; long long ld; int batch, h, w, c, dtype; } spp;
  struct { const void* img; int img_dtype; void* out; long long out_ld; int out_dtype, batch, h, w; } focus;
  struct { float* pred; int batch, anchors, nc; float conf; double nms; int variant, inplace; float* dets;
           long long* det_idx; int* det_count; int max_det; void* ws; long long ws_bytes; } post;
};

}  // namespace yx

struct yx_plan {
  std::vector<yx::Op> ops;
  int cur_lane = 0, cur_after = -1;
  bool pending_join = false;
  std::vector<cudaStream_t> lane_streams;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaStream_t capture_stream = nullptr;  // the caller's stream may be the legacy default stream, which cannot capture
  int launches = 0;
};

namespace yx {

static int run_op(const Op& o, cudaStream_t s) {
  switch (o.kind) {
    case OP_CONV_TC: return conv_tc_launch(o.tc, s);
    case OP_STEM: return stem_launch(o.stem, s);
    case OP_BNECK: return bneck_launch(o.bneck, s);
    case OP_CONV_SIMT: return conv_simt_launch(&o.conv, s);
    case OP_DWCONV: return dwconv_launch(o.dw.in, o.dw.in_ld, o.dw.w, o.dw.bias, o.dw.out, o.dw.out_ld, o.dw.batch,
                                         o.dw.in_h, o.dw.in_w, o.dw.c, o.dw.stride, o.dw.act, o.dw.dtype, s);
    case OP_SPP: return spp_launch(o.spp.buf, o.spp.ld, o.spp.batch, o.spp.h, o.spp.w, o.spp.c, o.spp.dtype, s);
    case OP_FOCUS: return focus_launch(o.focus.img, o.focus.img_dtype, o.focus.out, o.focus.out_ld, o.focus.out_dtype,
                                       o.focus.batch, o.focus.h, o.focus.w, s);
    case OP_POST: return postprocess_launch(o.post.pred, o.post.batch, o.post.anchors, o.post.nc, o.post.conf, o.post.nms,
                                            o.post.variant, o.post.inplace, o.post.dets, o.post.det_idx, o.post.det_count,
                                            o.post.max_det, o.post.ws, o.post.ws_bytes, s);
    case OP_POST_BEGIN: return postprocess_begin_launch(o.post.ws, o.post.batch, o.post.anchors, s);
    case OP_NMS: return nms_prefiltered_launch(o.post.batch, o.post.anchors, o.post.nms, o.post.variant, o.post.dets,
                                               o.post.det_idx, o.post.det_count, o.post.max_det, o.post.ws, o.post.ws_bytes, s);
  }
  return YX_ERR_INVALID_ARG;
}

}  // namespace yx

using namespace yx;

extern "C" {

const char* yx_strerror(int code) {
  switch (code) {
    case YX_OK: return "ok";
    case YX_ERR_INVALID_ARG: return "invalid argument";
    case YX_ERR_UNSUPPORTED: return "unsupported shape";
    case YX_ERR_CUDA: return "CUDA error";
    case YX_ERR_NO_DEVICE: return "no sm_100 device (there is no CPU fallback)";
    case YX_ERR_CAPACITY: return "workspace or output too small";
    default: return "unknown error";
  }
}
const char* yx_last_error(void) { return g_err; }
int yx_version(void) { return YX_VERSION; }

int yx_device_check(int dev) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device visible (%s)", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    cudaGetLastError();
    return YX_ERR_NO_DEVICE;
  }
  YX_REQUIRE(dev >= 0 && dev < count, YX_ERR_INVALID_ARG, "device %d out of range (0..%d)", dev, count - 1);
  int major = 0;
  YX_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  YX_REQUIRE(major == 10, YX_ERR_NO_DEVICE, "device %d is sm_%d0, need sm_100", dev, major);
  return YX_OK;
}

int yx_conv_bn_act_fwd(const yx_conv_desc* d, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  YX_REQUIRE(d != nullptr, YX_ERR_INVALID_ARG, "conv: null descriptor");
  if (d->dtype == YX_FP32) return conv_simt_launch(d, (cudaStream_t)stream);
  ConvTcLaunch* L = conv_tc_alloc();
  YX_REQUIRE(L != nullptr, YX_ERR_INVALID_ARG, "conv: out of host memory");
  rc = conv_tc_prepare(d, L);
  if (rc == YX_OK) rc = conv_tc_launch(L, (cudaStream_t)stream);
  conv_tc_free(L);
  return rc;
}

int yx_conv_schedule(const yx_conv_desc* d, int32_t* info, int32_t capacity) {
  int rc = require_device();
  if (rc) return rc;
  YX_REQUIRE(d != nullptr && (info != nullptr || capacity <= 0), YX_ERR_INVALID_ARG, "conv_schedule: null argument");
  YX_REQUIRE(d->dtype != YX_FP32, YX_ERR_UNSUPPORTED, "conv_schedule: fp32 convs run on the SIMT kernel (no tile schedule)");
  return conv_tc_schedule(d, info, capacity);
}

int yx_bottleneck_supported(const yx_bneck_desc* d) { return bneck_supported(d) ? 1 : 0; }

int yx_bottleneck_fwd(const yx_bneck_desc* d, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  BneckLaunch* L = bneck_alloc();
  YX_REQUIRE(L != nullptr, YX_ERR_INVALID_ARG, "bottleneck: out of host memory");
  rc = bneck_prepare(d, L);
  if (rc == YX_OK) rc = bneck_launch(L, (cudaStream_t)stream);
  bneck_free(L);
  return rc;
}

int yx_conv_bn_act_fwd_simt(const yx_conv_desc* d, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return conv_simt_launch(d, (cudaStream_t)stream);
}

int yx_dwconv3x3_bn_act_fwd(const void* in, int64_t in_ld, const void* w, const float* bias, void* out,
                            int64_t out_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride,
                            int32_t act, int32_t dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return dwconv_launch(in, in_ld, w, bias, out, out_ld, batch, in_h, in_w, c, stride, act, dtype, (cudaStream_t)stream);
}

int yx_spp_maxpool(void* buf, int64_t ld, int32_t batch, int32_t h, int32_t w, int32_t c, int32_t dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return spp_launch(buf, ld, batch, h, w, c, dtype, (cudaStream_t)stream);
}

int yx_focus_s2d(const void* img, int32_t img_dtype, void* out, int64_t out_ld, int32_t out_dtype, int32_t batch,
                 int32_t h, int32_t w, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return focus_launch(img, img_dtype, out, out_ld, out_dtype, batch, h, w, (cudaStream_t)stream);
}

int yx_focus_conv_bn_act_fwd(const void* img, int32_t img_dtype, const void* w, const float* bias, void* out,
                             int64_t out_ld, int32_t batch, int32_t h, int32_t wd, int32_t out_c, int32_t act,
                             int32_t dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  StemLaunch* L = stem_alloc();
  YX_REQUIRE(L != nullptr, YX_ERR_INVALID_ARG, "stem: out of host memory");
  rc = stem_prepare(img, img_dtype, w, bias, out, out_ld, batch, h, wd, out_c, act, dtype, L);
  if (rc == YX_OK) rc = stem_launch(L, (cudaStream_t)stream);
  stem_free(L);
  return rc;
}

int yx_pack_weights(const float* src, const float* gamma, const float* beta, const float* mean, const float* var,
                    const float* conv_bias, float eps, int32_t o, int32_t i, int32_t kh, int32_t kw, void* dst_w,
                    int32_t dst_dtype, int32_t dst_o_off, int32_t dst_i_off, int32_t dst_i_total, float* dst_b,
                    int32_t depthwise, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return pack_launch(src, gamma, beta, mean, var, conv_bias, eps, o, i, kh, kw, dst_w, dst_dtype, dst_o_off, dst_i_off,
                     dst_i_total, dst_b, depthwise, (cudaStream_t)stream);
}

int yx_head_decode(float* pred, int32_t batch, int32_t anchors, int32_t nc, const int32_t* hw, const int32_t* strides,
                   int32_t n_levels, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return decode_launch(pred, batch, anchors, nc, hw, strides, n_levels, (cudaStream_t)stream);
}

int64_t yx_postprocess_workspace_bytes(int32_t batch, int32_t anchors) { return postprocess_ws_bytes(batch, anchors); }

int yx_postprocess(float* pred, int32_t batch, int32_t anchors, int32_t nc, float conf_thre, double nms_thre,
                   int32_t nms_variant, int32_t inplace_xyxy, float* dets, int64_t* det_idx, int32_t* det_count,
                   int32_t max_det, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return postprocess_launch(pred, batch, anchors, nc, conf_thre, nms_thre, nms_variant, inplace_xyxy, dets,
                            (long long*)det_idx, det_count, max_det, workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_postprocess_workspace_ptrs(void* workspace, int32_t batch, int32_t anchors, float** cand, uint64_t** keys,
                                  int32_t** counts) {
  return postprocess_ws_ptrs(workspace, batch, anchors, cand, (unsigned long long**)keys, counts);
}

int yx_postprocess_begin(void* workspace, int32_t batch, int32_t anchors, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return postprocess_begin_launch(workspace, batch, anchors, (cudaStream_t)stream);
}

int yx_nms_prefiltered(int32_t batch, int32_t anchors, double nms_thre, int32_t nms_variant, float* dets,
                       int64_t* det_idx, int32_t* det_count, int32_t max_det, void* workspace,
                       int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return nms_prefiltered_launch(batch, anchors, nms_thre, nms_variant, dets, (long long*)det_idx, det_count, max_det,
                                workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_score_filter_compact(const float* pred, int32_t batch, int32_t anchors, int32_t nc, float conf_thre,
                            float* cand, int32_t* cand_idx, int32_t* cand_count, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return filter_compact_launch(pred, batch, anchors, nc, conf_thre, cand, cand_idx, cand_count, workspace,
                               workspace_bytes, (cudaStream_t)stream);
}

int yx_batched_nms(const float* boxes, const float* scores, const int32_t* cls, const int32_t* counts, int32_t batch,
                   int32_t n_max, double nms_thre, int32_t nms_variant, int32_t* keep, int32_t* keep_count,
                   void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return batched_nms_launch(boxes, scores, cls, counts, batch, n_max, nms_thre, nms_variant, keep, keep_count,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_bboxes_iou(const float* a, int32_t n, const float* b, int32_t m, int32_t xyxy, float* out, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return iou_launch(a, n, b, m, xyxy, out, (cudaStream_t)stream);
}

int64_t yx_simota_workspace_bytes(int32_t batch, int32_t anchors, int32_t max_gt, int32_t levels) {
  return simota_ws_bytes(batch, anchors, max_gt, levels);
}

int yx_simota_assign(const float* pred, const float* labels, const float* x_shift, const float* y_shift,
                     const float* stride_per_anchor, int32_t batch, int32_t anchors, int32_t nc, int32_t max_gt,
                     int32_t levels, uint8_t* fg_mask, int32_t* matched_gt, float* matched_iou, int32_t* matched_cls,
                     int32_t* num_fg, int32_t* num_gt, int32_t* status, void* workspace, int64_t workspace_bytes,
                     void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return simota_assign_launch(pred, labels, x_shift, y_shift, stride_per_anchor, batch, anchors, nc, max_gt, levels,
                              fg_mask, matched_gt, matched_iou, matched_cls, num_fg, num_gt, status, workspace,
                              workspace_bytes, (cudaStream_t)stream);
}

int yx_simota_matching(const float* cost, const float* ious, int32_t num_gt, int32_t n, int64_t ld,
                       int32_t* match_gt, float* match_iou, int32_t* num_fg, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return simota_matching_launch(cost, ious, num_gt, n, ld, match_gt, match_iou, num_fg, (cudaStream_t)stream);
}

int yx_head_train_decode(const void* reg, const void* obj, const void* cls, int32_t dtype, int32_t batch, int32_t nc,
                         int32_t h, int32_t w, float stride, int32_t anchors, int32_t anchor_off, float* out,
                         float* origin, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return head_train_decode_launch(reg, obj, cls, dtype, batch, nc, h, w, stride, anchors, anchor_off, out, origin,
                                  (cudaStream_t)stream);
}

int yx_head_train_decode_bwd(const float* grad_out, const float* out, const float* grad_origin, int32_t dtype,
                             int32_t batch, int32_t nc, int32_t h, int32_t w, float stride, int32_t anchors,
                             int32_t anchor_off, void* grad_reg, void* grad_obj, void* grad_cls, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return head_train_decode_bwd_launch(grad_out, out, grad_origin, dtype, batch, nc, h, w, stride, anchors, anchor_off,
                                      grad_reg, grad_obj, grad_cls, (cudaStream_t)stream);
}

int yx_sgd_ema_step(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, float lr,
                    float momentum, int32_t nesterov, int32_t first_step, float ema_decay, float ema_rest,
                    const float* hyper, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return sgd_ema_launch(reinterpret_cast<const long long*>(table), chunks, n_chunks, chunk_elems, lr, momentum, nesterov,
                        first_step, ema_decay, ema_rest, hyper, (cudaStream_t)stream);
}

int yx_allreduce_sgd_ema_step(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, float momentum,
                              int32_t nesterov, int32_t first_step, const float* hyper, const int64_t* peer_grad_ptrs,
                              const int64_t* peer_flag_ptrs, int64_t flat_elems, int32_t rank, int32_t world, uint32_t* state,
                              void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return allreduce_sgd_ema_launch(reinterpret_cast<const long long*>(table), chunks, n_chunks, chunk_elems, momentum, nesterov, first_step,
                                  hyper, reinterpret_cast<const long long*>(peer_grad_ptrs), reinterpret_cast<const long long*>(peer_flag_ptrs),
                                  flat_elems, rank, world, state, (cudaStream_t)stream);
}

int64_t yx_bn_act_workspace_bytes(int32_t n, int32_t c, int32_t hw) { return bn_act_ws_bytes(n, c, hw); }

int yx_bn_act_train_fwd(const void* x, int32_t dtype, int32_t channels_last, int32_t n, int32_t c, int32_t hw, const float* gamma,
                        const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                        int64_t* num_batches_tracked, int32_t act, void* y, float* save_mean, float* save_invstd, void* workspace,
                        int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return bn_act_train_fwd_launch(x, dtype, channels_last, n, c, hw, gamma, beta, eps, momentum, running_mean, running_var,
                                 reinterpret_cast<long long*>(num_batches_tracked), act, y, save_mean,
                                 save_invstd, workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_bn_act_train_bwd(const void* x, const void* dy, int32_t dtype, int32_t channels_last, int32_t n, int32_t c, int32_t hw,
                        const float* gamma, const float* beta, const float* save_mean, const float* save_invstd,
                        int32_t act, void* dx, float* dgamma, float* dbeta, float* acc_dgamma, float* acc_dbeta, int64_t dy_ld,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return bn_act_train_bwd_launch(x, dy, dtype, channels_last, n, c, hw, gamma, beta, save_mean, save_invstd, act, dx, dgamma, dbeta,
                                 acc_dgamma, acc_dbeta, dy_ld, workspace,
                                 workspace_bytes, (cudaStream_t)stream);
}

int64_t yx_conv_wgrad_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, int32_t in_c, int32_t out_h, int32_t out_w,
                                      int32_t out_c, int32_t ksize, int32_t stride) {
  if (require_device()) return -1;
  return wgrad_ws_bytes(batch, in_h, in_w, in_c, out_h, out_w, out_c, ksize, stride);
}

int yx_conv_wgrad(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, int32_t dtype, int32_t batch, int32_t in_h,
                  int32_t in_w, int32_t in_c, int32_t out_h, int32_t out_w, int32_t out_c, int32_t ksize, int32_t stride,
                  int32_t in_c_real, int32_t out_c_real, float* dw, int64_t dw_stride_o, int64_t dw_stride_i, int64_t dw_stride_tap,
                  int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return wgrad_launch(x, x_ld, dy, dy_ld, dtype, batch, in_h, in_w, in_c, out_h, out_w, out_c, ksize, stride, in_c_real, out_c_real,
                      dw, dw_stride_o, dw_stride_i, dw_stride_tap, accumulate, workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_pack_train_weights(const float* w, int64_t stride_o, int64_t stride_i, int64_t stride_tap, int32_t o, int32_t i, int32_t taps,
                          int32_t o_pad, int32_t i_pad, void* w_fwd, void* w_dgrad, int32_t subpixel, int32_t dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return pack_train_weights_launch(w, stride_o, stride_i, stride_tap, o, i, taps, o_pad, i_pad, w_fwd, w_dgrad, subpixel, dtype, (cudaStream_t)stream);
}

int yx_spp_maxpool_bwd(const void* cat, int64_t ld, const void* dout, int64_t dout_ld, float* dx32, int32_t batch, int32_t h,
                       int32_t w, int32_t c, int32_t dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return spp_bwd_launch(cat, ld, dout, dout_ld, dx32, batch, h, w, c, dtype, (cudaStream_t)stream);
}

int yx_pack_train_weights_multi(const int64_t* table, const int32_t* chunks, int32_t n_chunks, int32_t chunk_elems, int32_t dtype,
                                void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return pack_train_weights_multi_launch(reinterpret_cast<const long long*>(table), chunks, n_chunks, chunk_elems, dtype, (cudaStream_t)stream);
}

int yx_dilate2(const void* dy, void* z, int32_t batch, int32_t oh, int32_t ow, int32_t zh, int32_t zw, int32_t c, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return dilate2_launch(dy, z, batch, oh, ow, zh, zw, c, (cudaStream_t)stream);
}

int yx_dwconv3x3_train_fwd(const void* x, int64_t x_ld, const float* w, int64_t w_stride_c, int64_t w_stride_tap, void* y,
                           int64_t y_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride, int32_t dtype,
                           void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return dw_train_fwd_launch(x, x_ld, w, w_stride_c, w_stride_tap, y, y_ld, batch, in_h, in_w, c, stride, dtype, (cudaStream_t)stream);
}

int yx_dwconv3x3_dgrad(const void* dy, int64_t dy_ld, const float* w, int64_t w_stride_c, int64_t w_stride_tap, void* dx,
                       int64_t dx_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride, int32_t dtype,
                       void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return dw_dgrad_launch(dy, dy_ld, w, w_stride_c, w_stride_tap, dx, dx_ld, batch, in_h, in_w, c, stride, dtype, (cudaStream_t)stream);
}

int64_t yx_dwconv3x3_wgrad_workspace_bytes(int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride) {
  if (require_device()) return -1;
  return dw_wgrad_ws_bytes(batch, in_h, in_w, c, stride);
}

int yx_dwconv3x3_wgrad(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, int32_t dtype, int32_t batch, int32_t in_h,
                       int32_t in_w, int32_t c, int32_t stride, float* dw, int64_t dw_stride_c, int64_t dw_stride_tap,
                       int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return dw_wgrad_launch(x, x_ld, dy, dy_ld, dtype, batch, in_h, in_w, c, stride, dw, dw_stride_c, dw_stride_tap, accumulate,
                         workspace, workspace_bytes, (cudaStream_t)stream);
}

int yx_letterbox_u8(const yx_letterbox_image* images, int32_t batch, int32_t channels, int32_t H, int32_t W, void* out,
                    int32_t out_dtype, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return letterbox_launch(images, batch, channels, H, W, out, out_dtype, (cudaStream_t)stream);
}

int yx_coco_rows(const float* dets, const int32_t* det_count, int32_t batch, int32_t max_det, const float* scale,
                 const int64_t* image_ids, const int32_t* class_ids, int32_t n_class_ids, float* bbox, float* score,
                 int32_t* category, int64_t* image_id, int32_t* total, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return coco_rows_launch(dets, det_count, batch, max_det, scale, reinterpret_cast<const long long*>(image_ids), class_ids,
                          n_class_ids, bbox, score, category, reinterpret_cast<long long*>(image_id), total,
                          (cudaStream_t)stream);
}

int yx_head_losses(const float* pred, const float* labels, int32_t max_gt, const uint8_t* fg_mask,
                   const int32_t* matched_gt, const float* matched_iou, const int32_t* matched_cls,
                   const float* origin, const float* x_shift, const float* y_shift, const float* stride,
                   int32_t batch, int32_t anchors, int32_t nc, int32_t giou, float reg_weight, double* sums,
                   float* grad, float* grad_origin, void* stream) {
  int rc = require_device();
  if (rc) return rc;
  return head_loss_launch(pred, labels, max_gt, fg_mask, matched_gt, matched_iou, matched_cls, origin, x_shift, y_shift,
                          stride, batch, anchors, nc, giou, reg_weight, sums, grad, grad_origin, (cudaStream_t)stream);
}

// ---- plan ----
yx_plan* yx_plan_create(void) { return new (std::nothrow) yx_plan(); }

void yx_plan_destroy(yx_plan* p) {
  if (!p) return;
  if (p->exec) cudaGraphExecDestroy(p->exec);
  if (p->graph) cudaGraphDestroy(p->graph);
  if (p->capture_stream) cudaStreamDestroy(p->capture_stream);
  for (auto st : p->lane_streams) if (st) cudaStreamDestroy(st);
  for (auto& o : p->ops) {
    if (o.tc) conv_tc_free(o.tc);
    if (o.stem) stem_free(o.stem);
    if (o.bneck) bneck_free(o.bneck);
  }
  delete p;
}

static void plan_push(yx_plan* p, yx::Op& o) {
  o.lane = p->cur_lane;
  o.after = p->cur_lane ? p->cur_after : -1;
  o.join = (p->cur_lane == 0) && p->pending_join;
  if (o.join) p->pending_join = false;
  p->ops.push_back(o);
}

static void plan_invalidate(yx_plan* p) {
  if (p->exec) { cudaGraphExecDestroy(p->exec); p->exec = nullptr; }
  if (p->graph) { cudaGraphDestroy(p->graph); p->graph = nullptr; }
}

int yx_plan_add_conv(yx_plan* p, const yx_conv_desc* d) {
  YX_REQUIRE(p && d, YX_ERR_INVALID_ARG, "plan_add_conv: null");
  int rc = require_device();
  if (rc) return rc;
  Op o;
  memset(&o, 0, sizeof(o));
  if (d->dtype == YX_FP32) {
    o.kind = OP_CONV_SIMT;
    o.conv = *d;
    EpiParams e;
    rc = fill_epi_params(d, &e);
    if (rc) return rc;
  } else {
    o.kind = OP_CONV_TC;
    o.tc = conv_tc_alloc();
    YX_REQUIRE(o.tc != nullptr, YX_ERR_INVALID_ARG, "plan_add_conv: out of host memory");
    rc = conv_tc_prepare(d, o.tc);
    if (rc) { conv_tc_free(o.tc); return rc; }
  }
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_bottleneck(yx_plan* p, const yx_bneck_desc* d) {
  YX_REQUIRE(p && d, YX_ERR_INVALID_ARG, "plan_add_bottleneck: null");
  int rc = require_device();
  if (rc) return rc;
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_BNECK;
  o.bneck = bneck_alloc();
  YX_REQUIRE(o.bneck != nullptr, YX_ERR_INVALID_ARG, "plan_add_bottleneck: out of host memory");
  rc = bneck_prepare(d, o.bneck);
  if (rc) { bneck_free(o.bneck); return rc; }
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_dwconv(yx_plan* p, const void* in, int64_t in_ld, const void* w, const float* bias, void* out,
                       int64_t out_ld, int32_t batch, int32_t in_h, int32_t in_w, int32_t c, int32_t stride,
                       int32_t act, int32_t dtype) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_dwconv: null plan");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_DWCONV;
  o.dw = {in, in_ld, w, bias, out, out_ld, batch, in_h, in_w, c, stride, act, dtype};
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_spp(yx_plan* p, void* buf, int64_t ld, int32_t batch, int32_t h, int32_t w, int32_t c, int32_t dtype) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_spp: null plan");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_SPP;
  o.spp = {buf, ld, batch, h, w, c, dtype};
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_focus(yx_plan* p, const void* img, int32_t img_dtype, void* out, int64_t out_ld, int32_t out_dtype,
                      int32_t batch, int32_t h, int32_t w) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_focus: null plan");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_FOCUS;
  o.focus = {img, img_dtype, out, out_ld, out_dtype, batch, h, w};
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_focus_conv(yx_plan* p, const void* img, int32_t img_dtype, const void* w, const float* bias, void* out,
                           int64_t out_ld, int32_t batch, int32_t h, int32_t wd, int32_t out_c, int32_t act,
                           int32_t dtype) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_focus_conv: null plan");
  int rc = require_device();
  if (rc) return rc;
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_STEM;
  o.stem = stem_alloc();
  YX_REQUIRE(o.stem != nullptr, YX_ERR_INVALID_ARG, "plan_add_focus_conv: out of host memory");
  rc = stem_prepare(img, img_dtype, w, bias, out, out_ld, batch, h, wd, out_c, act, dtype, o.stem);
  if (rc) { stem_free(o.stem); return rc; }
  plan_push(p, o);
  p->launches += 1;
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_postprocess(yx_plan* p, float* pred, int32_t batch, int32_t anchors, int32_t nc, float conf_thre,
                            double nms_thre, int32_t nms_variant, int32_t inplace_xyxy, float* dets,
                            int64_t* det_idx, int32_t* det_count, int32_t max_det, void* workspace,
                            int64_t workspace_bytes) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_postprocess: null plan");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_POST;
  o.post = {pred, batch, anchors, nc, conf_thre, nms_thre, nms_variant, inplace_xyxy, dets, (long long*)det_idx,
            det_count, max_det, workspace, workspace_bytes};
  plan_push(p, o);
  p->launches += 2;  // filter + sort/NMS kernels (plus one memset node)
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_postprocess_begin(yx_plan* p, void* workspace, int32_t batch, int32_t anchors) {
  YX_REQUIRE(p && workspace && batch > 0 && anchors > 0, YX_ERR_INVALID_ARG, "plan_add_postprocess_begin: bad arguments");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_POST_BEGIN;
  o.post.ws = workspace; o.post.batch = batch; o.post.anchors = anchors;
  plan_push(p, o);            // a memset node, not a kernel launch
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_add_nms_prefiltered(yx_plan* p, int32_t batch, int32_t anchors, double nms_thre, int32_t nms_variant,
                                float* dets, int64_t* det_idx, int32_t* det_count, int32_t max_det, void* workspace,
                                int64_t workspace_bytes) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_add_nms_prefiltered: null plan");
  Op o;
  memset(&o, 0, sizeof(o));
  o.kind = OP_NMS;
  o.post = {nullptr, batch, anchors, 0, 0.0f, nms_thre, nms_variant, 0, dets, (long long*)det_idx, det_count, max_det,
            workspace, workspace_bytes};
  plan_push(p, o);
  p->launches += 1;  // sort/NMS kernel
  plan_invalidate(p);
  return YX_OK;
}

int yx_plan_begin_lane(yx_plan* p, int32_t lane, int32_t after_op) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_begin_lane: null plan");
  YX_REQUIRE(lane >= 1 && lane <= 8, YX_ERR_INVALID_ARG, "plan_begin_lane: lane %d (1..8)", lane);
  YX_REQUIRE(after_op < (int)p->ops.size(), YX_ERR_INVALID_ARG, "plan_begin_lane: after_op %d is not an existing op", after_op);
  YX_REQUIRE(after_op < 0 || p->ops[after_op].lane == 0, YX_ERR_INVALID_ARG, "plan_begin_lane: after_op must be a main-lane op");
  p->cur_lane = lane;
  p->cur_after = after_op;
  return YX_OK;
}

int yx_plan_end_lane(yx_plan* p) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_end_lane: null plan");
  p->cur_lane = 0;
  p->cur_after = -1;
  return YX_OK;
}

int yx_plan_join_lanes(yx_plan* p) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_join_lanes: null plan");
  p->cur_lane = 0;
  p->pending_join = true;     // the next main-lane op (or the end of the plan) waits for every side lane
  return YX_OK;
}

int yx_plan_num_launches(const yx_plan* p) { return p ? p->launches : 0; }
int yx_plan_num_ops(const yx_plan* p) { return p ? (int)p->ops.size() : 0; }

int yx_plan_profile(yx_plan* p, void* stream, float* ms, int32_t* kinds, int32_t capacity) {
  YX_REQUIRE(p && ms && kinds, YX_ERR_INVALID_ARG, "plan_profile: null");
  const int n = (int)p->ops.size();
  YX_REQUIRE(capacity >= n, YX_ERR_CAPACITY, "plan_profile: capacity %d < %d ops", capacity, n);
  int rc = require_device();
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) YX_CUDA(cudaEventCreate(&e));
  YX_CUDA(cudaEventRecord(ev[0], s));
  for (int i = 0; i < n; ++i) {
    rc = run_op(p->ops[i], s);
    if (rc) break;
    cudaEventRecord(ev[i + 1], s);
  }
  cudaError_t e = cudaStreamSynchronize(s);
  if (rc == YX_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
  if (rc == YX_OK) {
    for (int i = 0; i < n; ++i) {
      cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
      kinds[i] = (int32_t)p->ops[i].kind;
    }
  }
  for (auto& ee : ev) cudaEventDestroy(ee);
  return rc;
}

int yx_plan_run(yx_plan* p, void* stream, int32_t use_graph) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "plan_run: null plan");
  int rc = require_device();
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (!use_graph) {
    for (const auto& o : p->ops) {
      rc = run_op(o, s);
      if (rc) return rc;
    }
    return YX_OK;
  }
  if (!p->exec) {
    // warm every kernel once outside capture (cudaFuncSetAttribute etc. are not capturable)
    for (const auto& o : p->ops) {
      rc = run_op(o, s);
      if (rc) return rc;
    }
    YX_CUDA(cudaStreamSynchronize(s));
    if (!p->capture_stream) YX_CUDA(cudaStreamCreateWithFlags(&p->capture_stream, cudaStreamNonBlocking));
    cudaStream_t cs = p->capture_stream;
    // side lanes: one capture stream per lane, forked from / joined to the main stream with events, so that
    // independent branches (the three head levels) become parallel branches of the graph
    int max_lane = 0;
    for (const auto& o : p->ops) if (o.lane > max_lane) max_lane = o.lane;
    while ((int)p->lane_streams.size() < max_lane) {
      cudaStream_t st = nullptr;
      YX_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
      p->lane_streams.push_back(st);
    }
    const int n_ops = (int)p->ops.size();
    std::vector<cudaEvent_t> after_ev(n_ops, nullptr);
    std::vector<cudaEvent_t> all_ev;
    std::vector<char> lane_open(max_lane + 1, 0);     // lane currently holds un-joined work
    std::vector<int> lane_after(max_lane + 1, -2);    // dependency the lane stream has already been made to wait on
    if (max_lane > 0)
      for (const auto& o : p->ops)
        if (o.lane > 0 && o.after >= 0 && !after_ev[o.after]) {
          YX_CUDA(cudaEventCreateWithFlags(&after_ev[o.after], cudaEventDisableTiming));
          all_ev.push_back(after_ev[o.after]);
        }
    auto join_all = [&]() -> int {
      for (int l = 1; l <= max_lane; ++l)
        if (lane_open[l]) {
          cudaEvent_t e = nullptr;
          YX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
          all_ev.push_back(e);
          YX_CUDA(cudaEventRecord(e, p->lane_streams[l - 1]));
          YX_CUDA(cudaStreamWaitEvent(cs, e, 0));
          lane_open[l] = 0;
          lane_after[l] = -2;
        }
      return YX_OK;
    };
    YX_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < n_ops && rc == YX_OK; ++i) {
      const auto& o = p->ops[i];
      const int lane = max_lane > 0 ? o.lane : 0;
      if (lane == 0) {
        if (o.join && max_lane > 0) rc = join_all();
        if (rc == YX_OK) rc = run_op(o, cs);
        if (rc == YX_OK && after_ev[i]) {
          cudaError_t e = cudaEventRecord(after_ev[i], cs);
          if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventRecord", __FILE__, __LINE__);
        }
      } else {
        cudaStream_t ls = p->lane_streams[lane - 1];
        if (!lane_open[lane] || lane_after[lane] != o.after) {
          // fork: the lane joins the capture by waiting on a main-stream event (the op it depends on, or "now")
          cudaEvent_t dep = o.after >= 0 ? after_ev[o.after] : nullptr;
          if (!dep) {
            cudaError_t e = cudaEventCreateWithFlags(&dep, cudaEventDisableTiming);
            if (e == cudaSuccess) { all_ev.push_back(dep); e = cudaEventRecord(dep, cs); }
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventRecord", __FILE__, __LINE__);
          }
          if (rc == YX_OK) {
            cudaError_t e = cudaStreamWaitEvent(ls, dep, 0);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamWaitEvent", __FILE__, __LINE__);
          }
          lane_open[lane] = 1;
          lane_after[lane] = o.after;
        }
        if (rc == YX_OK) rc = run_op(o, ls);
      }
    }
    if (rc == YX_OK && max_lane > 0) rc = join_all();
    if (rc) {
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(cs, &g);
      if (g) cudaGraphDestroy(g);
      for (auto e : all_ev) cudaEventDestroy(e);
      return rc;
    }
    YX_CUDA(cudaStreamEndCapture(cs, &p->graph));
    for (auto e : all_ev) cudaEventDestroy(e);
    YX_CUDA(cudaGraphInstantiate(&p->exec, p->graph, 0));
  }
  YX_CUDA(cudaGraphLaunch(p->exec, s));
  return YX_OK;
}

}  // extern "C"
