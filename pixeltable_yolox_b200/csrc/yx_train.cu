// Training-side kernels next to SimOTA (yx_simota.cu) and the fused head losses (yx_losses.cu):
//
//  1. head_train_decode (+ backward): the training branch of YoloxHead.forward for one level,
//     yolox/models/yolo_head.py:161-201 and get_output_and_grid (:213-231): cat[reg, obj, cls] -> [B, HW, 5+nc] rows,
//     xy = (xy + grid) * stride, wh = exp(wh) * stride, raw logits for obj / cls, plus the raw regression rows
//     (`origin_preds`, :190-200) when the L1 term is on. The reference runs ~12 elementwise / permute / cat kernels per
//     level (and as many in backward); here one transposing pass each way: NCHW conv outputs are read along W
//     (coalesced), staged in shared memory and written as whole [5+nc] rows (coalesced), fp32 out.
//  2. sgd_ema: the reference's optimizer step and EMA update as ONE multi-tensor launch over every parameter and buffer:
//     torch.optim.SGD(momentum, nesterov=True, per-group weight decay) as configured in yolox/config.py:307-333, and
//     ModelEMA.update (yolox/utils/ema.py:46-58): ema = d * ema + (1 - d) * value for every floating-point state tensor.
#include <stdlib.h>
#include <string.h>

#include "yx_common.cuh"

namespace yx {

// ------------------------------------------------------------------------------------------
// 1. training-branch head rows
// ------------------------------------------------------------------------------------------
static constexpr int kHtPix = 32;       // pixels (rows of the output) per CTA
static constexpr int kHtThreads = 256;

template <typename T>
__global__ void __launch_bounds__(kHtThreads)
head_train_decode_kernel(const T* __restrict__ reg, const T* __restrict__ obj, const T* __restrict__ cls, int nc, int hw, int w,
                         float stride, int anchors, int anchor_off, float* __restrict__ out, float* __restrict__ origin) {
  extern __shared__ float ht_tile[];                 // [5+nc][kHtPix + 1]
  const int nch = 5 + nc;
  const int b = blockIdx.y, pix0 = blockIdx.x * kHtPix;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pix = pix0 + lane;
  const bool ok = pix < hw;
  const float gx = (float)(pix % w), gy = (float)(pix / w);
  for (int ch = warp; ch < nch; ch += kHtThreads / 32) {
    const T* src = ch < 4 ? reg + ((long long)b * 4 + ch) * hw : (ch == 4 ? obj + (long long)b * hw : cls + ((long long)b * nc + (ch - 5)) * hw);
    float v = ok ? Cvt<T>::to_f(src[pix]) : 0.0f;
    if (ch < 4 && origin && ok) origin[((long long)b * anchors + anchor_off + pix) * 4 + ch] = v;
    if (ch == 0) v = (v + gx) * stride;
    else if (ch == 1) v = (v + gy) * stride;
    else if (ch < 4) v = expf(v) * stride;
    ht_tile[ch * (kHtPix + 1) + lane] = v;
  }
  __syncthreads();
  const int rows = min(kHtPix, hw - pix0);
  float* dst = out + ((long long)b * anchors + anchor_off + pix0) * nch;
  for (int i = threadIdx.x; i < rows * nch; i += kHtThreads) {
    const int r = i / nch, c = i - r * nch;
    dst[i] = ht_tile[c * (kHtPix + 1) + r];
  }
}

template <typename T>
__global__ void __launch_bounds__(kHtThreads)
head_train_decode_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ out, const float* __restrict__ gorigin,
                             int nc, int hw, float stride, int anchors, int anchor_off, T* __restrict__ greg,
                             T* __restrict__ gobj, T* __restrict__ gcls) {
  extern __shared__ float ht_tile[];
  const int nch = 5 + nc;
  const int b = blockIdx.y, pix0 = blockIdx.x * kHtPix;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rows = min(kHtPix, hw - pix0);
  const long long row0 = (long long)b * anchors + anchor_off + pix0;
  for (int i = threadIdx.x; i < rows * nch; i += kHtThreads) {
    const int r = i / nch, c = i - r * nch;
    float g = gout[row0 * nch + i];
    if (c < 2) g *= stride;                               // d (v + grid) * s / dv
    else if (c < 4) g *= out[row0 * nch + i];             // d exp(v) * s / dv = the decoded value itself
    if (c < 4 && gorigin) g += gorigin[(row0 + r) * 4 + c];
    ht_tile[c * (kHtPix + 1) + r] = g;
  }
  __syncthreads();
  const int pix = pix0 + lane;
  if (pix >= hw) return;
  for (int ch = warp; ch < nch; ch += kHtThreads / 32) {
    T* dst = ch < 4 ? greg + ((long long)b * 4 + ch) * hw : (ch == 4 ? gobj + (long long)b * hw : gcls + ((long long)b * nc + (ch - 5)) * hw);
    dst[pix] = Cvt<T>::from_f(ht_tile[ch * (kHtPix + 1) + lane]);
  }
}

static int head_train_check(int dtype, int batch, int nc, int h, int w, int anchors, int anchor_off) {
  YX_REQUIRE(dtype == YX_FP32 || dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_INVALID_ARG, "head_train_decode: dtype %d", dtype);
  YX_REQUIRE(batch > 0 && nc > 0 && h > 0 && w > 0, YX_ERR_INVALID_ARG, "head_train_decode: bad sizes");
  YX_REQUIRE(anchor_off >= 0 && anchor_off + h * w <= anchors, YX_ERR_INVALID_ARG, "head_train_decode: level [%d, %d) outside %d anchors",
             anchor_off, anchor_off + h * w, anchors);
  YX_REQUIRE((size_t)(5 + nc) * (kHtPix + 1) * 4 <= 48 * 1024, YX_ERR_UNSUPPORTED, "head_train_decode: %d classes exceed the row staging", nc);
  YX_REQUIRE(batch <= 65535, YX_ERR_UNSUPPORTED, "head_train_decode: batch %d", batch);
  return YX_OK;
}

int head_train_decode_launch(const void* reg, const void* obj, const void* cls, int dtype, int batch, int nc, int h, int w,
                             float stride, int anchors, int anchor_off, float* out, float* origin, cudaStream_t s) {
  YX_REQUIRE(reg && obj && cls && out, YX_ERR_INVALID_ARG, "head_train_decode: null pointer");
  int rc = head_train_check(dtype, batch, nc, h, w, anchors, anchor_off);
  if (rc) return rc;
  const int hw = h * w;
  const dim3 grid((unsigned)((hw + kHtPix - 1) / kHtPix), (unsigned)batch);
  const size_t smem = (size_t)(5 + nc) * (kHtPix + 1) * 4;
#define YX_GO(T) head_train_decode_kernel<T><<<grid, kHtThreads, smem, s>>>((const T*)reg, (const T*)obj, (const T*)cls, nc, hw, w, stride, anchors, anchor_off, out, origin)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int head_train_decode_bwd_launch(const float* gout, const float* out, const float* gorigin, int dtype, int batch, int nc, int h,
                                 int w, float stride, int anchors, int anchor_off, void* greg, void* gobj, void* gcls,
                                 cudaStream_t s) {
  YX_REQUIRE(gout && out && greg && gobj && gcls, YX_ERR_INVALID_ARG, "head_train_decode_bwd: null pointer");
  int rc = head_train_check(dtype, batch, nc, h, w, anchors, anchor_off);
  if (rc) return rc;
  const int hw = h * w;
  const dim3 grid((unsigned)((hw + kHtPix - 1) / kHtPix), (unsigned)batch);
  const size_t smem = (size_t)(5 + nc) * (kHtPix + 1) * 4;
#define YX_GO(T) head_train_decode_bwd_kernel<T><<<grid, kHtThreads, smem, s>>>(gout, out, gorigin, nc, hw, stride, anchors, anchor_off, (T*)greg, (T*)gobj, (T*)gcls)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

// ------------------------------------------------------------------------------------------
// 2. SGD (momentum, nesterov, weight decay) + EMA, every tensor in one launch
// ------------------------------------------------------------------------------------------
// table row (int64 x 6): param ptr | grad ptr (0: no optimizer step, EMA only -- BN running statistics) | momentum buffer
// ptr | ema ptr (0: none) | numel | weight-decay bits (float in the low 32 bits). chunks: (tensor index, first element).
static constexpr int kSgdThreads = 256;

__global__ void __launch_bounds__(kSgdThreads)
sgd_ema_kernel(const long long* __restrict__ table, const int* __restrict__ chunks, int chunk_elems, float lr, float momentum,
               int nesterov, int first_step, float ema_decay, float ema_rest, const float* __restrict__ hyper) {
  // hyper (device, may be null): {lr, ema_decay, 1 - ema_decay} read at run time, so that a CUDA graph that captured this
  // launch follows the learning-rate schedule and the EMA ramp without being re-captured
  if (hyper) { lr = hyper[0]; ema_decay = hyper[1]; ema_rest = hyper[2]; }
  const int t = chunks[2 * blockIdx.x], e0 = chunks[2 * blockIdx.x + 1];
  const long long* row = table + (long long)t * 6;
  float* p = reinterpret_cast<float*>(row[0]);
  const float* g = reinterpret_cast<const float*>(row[1]);
  float* buf = reinterpret_cast<float*>(row[2]);
  float* ema = reinterpret_cast<float*>(row[3]);
  const long long n = row[4];
  const float wd = __int_as_float((int)(row[5] & 0xffffffffll));
  const long long e1 = min(n, (long long)e0 + chunk_elems);
  // 16-byte vectors when the tensor allows it (every conv weight and BatchNorm vector of the named configs): the kernel moves
  // eight fp32 streams, 4-byte accesses left it at 3.1 TB/s
  const bool vec = (n & 3) == 0 && (e0 & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(buf) |
                     reinterpret_cast<uintptr_t>(ema)) & 15) == 0;
  if (vec) {
    for (long long i = (e0 >> 2) + threadIdx.x; i < (e1 >> 2); i += kSgdThreads) {
      const float4 pv = reinterpret_cast<const float4*>(p)[i];
      float v[4] = {pv.x, pv.y, pv.z, pv.w};
      if (g) {
        const float4 gv = reinterpret_cast<const float4*>(g)[i];
        float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
        if (momentum != 0.0f && !first_step) bq = reinterpret_cast<const float4*>(buf)[i];
        const float d4[4] = {gv.x, gv.y, gv.z, gv.w}, b4[4] = {bq.x, bq.y, bq.z, bq.w};
        float nb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float d = d4[k];
          if (wd != 0.0f) d = fmaf(wd, v[k], d);
          if (momentum != 0.0f) {
            nb[k] = first_step ? d : __fadd_rn(__fmul_rn(momentum, b4[k]), d);
            d = nesterov ? fmaf(momentum, nb[k], d) : nb[k];
          }
          v[k] = fmaf(-lr, d, v[k]);
        }
        if (momentum != 0.0f) reinterpret_cast<float4*>(buf)[i] = make_float4(nb[0], nb[1], nb[2], nb[3]);
        reinterpret_cast<float4*>(p)[i] = make_float4(v[0], v[1], v[2], v[3]);
      }
      if (ema) {
        const float4 eq = reinterpret_cast<const float4*>(ema)[i];
        const float e4[4] = {eq.x, eq.y, eq.z, eq.w};
        float r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = __fadd_rn(__fmul_rn(e4[k], ema_decay), __fmul_rn(ema_rest, v[k]));
        reinterpret_cast<float4*>(ema)[i] = make_float4(r[0], r[1], r[2], r[3]);
      }
    }
    return;
  }
  for (long long i = e0 + threadIdx.x; i < e1; i += kSgdThreads) {
    float v = p[i];
    if (g) {
      // torch.optim.SGD._single_tensor_sgd: d = g + wd * p; buf = first ? d : momentum * buf + d;
      //                                     d = nesterov ? d + momentum * buf : buf; p -= lr * d
      float d = g[i];
      if (wd != 0.0f) d = fmaf(wd, v, d);
      if (momentum != 0.0f) {
        const float bv = first_step ? d : __fadd_rn(__fmul_rn(momentum, buf[i]), d);   // buf.mul_(momentum).add_(d): two roundings
        buf[i] = bv;
        d = nesterov ? fmaf(momentum, bv, d) : bv;
      }
      v = fmaf(-lr, d, v);
      p[i] = v;
    }
    // v *= d; v += (1 - d) * msd[k]  (ema.py:56-58): three roundings, (1 - d) evaluated in double on the host
    if (ema) ema[i] = __fadd_rn(__fmul_rn(ema[i], ema_decay), __fmul_rn(ema_rest, v));
  }
}

int sgd_ema_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, float lr, float momentum,
                   int nesterov, int first_step, float ema_decay, float ema_rest, const float* hyper, cudaStream_t s) {
  YX_REQUIRE(table && chunks, YX_ERR_INVALID_ARG, "sgd_ema: null table");
  YX_REQUIRE(n_chunks >= 0 && chunk_elems > 0, YX_ERR_INVALID_ARG, "sgd_ema: bad chunking");
  if (n_chunks == 0) return YX_OK;
  sgd_ema_kernel<<<n_chunks, kSgdThreads, 0, s>>>(table, chunks, chunk_elems, lr, momentum, nesterov, first_step, ema_decay, ema_rest, hyper);
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}


// ------------------------------------------------------------------------------------------
// 3. Training-mode BatchNorm + activation, forward and backward (the BN + SiLU of every BaseConv in the training step:
//    yolox/models/network_blocks.py:27-52 with nn.BatchNorm2d in train mode, eps / momentum from yolox/config.py:165-176)
// ------------------------------------------------------------------------------------------
// torch runs four to six kernels per layer and direction (collect statistics, transform, silu; silu_backward,
// batch_norm_backward); at 8 images per GPU they were 52 % of the step's GPU time (8.7 of 16.8 ms, tools/gpu_prof_train.py).
// Here: x is the conv output [N, C, H*W] (NCHW, bf16 / fp16 / fp32), statistics in fp32.
//   forward : bn_stats (partial sum / sum of squares per (channel, slab chunk)) -> bn_finalize (mean, 1/std, running
//             statistics with torch's unbiased variance) -> bn_act_apply (y = act(x_hat * gamma + beta))
//   backward: bn_act_bwd_reduce (dz = dy * act'(z); sum dz, sum dz * x_hat) -> finalize (dgamma, dbeta) ->
//             bn_act_bwd_apply (dx = gamma / std * (dz - dbeta / M - x_hat * dgamma / M))
// z and x_hat are recomputed from x, never stored. 16-byte loads when H*W is a multiple of 8 (every map of the named configs).
static constexpr int kBnThreads = 256;
static constexpr int kBnChunk = 8192;        // elements of one (n, c) slab per CTA

template <typename T> struct Vec8;
template <> struct Vec8<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { v[2 * j] = __uint_as_float(w[j] << 16); v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u); }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]); w[j] = *reinterpret_cast<uint32_t*>(&h); }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
template <> struct Vec8<__half> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const __half* p, float (&v)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j])); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
  }
  static __device__ __forceinline__ void store(__half* p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]); w[j] = *reinterpret_cast<uint32_t*>(&h); }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
template <> struct Vec8<float> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
};

__device__ __forceinline__ float2 block_sum2(float a, float b) {
  __shared__ float sa[kBnThreads / 32], sb[kBnThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sa[warp] = a; sb[warp] = b; }
  __syncthreads();
  if (warp == 0) {
    a = lane < kBnThreads / 32 ? sa[lane] : 0.0f; b = lane < kBnThreads / 32 ? sb[lane] : 0.0f;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  }
  return make_float2(a, b);       // valid in thread 0
}

// act: YX_ACT_SILU / RELU / LRELU / NONE. value and derivative at z.
__device__ __forceinline__ float bn_act(float z, int act) {
  if (act == YX_ACT_SILU) return z / (1.0f + __expf(-z));
  if (act == YX_ACT_RELU) return fmaxf(z, 0.0f);
  if (act == YX_ACT_LRELU) return z > 0.0f ? z : 0.1f * z;
  return z;
}
// bf16 tensors (8-bit significand): SiLU and its derivative from ONE MUFU, sigmoid(z) = 0.5 + 0.5 * tanh(z / 2) with
// tanh.approx (2^-11 absolute, below the output rounding) instead of ex2 + a full-precision division: the forward apply pass
// of the 52 MB stem tensor was issue-bound (56 us for 105 MB), like the inference epilogues before the same change.
template <typename T> struct BnFast { static constexpr bool value = false; };
template <> struct BnFast<__nv_bfloat16> { static constexpr bool value = true; };
__device__ __forceinline__ float tanh_approx(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x));
  return t;
}
template <bool FAST>
__device__ __forceinline__ float bn_act_t(float z, int act) {
  if (FAST && act == YX_ACT_SILU) { const float h = 0.5f * z; return fmaf(h, tanh_approx(h), h); }
  return bn_act(z, act);
}
__device__ __forceinline__ float bn_act_grad(float z, int act);
template <bool FAST>
__device__ __forceinline__ float bn_act_grad_t(float z, int act) {
  if (FAST && act == YX_ACT_SILU) {
    const float s = fmaf(0.5f, tanh_approx(0.5f * z), 0.5f);
    return s * fmaf(z, 1.0f - s, 1.0f);
  }
  return bn_act_grad(z, act);
}
__device__ __forceinline__ float bn_act_grad(float z, int act) {
  if (act == YX_ACT_SILU) { const float s = 1.0f / (1.0f + __expf(-z)); return s * (1.0f + z * (1.0f - s)); }
  if (act == YX_ACT_RELU) return z > 0.0f ? 1.0f : 0.0f;
  if (act == YX_ACT_LRELU) return z > 0.0f ? 1.0f : 0.1f;
  return 1.0f;
}

// grid (chunks, C, N): CTA (k, c, n) covers elements [k * kBnChunk, ...) of slab (n, c). part: [C][N * chunks][2]
template <typename T, bool BWD>
__global__ void __launch_bounds__(kBnThreads)
bn_reduce_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ mean, const float* __restrict__ invstd,
                 const float* __restrict__ gamma, const float* __restrict__ beta, int C, int HW, int act, float* __restrict__ part) {
  pdl_wait();               // programmatic dependent launch: our prologue overlapped the predecessor's tail
  pdl_launch_dependents();
  const int c = blockIdx.y, n = blockIdx.z, k = blockIdx.x;
  const long long base = ((long long)n * C + c) * HW;
  const int lo = k * kBnChunk, hi = min(HW, lo + kBnChunk);
  float s0 = 0.0f, s1 = 0.0f;
  float mu = 0.0f, a = 1.0f, b = 0.0f, is = 1.0f;
  if (BWD) { mu = mean[c]; is = invstd[c]; a = gamma[c]; b = beta[c]; }
  auto one = [&](float xv, float dv) {
    if (BWD) {
      const float xh = (xv - mu) * is;
      const float dz = dv * bn_act_grad(fmaf(xh, a, b), act);
      s0 += dz; s1 = fmaf(dz, xh, s1);
    } else {
      s0 += xv; s1 = fmaf(xv, xv, s1);
    }
  };
  if ((HW & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (!BWD || (reinterpret_cast<uintptr_t>(dy) & 15) == 0)) {
    for (int i = lo + threadIdx.x * 8; i < hi; i += kBnThreads * 8) {
      float xv[8], dv[8];
      Vec8<T>::load(x + base + i, xv);
      if (BWD) Vec8<T>::load(dy + base + i, dv);
#pragma unroll
      for (int j = 0; j < 8; ++j) one(xv[j], BWD ? dv[j] : 0.0f);
    }
  } else {
    for (int i = lo + threadIdx.x; i < hi; i += kBnThreads) one(Cvt<T>::to_f(x[base + i]), BWD ? Cvt<T>::to_f(dy[base + i]) : 0.0f);
  }
  const float2 r = block_sum2(s0, s1);
  if (threadIdx.x == 0) {
    const long long p = ((long long)c * gridDim.z * gridDim.x + (long long)n * gridDim.x + k) * 2;
    part[p] = r.x; part[p + 1] = r.y;
  }
}

// one warp per channel (the S partials of a channel are contiguous: coalesced loads, fp64 shuffle reduction; one THREAD per
// channel walked its up to 592 partials serially and cost 44 us per launch, 6.5 ms of the channels_last training step).
// FWD: mean / invstd + running statistics; BWD: dbeta (sum dz), dgamma (sum dz * x_hat)
__global__ void bn_finalize_kernel(const float* __restrict__ part, int C, int S, double M, float eps, float momentum,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ out0, float* __restrict__ out1, int bwd, long long* __restrict__ nbt,
                                   float* __restrict__ acc0, float* __restrict__ acc1) {
  pdl_wait();               // programmatic dependent launch: our prologue overlapped the predecessor's tail
  pdl_launch_dependents();
  const int c = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  if (nbt && c == 0 && lane == 0) *nbt += 1;           // nn.BatchNorm2d.num_batches_tracked
  const float2* p2 = reinterpret_cast<const float2*>(part) + (long long)c * S;
  double a = 0.0, b = 0.0;
  for (int s = lane; s < S; s += 32) { const float2 v = p2[s]; a += (double)v.x; b += (double)v.y; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  if (lane) return;
  if (bwd) {
    out0[c] = (float)a; out1[c] = (float)b;
    if (acc0) acc0[c] += (float)a;                       // gradient accumulation into the parameters' .grad (dbeta, dgamma)
    if (acc1) acc1[c] += (float)b;
    return;
  }
  const double mean = a / M;
  double var = b / M - mean * mean;
  if (var < 0.0) var = 0.0;
  out0[c] = (float)mean;
  out1[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) {                                  // F.batch_norm: running_var takes the unbiased estimate
    const double unbiased = M > 1.0 ? var * M / (M - 1.0) : var;
    running_mean[c] = (float)((1.0 - (double)momentum) * (double)running_mean[c] + (double)momentum * mean);
    running_var[c] = (float)((1.0 - (double)momentum) * (double)running_var[c] + (double)momentum * unbiased);
  }
}

// FWD: y = act(x_hat * gamma + beta).  BWD: dx = gamma * invstd * (dz - dbeta / M - x_hat * dgamma / M)
template <typename T, bool BWD>
__global__ void __launch_bounds__(kBnThreads)
bn_apply_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ mean, const float* __restrict__ invstd,
                const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ dbeta,
                const float* __restrict__ dgamma, float inv_m, int C, int HW, int act, T* __restrict__ out) {
  pdl_wait();               // programmatic dependent launch: our prologue overlapped the predecessor's tail
  pdl_launch_dependents();
  const int c = blockIdx.y, n = blockIdx.z, k = blockIdx.x;
  const long long base = ((long long)n * C + c) * HW;
  const int lo = k * kBnChunk, hi = min(HW, lo + kBnChunk);
  const float mu = mean[c], is = invstd[c], g = gamma[c], b = beta[c];
  float k0 = 0.0f, k1 = 0.0f, gi = 0.0f;
  if (BWD) { k0 = dbeta[c] * inv_m; k1 = dgamma[c] * inv_m; gi = g * is; }
  auto one = [&](float xv, float dv) -> float {
    const float xh = (xv - mu) * is;
    const float z = fmaf(xh, g, b);
    if (!BWD) return bn_act(z, act);
    const float dz = dv * bn_act_grad(z, act);
    return gi * (dz - k0 - xh * k1);
  };
  const bool vec = (HW & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                   (!BWD || (reinterpret_cast<uintptr_t>(dy) & 15) == 0);
  if (vec) {
    for (int i = lo + threadIdx.x * 8; i < hi; i += kBnThreads * 8) {
      float xv[8], dv[8], r[8];
      Vec8<T>::load(x + base + i, xv);
      if (BWD) Vec8<T>::load(dy + base + i, dv);
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = one(xv[j], BWD ? dv[j] : 0.0f);
      Vec8<T>::store(out + base + i, r);
    }
  } else {
    for (int i = lo + threadIdx.x; i < hi; i += kBnThreads)
      out[base + i] = Cvt<T>::from_f(one(Cvt<T>::to_f(x[base + i]), BWD ? Cvt<T>::to_f(dy[base + i]) : 0.0f));
  }
}

// ---- channels-last: x is [M = N*H*W][C] with C contiguous (torch.channels_last, the layout of every kernel of this package and
// of cuDNN's 16-bit kernels: with NCHW tensors 1.9 ms of a 8.7 ms step were cuDNN's own nchw<->nhwc conversion kernels). A
// thread owns 8 consecutive channels (one 16-byte load per row) and strides over the rows of its CTA's slab; the threads of a
// column are reduced through shared memory. Requires C % 8 == 0.
// (A single cooperative launch per direction -- statistics, grid barrier, finalize spread over the grid, grid barrier, apply from
// L2 -- measured SLOWER than three launches: 16 vs 11 us on a 0.8 MB tensor, 81 vs 50 us on 52 MB; the sense-reversing barrier
// with its fences costs more than the launch it saves. Kept out of the build.)
__device__ __forceinline__ void bn_ld8(const float* p, float (&v)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// partial sums of every channel over the CTA's row slab; U rows in flight per thread. part: [C][S] float2
template <typename T, bool BWD, int U>
__global__ void __launch_bounds__(kBnThreads)
bn_reduce_nhwc_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ mean, const float* __restrict__ invstd,
                      const float* __restrict__ gamma, const float* __restrict__ beta, long long M, int C, int rows_per_cta, int act,
                      float* __restrict__ part, long long dy_ld) {
  pdl_wait();               // programmatic dependent launch: our prologue overlapped the predecessor's tail
  pdl_launch_dependents();
  __shared__ float red[kBnThreads][17];
  const int S = gridDim.x;
  const int cg = C >> 3;
  const int tpr = cg < kBnThreads ? cg : kBnThreads;          // threads per row
  const int rpi = kBnThreads / tpr;                            // rows per iteration
  const int col = threadIdx.x % tpr, row0 = threadIdx.x / tpr;
  const long long m_lo = (long long)blockIdx.x * rows_per_cta, m_hi = min(M, m_lo + rows_per_cta);
  const bool active = row0 < rpi;
  for (int cc = col; cc < cg; cc += tpr) {
    float s0[8], s1[8], mu[8], is[8], a[8], b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s0[j] = 0.0f; s1[j] = 0.0f; }
    if (BWD) { bn_ld8(mean + cc * 8, mu); bn_ld8(invstd + cc * 8, is); bn_ld8(gamma + cc * 8, a); bn_ld8(beta + cc * 8, b); }
    if (active) {
      for (long long m = m_lo + row0; m < m_hi; m += (long long)U * rpi) {
        float xv[U][8], dv[U][8];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long mm = m + (long long)u * rpi;
          if (mm < m_hi) {
            Vec8<T>::load(x + mm * C + cc * 8, xv[u]);
            if (BWD) Vec8<T>::load(dy + mm * dy_ld + cc * 8, dv[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (m + (long long)u * rpi < m_hi) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (BWD) {
                const float xh = (xv[u][j] - mu[j]) * is[j];
                const float dz = dv[u][j] * bn_act_grad_t<BnFast<T>::value>(fmaf(xh, a[j], b[j]), act);
                s0[j] += dz; s1[j] = fmaf(dz, xh, s1[j]);
              } else {
                s0[j] += xv[u][j]; s1[j] = fmaf(xv[u][j], xv[u][j], s1[j]);
              }
            }
          }
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) { red[threadIdx.x][j] = s0[j]; red[threadIdx.x][8 + j] = s1[j]; }
    __syncthreads();
    // column sums: thread t < 16 * tpr... every (column, value) pair gets its own thread when there are enough
    for (int t = threadIdx.x; t < tpr * 16; t += kBnThreads) {
      const int cl = t >> 4, j = t & 15;
      float acc = 0.0f;
      for (int r = 0; r < rpi; ++r) acc += red[r * tpr + cl][j];
      // j < 8: sum 0 of channel (cc0 + cl) * 8 + j; j >= 8: sum 1 of channel ... + j - 8, where cc0 = cc - col
      part[((long long)((cc - col + cl) * 8 + (j & 7)) * S + blockIdx.x) * 2 + (j >> 3)] = acc;
    }
  }
}

// FWD: y = act(x_hat * gamma + beta).  BWD: dx = gamma * invstd * (dz - dbeta / M - x_hat * dgamma / M)
template <typename T, bool BWD, int U>
__global__ void __launch_bounds__(kBnThreads)
bn_apply_nhwc_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ mean, const float* __restrict__ invstd,
                     const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ dbeta,
                     const float* __restrict__ dgamma, float inv_m, long long M, int C, int rows_per_cta, int act, T* __restrict__ out,
                     long long dy_ld) {
  pdl_wait();               // programmatic dependent launch: our prologue overlapped the predecessor's tail
  pdl_launch_dependents();
  const int cg = C >> 3;
  const int tpr = cg < kBnThreads ? cg : kBnThreads;
  const int rpi = kBnThreads / tpr;
  const int col = threadIdx.x % tpr, row0 = threadIdx.x / tpr;
  const long long m_lo = (long long)blockIdx.x * rows_per_cta, m_hi = min(M, m_lo + rows_per_cta);
  if (row0 >= rpi) return;
  for (int cc = col; cc < cg; cc += tpr) {
    float mu[8], is[8], g[8], b[8], k0[8], k1[8];
    bn_ld8(mean + cc * 8, mu); bn_ld8(invstd + cc * 8, is); bn_ld8(gamma + cc * 8, g); bn_ld8(beta + cc * 8, b);
    if (BWD) {
      bn_ld8(dbeta + cc * 8, k0); bn_ld8(dgamma + cc * 8, k1);
#pragma unroll
      for (int j = 0; j < 8; ++j) { k0[j] *= inv_m; k1[j] *= inv_m; }
    }
    for (long long m = m_lo + row0; m < m_hi; m += (long long)U * rpi) {
      float xv[U][8], dv[U][8];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long mm = m + (long long)u * rpi;
        if (mm < m_hi) {
          Vec8<T>::load(x + mm * C + cc * 8, xv[u]);
          if (BWD) Vec8<T>::load(dy + mm * dy_ld + cc * 8, dv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long mm = m + (long long)u * rpi;
        if (mm < m_hi) {
          float r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float xh = (xv[u][j] - mu[j]) * is[j];
            const float z = fmaf(xh, g[j], b[j]);
            if (!BWD) r[j] = bn_act_t<BnFast<T>::value>(z, act);
            else r[j] = g[j] * is[j] * (dv[u][j] * bn_act_grad_t<BnFast<T>::value>(z, act) - k0[j] - xh * k1[j]);
          }
          Vec8<T>::store(out + mm * C + cc * 8, r);
        }
      }
    }
  }
}

// row slabs of the channels-last kernels: at least `min_rows` rows per CTA, at most `waves` CTAs per SM
static int bn_nhwc_slabs(long long M, int min_rows, int waves, int* rows_per_cta) {
  long long s = (M + min_rows - 1) / min_rows;
  long long cap = (long long)waves * num_sms();
  if (cap > 1024) cap = 1024;                           // bn_act_ws_bytes reserves 1024 slabs per channel
  if (s > cap) s = cap;
  if (s < 1) s = 1;
  *rows_per_cta = (int)((M + s - 1) / s);
  return (int)((M + *rows_per_cta - 1) / *rows_per_cta);
}

long long bn_act_ws_bytes(int n, int c, int hw) {
  if (n <= 0 || c <= 0 || hw <= 0) return 256;
  const long long chunks = (hw + kBnChunk - 1) / kBnChunk;
  long long parts = (long long)n * chunks;
  const long long nhwc_parts = 1024;                         // the fused channels_last kernel never uses more CTAs
  if (parts < nhwc_parts) parts = nhwc_parts;
  return (((long long)c * parts * 2 * 4) + 255) & ~255LL;
}

static int bn_check(int dtype, int n, int c, int hw, int act) {
  YX_REQUIRE(dtype == YX_FP32 || dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_INVALID_ARG, "bn_act: dtype %d", dtype);
  YX_REQUIRE(n > 0 && c > 0 && hw > 0 && n <= 65535 && c <= 65535, YX_ERR_INVALID_ARG, "bn_act: bad sizes");
  YX_REQUIRE(act == YX_ACT_SILU || act == YX_ACT_RELU || act == YX_ACT_LRELU || act == YX_ACT_NONE, YX_ERR_INVALID_ARG, "bn_act: act %d", act);
  return YX_OK;
}

int bn_act_train_fwd_launch(const void* x, int dtype, int nhwc, int n, int c, int hw, const float* gamma, const float* beta, float eps,
                            float momentum, float* running_mean, float* running_var, long long* nbt, int act, void* y, float* save_mean,
                            float* save_invstd, void* ws, long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(x && gamma && beta && y && save_mean && save_invstd && ws, YX_ERR_INVALID_ARG, "bn_act_fwd: null pointer");
  int rc = bn_check(dtype, n, c, hw, act);
  if (rc) return rc;
  YX_REQUIRE(bn_act_ws_bytes(n, c, hw) <= ws_bytes, YX_ERR_CAPACITY, "bn_act_fwd: workspace too small");
  float* part = reinterpret_cast<float*>(ws);
  if (nhwc) {
    YX_REQUIRE(c <= 2048, YX_ERR_UNSUPPORTED, "bn_act_fwd(channels_last): C = %d > 2048", c);
    YX_REQUIRE(c % 8 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0, YX_ERR_INVALID_ARG,
               "bn_act_fwd(channels_last): C %% 8 == 0 and 16-byte aligned tensors required");
    const long long M = (long long)n * hw;
    int rows = 0, rows2 = 0;
    const int S = bn_nhwc_slabs(M, 64, 4, &rows), S2 = bn_nhwc_slabs(M, 32, 6, &rows2);
#define YX_GO(T) launch_kernel(bn_reduce_nhwc_kernel<T, false, 4>, dim3(S), dim3(kBnThreads), 0, s, (const T*)x, nullptr, nullptr, nullptr, nullptr, nullptr, M, c, rows, act, part, (long long)c)
    if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
    launch_kernel(bn_finalize_kernel, dim3((c + 3) / 4), dim3(128), 0, s, part, c, S, (double)M, eps, momentum, running_mean, running_var, save_mean, save_invstd, 0, nbt, (float*)nullptr, (float*)nullptr);
#define YX_GO(T) launch_kernel(bn_apply_nhwc_kernel<T, false, 4>, dim3(S2), dim3(kBnThreads), 0, s, (const T*)x, nullptr, save_mean, save_invstd, gamma, beta, nullptr, nullptr, 0.0f, M, c, rows2, act, (T*)y, (long long)c)
    if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
    YX_CUDA(cudaGetLastError());
    return YX_OK;
  }
  const int chunks = (hw + kBnChunk - 1) / kBnChunk;
  const dim3 grid((unsigned)chunks, (unsigned)c, (unsigned)n);
#define YX_GO(T) launch_kernel(bn_reduce_kernel<T, false>, dim3(grid), dim3(kBnThreads), 0, s, (const T*)x, nullptr, nullptr, nullptr, nullptr, nullptr, c, hw, act, part)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  launch_kernel(bn_finalize_kernel, dim3((c + 3) / 4), dim3(128), 0, s, part, c, n * chunks, (double)n * hw, eps, momentum, running_mean, running_var,
                                                     save_mean, save_invstd, 0, nbt, (float*)nullptr, (float*)nullptr);
#define YX_GO(T) launch_kernel(bn_apply_kernel<T, false>, dim3(grid), dim3(kBnThreads), 0, s, (const T*)x, nullptr, save_mean, save_invstd, gamma, beta, nullptr, nullptr, 0.0f, c, hw, act, (T*)y)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int bn_act_train_bwd_launch(const void* x, const void* dy, int dtype, int nhwc, int n, int c, int hw, const float* gamma, const float* beta,
                            const float* save_mean, const float* save_invstd, int act, void* dx, float* dgamma, float* dbeta,
                            float* acc_dgamma, float* acc_dbeta, long long dy_ld, void* ws, long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(x && dy && gamma && beta && save_mean && save_invstd && dx && dgamma && dbeta && ws, YX_ERR_INVALID_ARG, "bn_act_bwd: null pointer");
  int rc = bn_check(dtype, n, c, hw, act);
  if (rc) return rc;
  YX_REQUIRE(bn_act_ws_bytes(n, c, hw) <= ws_bytes, YX_ERR_CAPACITY, "bn_act_bwd: workspace too small");
  float* part = reinterpret_cast<float*>(ws);
  if (nhwc) {
    YX_REQUIRE(c <= 2048, YX_ERR_UNSUPPORTED, "bn_act_bwd(channels_last): C = %d > 2048", c);
    YX_REQUIRE(c % 8 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)dy & 15) == 0 && ((uintptr_t)dx & 15) == 0, YX_ERR_INVALID_ARG,
               "bn_act_bwd(channels_last): C %% 8 == 0 and 16-byte aligned tensors required");
    if (dy_ld <= 0) dy_ld = c;
    YX_REQUIRE(dy_ld >= c && dy_ld % 8 == 0, YX_ERR_INVALID_ARG, "bn_act_bwd(channels_last): dy pixel stride %lld", dy_ld);
    const long long M = (long long)n * hw;
    int rows = 0, rows2 = 0;
    const int S = bn_nhwc_slabs(M, 64, 4, &rows), S2 = bn_nhwc_slabs(M, 32, 6, &rows2);
#define YX_GO(T) launch_kernel(bn_reduce_nhwc_kernel<T, true, 2>, dim3(S), dim3(kBnThreads), 0, s, (const T*)x, (const T*)dy, save_mean, save_invstd, gamma, beta, M, c, rows, act, part, dy_ld)
    if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
    launch_kernel(bn_finalize_kernel, dim3((c + 3) / 4), dim3(128), 0, s, part, c, S, (double)M, 0.0f, 0.0f, nullptr, nullptr, dbeta, dgamma, 1, (long long*)nullptr, acc_dbeta, acc_dgamma);
    const float inv_m = (float)(1.0 / (double)M);
#define YX_GO(T) launch_kernel(bn_apply_nhwc_kernel<T, true, 2>, dim3(S2), dim3(kBnThreads), 0, s, (const T*)x, (const T*)dy, save_mean, save_invstd, gamma, beta, dbeta, dgamma, inv_m, M, c, rows2, act, (T*)dx, dy_ld)
    if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
    YX_CUDA(cudaGetLastError());
    return YX_OK;
  }
  const int chunks = (hw + kBnChunk - 1) / kBnChunk;
  const dim3 grid((unsigned)chunks, (unsigned)c, (unsigned)n);
#define YX_GO(T) launch_kernel(bn_reduce_kernel<T, true>, dim3(grid), dim3(kBnThreads), 0, s, (const T*)x, (const T*)dy, save_mean, save_invstd, gamma, beta, c, hw, act, part)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  launch_kernel(bn_finalize_kernel, dim3((c + 3) / 4), dim3(128), 0, s, part, c, n * chunks, (double)n * hw, 0.0f, 0.0f, nullptr, nullptr, dbeta, dgamma, 1, (long long*)nullptr, acc_dbeta, acc_dgamma);
  const float inv_m = (float)(1.0 / ((double)n * hw));
#define YX_GO(T) launch_kernel(bn_apply_kernel<T, true>, dim3(grid), dim3(kBnThreads), 0, s, (const T*)x, (const T*)dy, save_mean, save_invstd, gamma, beta, dbeta, dgamma, inv_m, c, hw, act, (T*)dx)
  if (dtype == YX_FP32) YX_GO(float); else if (dtype == YX_BF16) YX_GO(__nv_bfloat16); else YX_GO(__half);
#undef YX_GO
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

// ------------------------------------------------------------------------------------------
// SPP max pools, backward (SPPBottleneck, network_blocks.py:120-142: cat[x, m5(x), m9(x), m13(x)]): the gradient of every
// pooled value goes to the FIRST maximum of its window in row-major order (torch's max_pool2d: `val > max` while scanning).
// One thread per (pixel, 8 channels) scans the 13x13 window once and tracks the first maximum of the three nested windows;
// the three gradients are added to dx32 (fp32, pre-loaded with the gradient of the identity segment) with atomics.
//   cat  : NHWC buffer whose channels [0, c) hold x (pixel stride ld)      dout : NHWC gradient of the 4c-channel cat
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void spp_bwd_kernel(const T* __restrict__ cat, long long ld, const T* __restrict__ dout, long long dld,
                               float* __restrict__ dx32, int batch, int h, int w, int c) {
  const int c8 = c >> 3;
  const long long total = (long long)batch * h * w * c8;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(e % c8);
    long long r = e / c8;
    const int x0 = (int)(r % w); r /= w;
    const int y0 = (int)(r % h);
    const int b = (int)(r / h);
    float best[3][8];
    int arg[3][8];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) { best[k][j] = -INFINITY; arg[k][j] = -1; }
    for (int dy = -6; dy <= 6; ++dy) {
      const int yy = y0 + dy;
      if (yy < 0 || yy >= h) continue;
      for (int dx = -6; dx <= 6; ++dx) {
        const int xx = x0 + dx;
        if (xx < 0 || xx >= w) continue;
        float v[8];
        Vec8<T>::load(cat + (((long long)b * h + yy) * w + xx) * ld + cc * 8, v);
        const int pos = yy * w + xx;
        const int rad = max(abs(dy), abs(dx));             // inside the 5x5 / 9x9 / 13x13 window when rad <= 2 / 4 / 6
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          if (rad <= 2 * k + 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (v[j] > best[k][j] || arg[k][j] < 0) { best[k][j] = v[j]; arg[k][j] = pos; }
          }
        }
      }
    }
    const long long pix = ((long long)b * h + y0) * w + x0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float g[8];
      Vec8<T>::load(dout + pix * dld + (long long)(k + 1) * c + cc * 8, g);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (g[j] != 0.0f) atomicAdd(dx32 + ((long long)b * h * w + arg[k][j]) * c + cc * 8 + j, g[j]);
    }
  }
}

int spp_bwd_launch(const void* cat, long long ld, const void* dout, long long dld, float* dx32, int batch, int h, int w, int c,
                   int dtype, cudaStream_t s) {
  YX_REQUIRE(cat && dout && dx32, YX_ERR_INVALID_ARG, "spp_bwd: null pointer");
  YX_REQUIRE(c % 8 == 0 && ld >= c && dld >= 4LL * c && ld % 8 == 0 && dld % 8 == 0 && batch > 0 && h > 0 && w > 0, YX_ERR_INVALID_ARG, "spp_bwd: shape");
  YX_REQUIRE(((uintptr_t)cat & 15) == 0 && ((uintptr_t)dout & 15) == 0, YX_ERR_INVALID_ARG, "spp_bwd: 16-byte alignment");
  const long long total = (long long)batch * h * w * (c / 8);
  const int grid = (int)((total + 127) / 128 < 16384 ? (total + 127) / 128 : 16384);
  if (dtype == YX_BF16) spp_bwd_kernel<__nv_bfloat16><<<grid, 128, 0, s>>>((const __nv_bfloat16*)cat, ld, (const __nv_bfloat16*)dout, dld, dx32, batch, h, w, c);
  else if (dtype == YX_FP16) spp_bwd_kernel<__half><<<grid, 128, 0, s>>>((const __half*)cat, ld, (const __half*)dout, dld, dx32, batch, h, w, c);
  else if (dtype == YX_FP32) spp_bwd_kernel<float><<<grid, 128, 0, s>>>((const float*)cat, ld, (const float*)dout, dld, dx32, batch, h, w, c);
  else YX_REQUIRE(false, YX_ERR_INVALID_ARG, "spp_bwd: dtype %d", dtype);
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

}  // namespace yx
