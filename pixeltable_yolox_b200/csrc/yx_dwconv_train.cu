// Depthwise 3x3 convolution of the training step (pad 1, no bias, stride 1 or 2): forward, input gradient and weight
// gradient. Replaces what torch autograd / cuDNN computes for the depthwise BaseConv of DWConv
// (yolox/models/network_blocks.py:55-74) inside the training step of the depthwise configs (yolox_nano).
//
//   forward  y[b, p, c]  = sum_t  x[b, p*s + t - 1, c] * w16[c, t]
//   dgrad    dx[b, q, c] = sum_t  dy[b, (q + 1 - t) / s, c] * w16[c, t]      over the taps where the division is exact
//   wgrad    dW[c, t]    = sum_{b, p} dy[b, p, c] * x[b, p*s + t - 1, c]
//
// (t runs over the rows and the columns of the 3x3 window independently.) A depthwise conv has no GEMM structure worth the
// tensor cores: every layer is bound by HBM or by latency, so these are SIMT kernels on 16-byte channel vectors.
//
// The weight is read from the fp32 master parameter through its own strides and rounded to the 16-bit compute dtype in
// registers, which is what autocast's weight cast does: no packing launch, and forward and dgrad use the same rounded
// weight. Accumulation is fp32 everywhere. The weight gradient splits the pixels over CTAs, reduces inside a CTA in a fixed
// order and writes per-split partials; a second launch sums them in split order. No atomics: every result is deterministic.
//
// CTA shape (all three kernels): x = channel groups of 8 (a power of two, at most 32, i.e. 256 channels per CTA; grid.y
// covers the rest), y = pixel lanes, 256 threads.
#include "yx_common.cuh"

namespace yx {

static constexpr int kDwThreads = 256;
static constexpr int kDwChunk = 256;              // channels per CTA (32 groups of 8)

static inline void dw_block(int c, int* gx, int* gy, int* chunks) {
  const int groups = c / 8 < kDwChunk / 8 ? c / 8 : kDwChunk / 8;
  int x = 1;
  while (x < groups) x *= 2;
  *gx = x;
  *gy = kDwThreads / x;
  *chunks = (c + kDwChunk - 1) / kDwChunk;
}

template <typename T>
__device__ __forceinline__ void dw_load8(const T* p, float (&v)[8]) {
  constexpr bool fp16 = std::is_same<T, __half>::value;
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  unpack16(u.x, fp16, v[0], v[1]);
  unpack16(u.y, fp16, v[2], v[3]);
  unpack16(u.z, fp16, v[4], v[5]);
  unpack16(u.w, fp16, v[6], v[7]);
}

// Forward (DGRAD = false: src = x, dst = y) and input gradient (DGRAD = true: src = dy, dst = dx). One thread = one dst
// pixel x 8 channels; the CTA's 9 x 256 weights are rounded into shared memory once.
template <typename T, bool DGRAD>
__global__ void __launch_bounds__(kDwThreads)
dw_gather_kernel(const T* __restrict__ src, long long src_ld, int sh, int sw, const float* __restrict__ w, long long w_sc,
                 long long w_st, T* __restrict__ dst, long long dst_ld, int dh, int dwd, long long npix, int c, int stride) {
  constexpr bool fp16 = std::is_same<T, __half>::value;
  __shared__ __align__(16) float s_w[9][kDwChunk];
  const int c0 = blockIdx.y * kDwChunk;
  const int cc = c - c0 < kDwChunk ? c - c0 : kDwChunk;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  for (int e = tid; e < 9 * cc; e += kDwThreads) {
    const int t = e / cc, k = e - t * cc;
    s_w[t][k] = Cvt<T>::to_f(Cvt<T>::from_f(w[(long long)(c0 + k) * w_sc + (long long)t * w_st]));
  }
  __syncthreads();
  const int g = threadIdx.x * 8;
  const long long p = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  if (g >= cc || p >= npix) return;
  const int px = (int)(p % dwd);
  const long long r = p / dwd;
  const int py = (int)(r % dh);
  const long long b = r / dh;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    int sy;
    if (DGRAD) {
      const int n = py + 1 - i;                   // >= -1; stride 2: only the even n reach an output row
      if (n & (stride - 1)) continue;
      sy = n / stride;
    } else {
      sy = py * stride + i - 1;
    }
    if (sy < 0 || sy >= sh) continue;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      int sx;
      if (DGRAD) {
        const int n = px + 1 - j;
        if (n & (stride - 1)) continue;
        sx = n / stride;
      } else {
        sx = px * stride + j - 1;
      }
      if (sx < 0 || sx >= sw) continue;
      float v[8];
      dw_load8(src + ((b * sh + sy) * sw + sx) * src_ld + c0 + g, v);
      const float4 w0 = *reinterpret_cast<const float4*>(&s_w[3 * i + j][g]);
      const float4 w1 = *reinterpret_cast<const float4*>(&s_w[3 * i + j][g + 4]);
      acc[0] = fmaf(v[0], w0.x, acc[0]); acc[1] = fmaf(v[1], w0.y, acc[1]);
      acc[2] = fmaf(v[2], w0.z, acc[2]); acc[3] = fmaf(v[3], w0.w, acc[3]);
      acc[4] = fmaf(v[4], w1.x, acc[4]); acc[5] = fmaf(v[5], w1.y, acc[5]);
      acc[6] = fmaf(v[6], w1.z, acc[6]); acc[7] = fmaf(v[7], w1.w, acc[7]);
    }
  }
  uint4 o;
  o.x = pack16(acc[0], acc[1], fp16); o.y = pack16(acc[2], acc[3], fp16);
  o.z = pack16(acc[4], acc[5], fp16); o.w = pack16(acc[6], acc[7], fp16);
  *reinterpret_cast<uint4*>(dst + ((b * dh + py) * dwd + px) * dst_ld + c0 + g) = o;
}

// Weight gradient, pass 1: CTA (split, channel chunk) sums its range of output pixels into partial[split][9][c]. Each
// thread keeps 9 x 8 fp32 sums for its pixel lane; the lanes are reduced by an xor butterfly inside the warp and then warp
// by warp in order through shared memory, one tap at a time.
template <typename T>
__global__ void __launch_bounds__(kDwThreads)
dw_wgrad_kernel(const T* __restrict__ x, long long x_ld, int in_h, int in_w, const T* __restrict__ dy, long long dy_ld,
                int oh, int ow, long long npix, long long pix_per_split, int c, int stride, float* __restrict__ partial) {
  __shared__ __align__(16) float s_red[kDwThreads / 32][kDwChunk];
  const int c0 = blockIdx.y * kDwChunk;
  const int cc = c - c0 < kDwChunk ? c - c0 : kDwChunk;
  const int g = threadIdx.x * 8;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[t][k] = 0.f;
  const long long p0 = (long long)blockIdx.x * pix_per_split;
  const long long p1 = p0 + pix_per_split < npix ? p0 + pix_per_split : npix;
  if (g < cc) {
    const bool idx32 = npix <= 0xffffffffLL;      // 32-bit division for the pixel coordinates (addresses stay 64-bit)
    for (long long p = p0 + threadIdx.y; p < p1; p += blockDim.y) {
      int ox, oy;
      long long b;
      if (idx32) {
        unsigned q = (unsigned)p;
        ox = (int)(q % (unsigned)ow); q /= (unsigned)ow;
        oy = (int)(q % (unsigned)oh); b = q / (unsigned)oh;
      } else {
        ox = (int)(p % ow);
        const long long r = p / ow;
        oy = (int)(r % oh); b = r / oh;
      }
      // all ten loads are issued before the first FMA: a lane walks its pixels one after another, so the loop is bound by
      // the loads' latency (zero vectors stand in for the taps outside the map)
      const uint4 dv = *reinterpret_cast<const uint4*>(dy + p * dy_ld + c0 + g);
      uint4 xv[9];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int iy = oy * stride + i - 1;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const int ix = ox * stride + j - 1;
          xv[3 * i + j] = (iy >= 0 && iy < in_h && ix >= 0 && ix < in_w)
                              ? *reinterpret_cast<const uint4*>(x + ((b * in_h + iy) * in_w + ix) * x_ld + c0 + g)
                              : make_uint4(0, 0, 0, 0);
        }
      }
      constexpr bool fp16 = std::is_same<T, __half>::value;
      float d[8];
      unpack16(dv.x, fp16, d[0], d[1]); unpack16(dv.y, fp16, d[2], d[3]);
      unpack16(dv.z, fp16, d[4], d[5]); unpack16(dv.w, fp16, d[6], d[7]);
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        float v[8];
        unpack16(xv[t].x, fp16, v[0], v[1]); unpack16(xv[t].y, fp16, v[2], v[3]);
        unpack16(xv[t].z, fp16, v[4], v[5]); unpack16(xv[t].w, fp16, v[6], v[7]);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[t][k] = fmaf(d[k], v[k], acc[t][k]);
      }
    }
  }
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
      for (int off = 16; off >= (int)blockDim.x; off >>= 1) acc[t][k] += __shfl_xor_sync(0xffffffffu, acc[t][k], off);
    if (lane < (int)blockDim.x && g < cc) {
      *reinterpret_cast<float4*>(&s_red[warp][g]) = make_float4(acc[t][0], acc[t][1], acc[t][2], acc[t][3]);
      *reinterpret_cast<float4*>(&s_red[warp][g + 4]) = make_float4(acc[t][4], acc[t][5], acc[t][6], acc[t][7]);
    }
    __syncthreads();
    for (int e = tid; e < cc; e += kDwThreads) {
      float s = 0.f;
      for (int wi = 0; wi < kDwThreads / 32; ++wi) s += s_red[wi][e];
      partial[((long long)blockIdx.x * 9 + t) * c + c0 + e] = s;
    }
    __syncthreads();
  }
}

// Weight gradient, pass 2: dW[c, t] (=|+=) sum of the splits in split order, at the parameter's strides
__global__ void dw_wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int c, float* __restrict__ dw, long long sc,
                                       long long st, int accumulate) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;      // t * c + channel
  if (e >= 9 * c) return;
  float acc = 0.f;
#pragma unroll 8
  for (int s = 0; s < splits; ++s) acc += partial[(long long)s * 9 * c + e];
  const int t = e / c, ch = e - t * c;
  float* d = dw + (long long)ch * sc + (long long)t * st;
  *d = accumulate ? *d + acc : acc;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int dw_check(const char* what, int dtype, int batch, int in_h, int in_w, int c, int stride) {
  YX_REQUIRE(dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_UNSUPPORTED, "%s: 16-bit activations only", what);
  YX_REQUIRE(batch > 0 && in_h > 0 && in_w > 0 && c > 0, YX_ERR_INVALID_ARG, "%s: empty tensor", what);
  YX_REQUIRE(c % 8 == 0, YX_ERR_INVALID_ARG, "%s: the channel count %d is not a multiple of 8", what, c);
  YX_REQUIRE(stride == 1 || stride == 2, YX_ERR_UNSUPPORTED, "%s: stride %d", what, stride);
  return YX_OK;
}

static int dw_check_act(const char* what, const char* name, const void* p, long long ld, int c) {
  YX_REQUIRE(p, YX_ERR_INVALID_ARG, "%s: %s is a null pointer", what, name);
  YX_REQUIRE(((uintptr_t)p & 15) == 0 && ld % 8 == 0 && ld >= c, YX_ERR_INVALID_ARG,
             "%s: %s must be 16-byte aligned with a pixel stride that is a multiple of 8 and >= c (ld %lld, c %d)", what, name,
             ld, c);
  return YX_OK;
}

// Pixel splits of the weight gradient: about two CTAs per SM over the channel chunks, but at least 4 pixels per lane and at
// most 128 splits (the second launch sums them serially). Depends on the shape and the device only, so the summation order
// (and the result) is the same on every call.
static void dw_wgrad_plan(int batch, int in_h, int in_w, int c, int stride, int* splits, long long* pix_per_split) {
  int gx, gy, chunks;
  dw_block(c, &gx, &gy, &chunks);
  const int oh = (in_h - 1) / stride + 1, ow = (in_w - 1) / stride + 1;
  const long long npix = (long long)batch * oh * ow;
  long long s = 2LL * num_sms() / chunks;
  const long long by_work = npix / (4LL * gy);
  if (s > by_work) s = by_work;
  if (s > 128) s = 128;
  if (s < 1) s = 1;
  *pix_per_split = (npix + s - 1) / s;
  *splits = (int)((npix + *pix_per_split - 1) / *pix_per_split);
}

long long dw_wgrad_ws_bytes(int batch, int in_h, int in_w, int c, int stride) {
  if (dw_check("dwconv3x3_wgrad", YX_BF16, batch, in_h, in_w, c, stride) != YX_OK) return -1;
  int splits;
  long long pps;
  dw_wgrad_plan(batch, in_h, in_w, c, stride, &splits, &pps);
  return (long long)splits * 9 * c * 4;
}

template <bool DGRAD>
static int dw_gather_launch(const char* what, const void* src, long long src_ld, int sh, int sw, const float* w, long long w_sc,
                            long long w_st, void* dst, long long dst_ld, int dh, int dwd, int batch, int c, int stride, int dtype,
                            cudaStream_t stream) {
  YX_REQUIRE(w, YX_ERR_INVALID_ARG, "%s: null weight", what);
  int gx, gy, chunks;
  dw_block(c, &gx, &gy, &chunks);
  const long long npix = (long long)batch * dh * dwd;
  const long long gridx = (npix + gy - 1) / gy;
  YX_REQUIRE(gridx < (1LL << 31), YX_ERR_UNSUPPORTED, "%s: %lld pixels", what, npix);
  const dim3 grid((unsigned)gridx, (unsigned)chunks), block(gx, gy);
  if (dtype == YX_BF16)
    YX_CUDA(launch_kernel(dw_gather_kernel<__nv_bfloat16, DGRAD>, grid, block, 0, stream, (const __nv_bfloat16*)src, src_ld, sh, sw,
                          w, w_sc, w_st, (__nv_bfloat16*)dst, dst_ld, dh, dwd, npix, c, stride));
  else
    YX_CUDA(launch_kernel(dw_gather_kernel<__half, DGRAD>, grid, block, 0, stream, (const __half*)src, src_ld, sh, sw, w, w_sc,
                          w_st, (__half*)dst, dst_ld, dh, dwd, npix, c, stride));
  return YX_OK;
}

int dw_train_fwd_launch(const void* x, long long x_ld, const float* w, long long w_sc, long long w_st, void* y, long long y_ld,
                        int batch, int in_h, int in_w, int c, int stride, int dtype, cudaStream_t stream) {
  const char* what = "dwconv3x3_train_fwd";
  int rc = dw_check(what, dtype, batch, in_h, in_w, c, stride);
  if (!rc) rc = dw_check_act(what, "x", x, x_ld, c);
  if (!rc) rc = dw_check_act(what, "y", y, y_ld, c);
  if (rc) return rc;
  const int oh = (in_h - 1) / stride + 1, ow = (in_w - 1) / stride + 1;
  return dw_gather_launch<false>(what, x, x_ld, in_h, in_w, w, w_sc, w_st, y, y_ld, oh, ow, batch, c, stride, dtype, stream);
}

int dw_dgrad_launch(const void* dy, long long dy_ld, const float* w, long long w_sc, long long w_st, void* dx, long long dx_ld,
                    int batch, int in_h, int in_w, int c, int stride, int dtype, cudaStream_t stream) {
  const char* what = "dwconv3x3_dgrad";
  int rc = dw_check(what, dtype, batch, in_h, in_w, c, stride);
  if (!rc) rc = dw_check_act(what, "dy", dy, dy_ld, c);
  if (!rc) rc = dw_check_act(what, "dx", dx, dx_ld, c);
  if (rc) return rc;
  const int oh = (in_h - 1) / stride + 1, ow = (in_w - 1) / stride + 1;
  return dw_gather_launch<true>(what, dy, dy_ld, oh, ow, w, w_sc, w_st, dx, dx_ld, in_h, in_w, batch, c, stride, dtype, stream);
}

int dw_wgrad_launch(const void* x, long long x_ld, const void* dy, long long dy_ld, int dtype, int batch, int in_h, int in_w, int c,
                    int stride, float* dw, long long dw_sc, long long dw_st, int accumulate, void* ws, long long ws_bytes,
                    cudaStream_t stream) {
  const char* what = "dwconv3x3_wgrad";
  int rc = dw_check(what, dtype, batch, in_h, in_w, c, stride);
  if (!rc) rc = dw_check_act(what, "x", x, x_ld, c);
  if (!rc) rc = dw_check_act(what, "dy", dy, dy_ld, c);
  if (rc) return rc;
  YX_REQUIRE(dw && ws, YX_ERR_INVALID_ARG, "%s: null dw or workspace", what);
  int gx, gy, chunks, splits;
  long long pps;
  dw_block(c, &gx, &gy, &chunks);
  dw_wgrad_plan(batch, in_h, in_w, c, stride, &splits, &pps);
  const long long need = (long long)splits * 9 * c * 4;
  YX_REQUIRE(need <= ws_bytes, YX_ERR_CAPACITY, "%s: workspace of %lld bytes, need %lld", what, ws_bytes, need);
  const int oh = (in_h - 1) / stride + 1, ow = (in_w - 1) / stride + 1;
  const long long npix = (long long)batch * oh * ow;
  float* partial = reinterpret_cast<float*>(ws);
  const dim3 grid((unsigned)splits, (unsigned)chunks), block(gx, gy);
  if (dtype == YX_BF16)
    YX_CUDA(launch_kernel(dw_wgrad_kernel<__nv_bfloat16>, grid, block, 0, stream, (const __nv_bfloat16*)x, x_ld, in_h, in_w,
                          (const __nv_bfloat16*)dy, dy_ld, oh, ow, npix, pps, c, stride, partial));
  else
    YX_CUDA(launch_kernel(dw_wgrad_kernel<__half>, grid, block, 0, stream, (const __half*)x, x_ld, in_h, in_w, (const __half*)dy,
                          dy_ld, oh, ow, npix, pps, c, stride, partial));
  YX_CUDA(launch_kernel(dw_wgrad_reduce_kernel, dim3((9 * c + 255) / 256), dim3(256), 0, stream, (const float*)partial, splits, c,
                        dw, dw_sc, dw_st, accumulate));
  return YX_OK;
}

}  // namespace yx
