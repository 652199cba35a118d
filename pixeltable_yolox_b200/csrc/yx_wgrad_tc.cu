// Weight gradient of a dense conv on the tensor cores (tcgen05 / TMEM / TMA), plus the two small helpers the
// training conv stack needs around the forward kernel (weight packing for fprop + dgrad, zero-stuffing for the
// stride-2 dgrad).
//
// Replaces what torch autograd / cuDNN computes for BaseConv.conv and the prediction convs in the training step
// (yolox/core/trainer.py:96-129 -> loss.backward(); modules: yolox/models/network_blocks.py:27-52,
// yolox/models/yolo_head.py:94-120).
//
//   dW[o][t][i] = sum over output pixels p = (n, oy, ox) of  dy[p][o] * x[n, oy*s + r - pad, ox*s + q - pad][i],   t = 3*r + q
//
// GEMM view (per filter tap t and input-channel tile):  D[M = o, N = i] += A[K = pixels, M]^T * B_t[K = pixels, N].
// Both activations are NHWC, i.e. the channel (M / N) index is the contiguous one: both operands are "MN-major" UMMA
// operands. A TMA tiled load of box {c <= 64 channels, tw, th, 1} lands [tw*th pixel rows] x [c channels] with the
// hardware swizzle, which IS the canonical MN-major layout (rows of K at `row_bytes`, 8-row atoms at SBO = 8 * row_bytes,
// blocks of 64 / 32 / 16 channels at LBO = one TMA box). The tap shift and the conv's zero padding are TMA coordinates +
// out-of-bounds zero fill of the x load; stride 2 is elementStrides = 2. Nothing is transposed or materialised.
//
// Work decomposition: unit = (128-row tile of out channels, group of <= 512 / N accumulator slices, range of pixel tiles).
// A slice is one (input-channel tile of N <= 128, tap) pair = N TMEM columns; the pixel dimension (the GEMM's K) is split
// across CTAs so that a layer fills the 148 SMs; every CTA writes its fp32 partial [128][slices][N] and a second kernel
// sums the partials in a fixed order (deterministic, unlike atomics) into the gradient tensor with the weight's strides.
//
// One CTA = 6 warps: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2..5 epilogue (tcgen05.ld -> global).
#include <string.h>

#include "yx_common.cuh"

namespace yx {

static constexpr int kWgStages = 4;

struct WgradParams {
  int tw, th, tiles_w, tiles_h, batch;
  int KP, ksteps;                 // pixels per stage (multiple of 16), KP / 16
  int stride, pad, taps, ksize;
  int N, Ncol, n_tiles, n_blocks, ci_box;
  int co_box, m_blocks, m_tiles, out_c;
  int SG, n_groups, slices;       // slices = n_tiles * taps; SG slices per CTA
  int merged;                     // 1: the CTA's slices are ONE MMA operand of N = nsl * N columns (single-box slices)
  int ksplit, tiles_per_split, PT;
  int stages;
  unsigned rb_a, rb_b;            // bytes per pixel row of one A / B box
  unsigned a_block_bytes, b_block_bytes, a_bytes, stage_bytes;
  unsigned desc_hi_a, desc_hi_b, lbo_a16, lbo_b16, idesc;
  float* partial;
  long long split_stride, row_stride;   // elements
};

struct __align__(8) WgShared {
  uint64_t full[kWgStages];
  uint64_t empty[kWgStages];
  uint64_t tmem_full;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint64_t wg_desc(uint32_t addr, uint32_t lbo16, uint32_t hi) {
  return (uint64_t)(((addr & 0x3FFFFu) >> 4) | ((lbo16 & 0x3FFFu) << 16)) | ((uint64_t)hi << 32);
}

__global__ void __launch_bounds__(192, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x, const WgradParams p) {
  extern __shared__ uint8_t wg_smem_raw[];
  __shared__ WgShared sh;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(wg_smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int bid = (int)blockIdx.x;
  const int split = bid % p.ksplit;
  const int unit = bid / p.ksplit;
  const int group = unit % p.n_groups;
  const int m_tile = unit / p.n_groups;
  const int s0 = group * p.SG;
  const int nsl = min(p.SG, p.slices - s0);
  const int t0 = split * p.tiles_per_split;
  const int t1 = min(t0 + p.tiles_per_split, p.PT);
  const int m_real = min(p.m_blocks, (p.out_c - m_tile * 128 + p.co_box - 1) / p.co_box);

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&sh.full[s], 1); mbar_init(&sh.empty[s], 1); }
    mbar_init(&sh.tmem_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_dy);
    tma_prefetch_desc(&map_x);
  }
  if (warp == 1) { tmem_alloc(&sh.tmem_base, 512); tmem_relinquish(); }
  // rows of the M tile beyond out_c: their operand blocks are never loaded, they stay zero
  if (m_real < p.m_blocks) {
    const unsigned nz = (unsigned)(p.m_blocks - m_real) * p.a_block_bytes;
    for (int s = 0; s < p.stages; ++s) {
      uint4* z = reinterpret_cast<uint4*>(smem + (size_t)s * p.stage_bytes + (size_t)m_real * p.a_block_bytes);
      for (unsigned k = threadIdx.x; k < nz / 16; k += blockDim.x) z[k] = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  // programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch) overlapped the predecessor's tail;
  // from here on the kernel reads x / dy and (much later) overwrites the partial buffer the previous reduction read
  pdl_wait();
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sh.tmem_base;

  if (warp == 0) {
    if (elect_one_sync()) {
      const int tpi = p.tiles_w * p.tiles_h;
      const uint32_t tx = (uint32_t)m_real * p.a_block_bytes + (uint32_t)(nsl * p.n_blocks) * p.b_block_bytes;
      int it = 0;
      for (int pt = t0; pt < t1; ++pt, ++it) {
        const int s = it % p.stages;
        if (it >= p.stages) mbar_wait(&sh.empty[s], (uint32_t)((it / p.stages) - 1) & 1u);
        const int n = pt / tpi, rem = pt - n * tpi;
        const int ty = rem / p.tiles_w, txi = rem - ty * p.tiles_w;
        const int ox0 = txi * p.tw, oy0 = ty * p.th;
        uint8_t* st = smem + (size_t)s * p.stage_bytes;
        mbar_arrive_expect_tx(&sh.full[s], tx);
        for (int mb = 0; mb < m_real; ++mb)
          tma_load_4d(&map_dy, &sh.full[s], st + (size_t)mb * p.a_block_bytes, m_tile * 128 + mb * p.co_box, ox0, oy0, n);
        uint8_t* bst = st + p.a_bytes;
        for (int j = 0; j < nsl; ++j) {
          const int sl = s0 + j;
          const int n_tile = sl / p.taps, tap = sl - n_tile * p.taps;
          const int r = tap / p.ksize, q = tap - r * p.ksize;
          for (int nb = 0; nb < p.n_blocks; ++nb)
            tma_load_4d(&map_x, &sh.full[s], bst + (size_t)(j * p.n_blocks + nb) * p.b_block_bytes,
                        n_tile * p.N + nb * p.ci_box, ox0 * p.stride + q - p.pad, oy0 * p.stride + r - p.pad, n);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      int it = 0;
      for (int pt = t0; pt < t1; ++pt, ++it) {
        const int s = it % p.stages;
        mbar_wait(&sh.full[s], (uint32_t)(it / p.stages) & 1u);
        tc_fence_after();
        const uint32_t a0 = smem_u32(smem + (size_t)s * p.stage_bytes);
        const uint32_t b0 = a0 + p.a_bytes;
        if (p.merged) {
          // single-box slices (N = 16 / 32 / 64) lie back to back in the stage: together they are one MN-major operand of
          // nsl * N columns whose 16 / 32 / 64-channel blocks are LBO = one box apart -- one MMA per K step instead of nsl
          // (the stem's nine N = 16 taps: 9 x fewer, 9 x wider instructions; measured: no change in time, 125 vs 127 us -- that
          // layer is bound by the TMA's per-row rate on 32-byte pixel rows, 1 280 rows per 128-pixel tile, not by MMA issue)
          const uint32_t idesc = (p.idesc & ~(0x3Fu << 17)) | ((uint32_t)((nsl * p.N) >> 3) << 17);
          for (int ks = 0; ks < p.ksteps; ++ks) {
            const uint64_t ad = wg_desc(a0 + (uint32_t)ks * 16u * p.rb_a, p.lbo_a16, p.desc_hi_a);
            const uint64_t bd = wg_desc(b0 + (uint32_t)ks * 16u * p.rb_b, p.lbo_b16, p.desc_hi_b);
            umma_f16(tmem, ad, bd, idesc, (it | ks) ? 1u : 0u);
          }
        } else {
          for (int j = 0; j < nsl; ++j) {
            const uint32_t bj = b0 + (uint32_t)(j * p.n_blocks) * p.b_block_bytes;
            const uint32_t d = tmem + (uint32_t)(j * p.Ncol);
            for (int ks = 0; ks < p.ksteps; ++ks) {
              const uint64_t ad = wg_desc(a0 + (uint32_t)ks * 16u * p.rb_a, p.lbo_a16, p.desc_hi_a);
              const uint64_t bd = wg_desc(bj + (uint32_t)ks * 16u * p.rb_b, p.lbo_b16, p.desc_hi_b);
              umma_f16(d, ad, bd, p.idesc, (it | ks) ? 1u : 0u);
            }
          }
        }
        umma_commit(&sh.empty[s]);      // the slot is free once these MMAs have read it
      }
      umma_commit(&sh.tmem_full);
    }
  } else {
    const int q = warp & 3;             // TMEM lane quarter this warp may read
    mbar_wait(&sh.tmem_full, 0);
    tc_fence_after();
    const int o = m_tile * 128 + q * 32 + lane;
    float* dst = p.partial + (long long)split * p.split_stride + (long long)o * p.row_stride + (long long)s0 * p.N;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const int nchunks = p.N >> 4;
    for (int j = 0; j < nsl; ++j) {
      for (int c = 0; c < nchunks; ++c) {
        uint32_t v[16];
        tmem_ld_x16(tl + (uint32_t)(j * (p.merged ? p.N : p.Ncol) + c * 16), v);
        tmem_ld_wait();
        if (o < p.out_c) {
          float4* d4 = reinterpret_cast<float4*>(dst + j * p.N + c * 16);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            d4[k] = make_float4(__uint_as_float(v[4 * k]), __uint_as_float(v[4 * k + 1]), __uint_as_float(v[4 * k + 2]),
                                __uint_as_float(v[4 * k + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// sum of the per-split partials in split order -> dW with the weight tensor's own strides (fp32)
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, int ksplit, long long split_stride, long long row_stride,
                                    int N, int taps, int out_c, int in_c, int out_c_real, int in_c_real, float* __restrict__ dw,
                                    long long so, long long si, long long st, int accumulate) {
  pdl_wait();
  pdl_launch_dependents();
  const long long total = (long long)out_c * taps * in_c;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e % in_c);
    const long long ot = e / in_c;
    const int t = (int)(ot % taps);
    const int o = (int)(ot / taps);
    if (o >= out_c_real || i >= in_c_real) continue;
    const int n_tile = i / N, n = i - n_tile * N;
    const float* src = partial + (long long)o * row_stride + (long long)(n_tile * taps + t) * N + n;
    float acc = 0.f;
    for (int sp = 0; sp < ksplit; ++sp) acc += src[(long long)sp * split_stride];
    float* d = dw + (long long)o * so + (long long)i * si + (long long)t * st;
    *d = accumulate ? *d + acc : acc;
  }
}

// index of weight element (oo, tap = 3r + s, ii) in the dgrad operand.
//   rotated form  [i_pad][taps][o_pad]: tap reversed.
//   sub-pixel form [4 * i_pad][9][o_pad] (3x3 stride 2, pad 1): dx[2a + pa] = sum_oy dy[oy] W[r] with 2 oy - 1 + r = 2a + pa, i.e.
//   pa = 0: r = 1 reads dy[a]; pa = 1: r = 2 reads dy[a], r = 0 reads dy[a + 1]. As a pad-1 3x3 conv over dy (tap r' reads
//   dy[a + r' - 1]): r = 1 -> (pa 0, r' 1), r = 2 -> (pa 1, r' 1), r = 0 -> (pa 1, r' 2); same for columns.
__device__ __forceinline__ long long dgrad_index(int oo, int tp, int ii, int taps, int o_pad, int i_pad, int subpixel) {
  if (!subpixel) return ((long long)ii * taps + (taps - 1 - tp)) * o_pad + oo;
  const int r = tp / 3, s = tp - 3 * r;
  const int pa = r == 1 ? 0 : 1, rr = r == 0 ? 2 : 1;
  const int pb = s == 1 ? 0 : 1, ss = s == 0 ? 2 : 1;
  return ((long long)((pa * 2 + pb) * i_pad + ii) * 9 + (rr * 3 + ss)) * o_pad + oo;
}

// fp32 conv weight (any strides) -> 16-bit packed operands of yx_conv_bn_act_fwd:
//   wf [o_pad][taps][i_pad]                 forward:  y = conv(x, W)
//   wd [i_pad][taps][o_pad], tap reversed   dgrad:    dx = conv(dy or its zero-stuffed copy, W rotated by 180 degrees, o <-> i)
template <typename T>
__global__ void pack_train_weights_kernel(const float* __restrict__ w, long long so, long long si, long long st, int o, int i,
                                          int taps, int o_pad, int i_pad, T* __restrict__ wf, T* __restrict__ wd, int subpixel) {
  pdl_wait();
  pdl_launch_dependents();
  const long long total = (long long)o_pad * taps * i_pad;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int ii = (int)(e % i_pad);
    const long long ot = e / i_pad;
    const int t = (int)(ot % taps);
    const int oo = (int)(ot / taps);
    const float v = (oo < o && ii < i) ? w[(long long)oo * so + (long long)ii * si + (long long)t * st] : 0.f;
    const T h = Cvt<T>::from_f(v);
    if (wf) wf[e] = h;
    if (wd) wd[dgrad_index(oo, t, ii, taps, o_pad, i_pad, subpixel)] = h;
  }
}

// every conv weight of the model in ONE launch (83 launches of ~4 us each otherwise): table rows (int64 x 12) =
// src ptr | stride_o | stride_i | stride_tap | o | i | taps | o_pad | i_pad | wf ptr | wd ptr | subpixel; chunks rows = (tensor, first
// element of the [o_pad][taps][i_pad] index space); one CTA per chunk of chunk_elems elements.
template <typename T>
__global__ void pack_train_weights_multi_kernel(const long long* __restrict__ table, const int* __restrict__ chunks, int chunk_elems) {
  const int t = chunks[2 * blockIdx.x];
  const long long e0 = chunks[2 * blockIdx.x + 1];
  const long long* r = table + (long long)t * 12;
  const int subpixel = (int)r[11];
  const float* w = reinterpret_cast<const float*>(r[0]);
  const long long so = r[1], si = r[2], st = r[3];
  const int o = (int)r[4], i = (int)r[5], taps = (int)r[6], o_pad = (int)r[7], i_pad = (int)r[8];
  T* wf = reinterpret_cast<T*>(r[9]);
  T* wd = reinterpret_cast<T*>(r[10]);
  const long long total = (long long)o_pad * taps * i_pad;
  const long long e1 = e0 + chunk_elems < total ? e0 + chunk_elems : total;
  for (long long e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const int ii = (int)(e % i_pad);
    const long long ot = e / i_pad;
    const int tp = (int)(ot % taps);
    const int oo = (int)(ot / taps);
    const float v = (oo < o && ii < i) ? w[(long long)oo * so + (long long)ii * si + (long long)tp * st] : 0.f;
    const T h = Cvt<T>::from_f(v);
    if (wf) wf[e] = h;
    if (wd) wd[dgrad_index(oo, tp, ii, taps, o_pad, i_pad, subpixel)] = h;
  }
}

// z[b, 2*oy, 2*ox, :] = dy[b, oy, ox, :], every other pixel of z [b, zh, zw, c] zero (16-byte vectors)
__global__ void dilate2_kernel(const uint4* __restrict__ dy, uint4* __restrict__ z, int batch, int oh, int ow, int zh, int zw, int c8) {
  pdl_wait();
  pdl_launch_dependents();
  const long long total = (long long)batch * zh * zw * c8;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(e % c8);
    long long r = e / c8;
    const int x = (int)(r % zw); r /= zw;
    const int y = (int)(r % zh);
    const int b = (int)(r / zh);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (!(x & 1) && !(y & 1) && (y >> 1) < oh && (x >> 1) < ow) v = dy[(((long long)b * oh + (y >> 1)) * ow + (x >> 1)) * c8 + c];
    z[e] = v;
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int box_channels(int c) { return c % 64 == 0 ? 64 : (c % 32 == 0 ? 32 : 16); }

static int wgrad_plan(int batch, int in_h, int in_w, int in_c, int out_h, int out_w, int out_c, int ksize, int stride,
                      WgradParams* pp, size_t* smem_out) {
  YX_REQUIRE(batch > 0 && in_h > 0 && in_w > 0 && out_h > 0 && out_w > 0, YX_ERR_INVALID_ARG, "wgrad: empty tensor");
  YX_REQUIRE((ksize == 1 || ksize == 3) && (stride == 1 || stride == 2), YX_ERR_UNSUPPORTED, "wgrad: ksize %d stride %d", ksize, stride);
  YX_REQUIRE(in_c % 16 == 0 && out_c % 16 == 0 && in_c > 0 && out_c > 0, YX_ERR_INVALID_ARG,
             "wgrad: channel counts must be multiples of 16 (in %d, out %d); pad them", in_c, out_c);
  const int pad = (ksize - 1) / 2;
  YX_REQUIRE(out_h == (in_h + 2 * pad - ksize) / stride + 1 && out_w == (in_w + 2 * pad - ksize) / stride + 1, YX_ERR_INVALID_ARG,
             "wgrad: output size %dx%d does not follow from input %dx%d", out_h, out_w, in_h, in_w);
  WgradParams& p = *pp;
  memset(&p, 0, sizeof(p));
  p.batch = batch; p.stride = stride; p.pad = pad; p.ksize = ksize; p.taps = ksize * ksize; p.out_c = out_c;
  p.ci_box = box_channels(in_c);
  p.co_box = box_channels(out_c);
  p.rb_a = 2u * (unsigned)p.co_box; p.rb_b = 2u * (unsigned)p.ci_box;
  p.m_blocks = 128 / p.co_box;
  p.m_tiles = (out_c + 127) / 128;
  // N: the largest divisor of in_c that is a multiple of the box and <= 128
  p.N = p.ci_box;
  for (int n = p.ci_box; n <= 128 && n <= in_c; n += p.ci_box) if (in_c % n == 0) p.N = n;
  p.n_tiles = in_c / p.N;
  p.n_blocks = p.N / p.ci_box;
  p.Ncol = (p.N + 31) & ~31;
  p.slices = p.n_tiles * p.taps;
  // slices per CTA: measured on the yolox_s layers by sweeping it, about 128 accumulator columns per CTA is best
  // (N = 128: one slice, 36.6 -> 20.8 us for 256->256 3x3 @20x20; N = 64: two; N = 32: four): more CTAs on the (o, i, tap)
  // space and a shorter epilogue per CTA beat the saved re-loads of the dy tile; N = 16 keeps all nine taps together
  int sg_max = p.N <= 16 ? 512 / p.Ncol : (128 / p.N > 1 ? 128 / p.N : 1);
  if (sg_max > p.slices) sg_max = p.slices;
  p.n_groups = (p.slices + sg_max - 1) / sg_max;
  p.SG = (p.slices + p.n_groups - 1) / p.n_groups;
  p.n_groups = (p.slices + p.SG - 1) / p.SG;
  p.merged = (p.n_blocks == 1 && p.SG > 1 && p.SG * p.N <= 256) ? 1 : 0;

  const int budget = max_smem_optin() - 4096;                   // 1 KB alignment slack + static shared (barriers)
  const unsigned bpp = 256u + (unsigned)(p.SG * p.N) * 2u;   // bytes per pixel of one stage: 128 A channels + SG * N B channels
  int kp_max = (budget / 3) / (int)bpp / 16 * 16;
  if (kp_max > 128) kp_max = 128;
  if (kp_max < 16) kp_max = 16;
  long long best = -1;
  for (int tw = 1; tw <= 128; ++tw) {
    if (tw * stride > 256) break;
    for (int th = 1; tw * th <= kp_max; ++th) {
      if (th * stride > 256) break;
      const int kp = tw * th;
      if (kp % 16) continue;
      const long long tiles = ceil_div64(out_w, tw) * ceil_div64(out_h, th);
      const long long cost = tiles * (kp + 24);
      if (best < 0 || cost < best) { best = cost; p.tw = tw; p.th = th; }
    }
  }
  YX_REQUIRE(best >= 0, YX_ERR_UNSUPPORTED, "wgrad: no pixel tile fits");
  p.KP = p.tw * p.th; p.ksteps = p.KP / 16;
  p.tiles_w = (int)ceil_div64(out_w, p.tw); p.tiles_h = (int)ceil_div64(out_h, p.th);
  p.PT = batch * p.tiles_w * p.tiles_h;
  p.a_block_bytes = (unsigned)p.KP * p.rb_a;
  p.b_block_bytes = (unsigned)p.KP * p.rb_b;
  p.a_bytes = (unsigned)p.m_blocks * p.a_block_bytes;
  p.stage_bytes = (p.a_bytes + (unsigned)(p.SG * p.n_blocks) * p.b_block_bytes + 1023u) & ~1023u;
  p.stages = budget / (int)p.stage_bytes;
  if (p.stages > kWgStages) p.stages = kWgStages;
  YX_REQUIRE(p.stages >= 1, YX_ERR_UNSUPPORTED, "wgrad: a stage of %u bytes does not fit shared memory", p.stage_bytes);
  *smem_out = (size_t)p.stages * p.stage_bytes + 1024;

  const int units = p.m_tiles * p.n_groups;
  int ks = num_sms() / units;
  if (ks < 1) ks = 1;
  if (ks > p.PT) ks = p.PT;
  if (p.PT >= 8 && ks > p.PT / 4) ks = p.PT / 4;          // at least four pixel tiles per CTA: the pipeline needs something to overlap
  p.tiles_per_split = (p.PT + ks - 1) / ks;
  p.ksplit = (p.PT + p.tiles_per_split - 1) / p.tiles_per_split;
  p.row_stride = (long long)p.slices * p.N;
  p.split_stride = (long long)p.m_tiles * 128 * p.row_stride;
  return YX_OK;
}

long long wgrad_ws_bytes(int batch, int in_h, int in_w, int in_c, int out_h, int out_w, int out_c, int ksize, int stride) {
  WgradParams p; size_t smem = 0;
  if (wgrad_plan(batch, in_h, in_w, in_c, out_h, out_w, out_c, ksize, stride, &p, &smem) != YX_OK) return -1;
  return (long long)p.ksplit * p.split_stride * 4;
}

int wgrad_launch(const void* x, long long x_ld, const void* dy, long long dy_ld, int dtype, int batch, int in_h, int in_w, int in_c,
                 int out_h, int out_w, int out_c, int ksize, int stride, int in_c_real, int out_c_real, float* dw, long long dw_so,
                 long long dw_si, long long dw_st, int accumulate, void* ws, long long ws_bytes, cudaStream_t stream) {
  YX_REQUIRE(dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_UNSUPPORTED, "wgrad: 16-bit activations only");
  YX_REQUIRE(x && dy && dw && ws, YX_ERR_INVALID_ARG, "wgrad: null pointer");
  YX_REQUIRE(x_ld % 8 == 0 && dy_ld % 8 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)dy & 15) == 0, YX_ERR_INVALID_ARG,
             "wgrad: activations must be 16-byte aligned with a pixel stride that is a multiple of 8");
  YX_REQUIRE(in_c_real > 0 && in_c_real <= in_c && out_c_real > 0 && out_c_real <= out_c, YX_ERR_INVALID_ARG, "wgrad: real channel counts");
  WgradParams p;
  size_t smem = 0;
  int rc = wgrad_plan(batch, in_h, in_w, in_c, out_h, out_w, out_c, ksize, stride, &p, &smem);
  if (rc) return rc;
  YX_REQUIRE((long long)p.ksplit * p.split_stride * 4 <= ws_bytes, YX_ERR_CAPACITY, "wgrad: workspace of %lld bytes, need %lld",
             ws_bytes, (long long)p.ksplit * p.split_stride * 4);
  p.partial = reinterpret_cast<float*>(ws);
  p.lbo_a16 = p.a_block_bytes >> 4;
  p.lbo_b16 = p.b_block_bytes >> 4;
  p.desc_hi_a = umma_desc_hi(p.rb_a);
  p.desc_hi_b = umma_desc_hi(p.rb_b);
  p.idesc = umma_idesc(dtype, p.N, /*mn_major=*/true);

  CUtensorMap map_dy, map_x;
  {
    cuuint64_t dims[4] = {(cuuint64_t)out_c, (cuuint64_t)out_w, (cuuint64_t)out_h, (cuuint64_t)batch};
    cuuint64_t strides[3] = {(cuuint64_t)dy_ld * 2, (cuuint64_t)dy_ld * 2 * out_w, (cuuint64_t)dy_ld * 2 * out_w * out_h};
    cuuint32_t box[4] = {(cuuint32_t)p.co_box, (cuuint32_t)p.tw, (cuuint32_t)p.th, 1};
    rc = encode_tma(&map_dy, tma_dtype(dtype), 4, dy, dims, strides, box, nullptr, tma_swizzle(p.rb_a),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "wgrad dy");
    if (rc) return rc;
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)in_c, (cuuint64_t)in_w, (cuuint64_t)in_h, (cuuint64_t)batch};
    cuuint64_t strides[3] = {(cuuint64_t)x_ld * 2, (cuuint64_t)x_ld * 2 * in_w, (cuuint64_t)x_ld * 2 * in_w * in_h};
    cuuint32_t box[4] = {(cuuint32_t)p.ci_box, (cuuint32_t)(p.tw * stride), (cuuint32_t)(p.th * stride), 1};
    cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    rc = encode_tma(&map_x, tma_dtype(dtype), 4, x, dims, strides, box, estr, tma_swizzle(p.rb_b), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    "wgrad x");
    if (rc) return rc;
  }
  static bool smem_set[kMaxDevices] = {};
  YX_CUDA(opt_in_smem(smem_set, &wgrad_tc_kernel, [](int) {
    cudaFuncAttributes fa = {};
    cudaFuncGetAttributes(&fa, wgrad_tc_kernel);             // the opt-in limit covers static + dynamic shared memory
    return max_smem_optin() - (int)fa.sharedSizeBytes;
  }));
  const int grid = p.m_tiles * p.n_groups * p.ksplit;
  YX_CUDA(launch_kernel(wgrad_tc_kernel, dim3(grid), dim3(192), smem, stream, map_dy, map_x, p));
  const long long total = (long long)out_c * p.taps * in_c;
  const int rgrid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  YX_CUDA(launch_kernel(wgrad_reduce_kernel, dim3(rgrid), dim3(256), 0, stream, (const float*)p.partial, p.ksplit, p.split_stride,
                        p.row_stride, p.N, p.taps, out_c, in_c, out_c_real, in_c_real, dw, dw_so, dw_si, dw_st, accumulate));
  return YX_OK;
}

int pack_train_weights_launch(const float* w, long long so, long long si, long long st, int o, int i, int taps, int o_pad, int i_pad,
                              void* wf, void* wd, int subpixel, int dtype, cudaStream_t stream) {
  YX_REQUIRE(w && (wf || wd), YX_ERR_INVALID_ARG, "pack_train_weights: null pointer");
  YX_REQUIRE(!subpixel || taps == 9, YX_ERR_INVALID_ARG, "pack_train_weights: the sub-pixel dgrad form is for 3x3 convs");
  YX_REQUIRE(dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_UNSUPPORTED, "pack_train_weights: 16-bit destinations only");
  YX_REQUIRE(o > 0 && i > 0 && o <= o_pad && i <= i_pad && (taps == 1 || taps == 9), YX_ERR_INVALID_ARG, "pack_train_weights: shape");
  const long long total = (long long)o_pad * taps * i_pad;
  const int grid = (int)((total + 255) / 256 < 2048 ? (total + 255) / 256 : 2048);
  if (dtype == YX_BF16)
    YX_CUDA(launch_kernel(pack_train_weights_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, w, so, si, st, o, i, taps, o_pad, i_pad,
                       reinterpret_cast<__nv_bfloat16*>(wf), reinterpret_cast<__nv_bfloat16*>(wd), subpixel));
  else
    YX_CUDA(launch_kernel(pack_train_weights_kernel<__half>, dim3(grid), dim3(256), 0, stream, w, so, si, st, o, i, taps, o_pad, i_pad,
                       reinterpret_cast<__half*>(wf), reinterpret_cast<__half*>(wd), subpixel));
  return YX_OK;
}

int pack_train_weights_multi_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, int dtype, cudaStream_t stream) {
  YX_REQUIRE(table && chunks && n_chunks > 0 && chunk_elems > 0, YX_ERR_INVALID_ARG, "pack_train_weights_multi: arguments");
  YX_REQUIRE(dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_UNSUPPORTED, "pack_train_weights_multi: 16-bit destinations only");
  if (dtype == YX_BF16) pack_train_weights_multi_kernel<__nv_bfloat16><<<n_chunks, 256, 0, stream>>>(table, chunks, chunk_elems);
  else pack_train_weights_multi_kernel<__half><<<n_chunks, 256, 0, stream>>>(table, chunks, chunk_elems);
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int dilate2_launch(const void* dy, void* z, int batch, int oh, int ow, int zh, int zw, int c, cudaStream_t stream) {
  YX_REQUIRE(dy && z && c % 8 == 0 && batch > 0 && oh > 0 && ow > 0 && zh >= 2 * oh - 1 && zw >= 2 * ow - 1, YX_ERR_INVALID_ARG, "dilate2: shape");
  const long long total = (long long)batch * zh * zw * (c / 8);
  const int grid = (int)((total + 255) / 256 < 8192 ? (total + 255) / 256 : 8192);
  YX_CUDA(launch_kernel(dilate2_kernel, dim3(grid), dim3(256), 0, stream, reinterpret_cast<const uint4*>(dy), reinterpret_cast<uint4*>(z), batch, oh, ow,
                     zh, zw, c / 8));
  return YX_OK;
}

}  // namespace yx
