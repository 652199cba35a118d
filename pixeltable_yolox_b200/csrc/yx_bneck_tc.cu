// Fused Bottleneck for sm_100a: y = [x +] act(bn2(conv3x3(act(bn1(conv1x1(x)))))) in ONE kernel.
//   reference: Bottleneck.forward (yolox/models/network_blocks.py:77-99) = two BaseConv
//   (network_blocks.py:27-52) and the shortcut add; BN folded as in fuse_conv_and_bn
//   (yolox/utils/model_utils.py:33-75).
//
// The hidden tensor h = conv1(x) never touches HBM: per spatial tile (th x tw outputs)
//   1. TMA loads the (th+2) x (tw+2) halo of x as a K-major swizzled operand           (X slot)
//   2. GEMM1 (tcgen05): h_acc[halo pixel, C] = X * W1^T over the WHOLE halo (two 128-row MMA tiles),
//      fp32 accumulators in TMEM
//   3. epilogue 1: TMEM -> bias1 + act -> 16-bit, written back to shared memory in the same
//      canonical K-major swizzled layout (H slot); halo pixels outside the image are written as
//      ZERO (they are conv2's zero padding, not act(bias1)); fence.proxy.async publishes the tile
//   4. GEMM2: the nine taps of the 3x3 conv are nine row-shifted UMMA descriptors into the H slot
//      (tap (r,s) = rows shifted by r*(tw+2)+s) against the resident W2
//   5. epilogue 2: bias2 + act (+ x re-read at the centre pixel, an L2 hit) -> 256-bit stores
// W1 and the nine W2 tiles stay resident in shared memory for the whole kernel. One persistent CTA
// per SM walks a contiguous range of tiles; GEMM1 of tile i+1 is issued before GEMM2 of tile i so
// the two epilogue groups and the tensor core overlap. Channels: C in {16, 32, 64} (one swizzle row).
// HBM traffic per pixel: C in + C out (the unfused pair moves 5 C with the shortcut).
#include <string.h>

#include <new>

#include "yx_tc_epilogue.cuh"

namespace yx {

static constexpr int kBnX = 6;          // max X halo slots
static constexpr int kBnThreads = 64 + 256 + 256 + 32;   // TMA + GEMM2 warps, 8 epilogue-1 warps (4 per GEMM1 tile), 8 epilogue-2 warps, GEMM1 warp
static constexpr int kWarpG1 = 18;

struct BneckParams {
  int C, Cpad;               // channels (= N = K), TMEM column pitch
  int tw, th, pitch;         // spatial tile and accumulator row pitch (tw + 2)
  int tiles_w, tiles_h, num_tiles, tiles_per_img;
  int batch, H, W;
  int ksteps;                // C / 16
  int halo_rows;             // (th + 2) * pitch
  int nx;                    // X halo slots in the ring
  unsigned row_bytes, x_slot_bytes, h_slot_bytes, x_tx_bytes, w_tile_bytes, w_tx_bytes;
  unsigned desc_hi, idesc, tmem_cols, bias_bytes, swz_mask;
  unsigned mul_tpi, mul_tw;
  int act1;
  const float* bias1;
  EpiParams epi;             // second conv: bias2, act, out, res (= x when the block has a shortcut)
};

struct __align__(8) BneckShared {
  uint64_t xfull[kBnX], xempty[kBnX];
  uint64_t a1full[2], a1empty[2];
  uint64_t hfull[2], hempty[2];
  uint64_t a2full[2], a2empty[2];
  uint64_t wfull;
  uint32_t tmem_base;
};

template <bool FP16, int KS, bool SILU>
__global__ void __launch_bounds__(kBnThreads, 1)
bneck_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w1,
                const __grid_constant__ CUtensorMap map_w2, const BneckParams p) {
  extern __shared__ uint8_t smem_raw[];
  // pointer arithmetic on the __shared__ array (not an integer round trip) keeps the address space known to the
  // compiler: LDS/STS instead of generic loads for every bias / staging access
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  BneckShared* sh = reinterpret_cast<BneckShared*>(smem);
  float* sbias1 = reinterpret_cast<float*>(smem + 1024);
  float* sbias2 = sbias1 + p.bias_bytes / 4;
  uint8_t* xs = smem + 1024 + 2 * p.bias_bytes;                 // [kBnX] halo of x
  uint8_t* hs = xs + (size_t)p.nx * p.x_slot_bytes;                       // [2] hidden halo tile
  uint8_t* w1s = hs + 2 * p.h_slot_bytes;                         // [C x C]
  uint8_t* w2s = w1s + p.w_tile_bytes;                            // [9][C x C]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr bool fp16 = FP16;
  constexpr int C = 16 * KS;                            // channels: loops over them unroll completely
  {
    const bool half1 = (p.act1 == YX_ACT_SILU && !fp16);
    const float s1 = half1 ? 0.5f : 1.0f, s2 = epi_half_bias(p.epi) ? 0.5f : 1.0f;
    for (int i = threadIdx.x; i < p.C; i += blockDim.x) { sbias1[i] = p.bias1[i] * s1; sbias2[i] = p.epi.bias[i] * s2; }
  }
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x); tma_prefetch_desc(&map_w1); tma_prefetch_desc(&map_w2);
    for (int i = 0; i < p.nx; ++i) { mbar_init(&sh->xfull[i], 1); mbar_init(&sh->xempty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sh->a1full[i], 1); mbar_init(&sh->a1empty[i], 256);
      mbar_init(&sh->hfull[i], 256); mbar_init(&sh->hempty[i], 1);
      mbar_init(&sh->a2full[i], 1); mbar_init(&sh->a2empty[i], 128);
    }
    mbar_init(&sh->wfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(&sh->tmem_base, p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // Values every role needs are NOT kept in registers across the role branch: at the 96-register cap of this CTA size ptxas
  // spilled exactly those (tmem_base, tiles per image) to local memory, and with the L1 carved out for shared memory every
  // reload in the per-tile loops was an L2 round trip (~700 clk per tile in epilogue 1, the critical stage, measured
  // with a clock64 trace). Each role re-reads them from shared memory / the constant bank instead.
#define tmem_base (sh->tmem_base)
#define tiles_per_img (p.tiles_per_img)
  pdl_launch_dependents();      // the weights are constants: loaded before griddepcontrol.wait (see the producer)

  const long long T = p.num_tiles;
  const int t_begin = (int)(T * blockIdx.x / gridDim.x), t_end = (int)(T * (blockIdx.x + 1) / gridDim.x);
  const int n_my = t_end - t_begin;
  // TMEM columns: acc1[stage][m-tile] then acc2[stage]
  const uint32_t acc1_col = 0, acc2_col = (uint32_t)(4 * p.Cpad);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(&sh->wfull, p.w_tx_bytes * 10u);
      tma_load_2d(&map_w1, &sh->wfull, w1s, 0, 0);
      for (int tap = 0; tap < 9; ++tap) tma_load_2d(&map_w2, &sh->wfull, w2s + (size_t)tap * p.w_tile_bytes, tap * p.C, 0);
      pdl_wait();
      int sx = 0;
      uint32_t px = 0;
      for (int t = t_begin; t < t_end; ++t) {
        const int b = fast_div(t, p.mul_tpi, tiles_per_img);
        const int r = t - b * tiles_per_img;
        const int ty = fast_div(r, p.mul_tw, p.tiles_w);
        const int tx = r - ty * p.tiles_w;
        mbar_wait(&sh->xempty[sx], px ^ 1);
        mbar_arrive_expect_tx(&sh->xfull[sx], p.x_tx_bytes);
        tma_load_4d(&map_x, &sh->xfull[sx], xs + (size_t)sx * p.x_slot_bytes, 0, tx * p.tw - 1, ty * p.th - 1, b);
        if (++sx == p.nx) { sx = 0; px ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== GEMM2 issuer =====================
    const uint64_t dhi = ((uint64_t)p.desc_hi << 32) | (1u << 16);
    const uint32_t rb16 = p.row_bytes >> 4, prb16 = (uint32_t)p.pitch * rb16;
    const uint32_t x16 = smem_u32(xs) >> 4, xslot16 = p.x_slot_bytes >> 4;
    const uint32_t h16 = smem_u32(hs) >> 4, hslot16 = p.h_slot_bytes >> 4;
    const uint64_t w1d = dhi | (uint64_t)(smem_u32(w1s) >> 4);
    const uint32_t w2_16 = smem_u32(w2s) >> 4, wt16 = p.w_tile_bytes >> 4;
    const uint32_t idesc = p.idesc;
    constexpr int ks = KS;
    mbar_wait(&sh->wfull, 0);
    int sx = 0;
    uint32_t px = 0;
    for (int it = 0; it < n_my; ++it) {
      const int st = it & 1;
      const uint32_t ph = (uint32_t)((it >> 1) & 1);
      mbar_wait(&sh->hfull[st], ph);
      mbar_wait(&sh->a2empty[st], ph ^ 1);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint64_t hd = dhi | (uint64_t)(h16 + (uint32_t)st * hslot16);
        const uint32_t d2 = tmem_base + acc2_col + (uint32_t)(st * p.Cpad);
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const uint64_t a = hd + (uint64_t)((uint32_t)(tap / 3) * prb16 + (uint32_t)(tap % 3) * rb16);
          const uint64_t b = dhi | (uint64_t)(w2_16 + (uint32_t)tap * wt16);
#pragma unroll
          for (int j = 0; j < ks; ++j) umma_f16(d2, a + 2 * j, b + 2 * j, idesc, (uint32_t)((tap | j) != 0));
        }
        umma_commit(&sh->a2full[st]);
        umma_commit(&sh->hempty[st]);
      }
      __syncwarp();
    }
  } else if (warp == kWarpG1) {
    // ===================== GEMM1 issuer (own warp: its waits and commits never delay GEMM2) =====================
    const uint64_t dhi = ((uint64_t)p.desc_hi << 32) | (1u << 16);
    const uint32_t rb16 = p.row_bytes >> 4;
    const uint32_t x16 = smem_u32(xs) >> 4, xslot16 = p.x_slot_bytes >> 4;
    const uint64_t w1d = dhi | (uint64_t)(smem_u32(w1s) >> 4);
    const uint32_t idesc = p.idesc;
    constexpr int ks = KS;
    mbar_wait(&sh->wfull, 0);
    int sx = 0;
    uint32_t px = 0;
    // GEMM1 of tile k: whole halo (two 128-row tiles) x W1
    for (int k = 0; k < n_my; ++k) {
      const int st = k & 1;
      mbar_wait(&sh->xfull[sx], px);
      mbar_wait(&sh->a1empty[st], (uint32_t)(((k >> 1) & 1) ^ 1));
      tc_fence_after();
      if (elect_one_sync()) {
        const uint64_t xd = dhi | (uint64_t)(x16 + (uint32_t)sx * xslot16);
        const uint32_t d0 = tmem_base + acc1_col + (uint32_t)((st * 2) * p.Cpad);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const uint64_t a = xd + (uint64_t)(mt * 128) * rb16;
#pragma unroll
          for (int j = 0; j < ks; ++j) umma_f16(d0 + (uint32_t)(mt * p.Cpad), a + 2 * j, w1d + 2 * j, idesc, (uint32_t)(j != 0));
        }
        umma_commit(&sh->a1full[st]);
        umma_commit(&sh->xempty[sx]);
      }
      __syncwarp();
      if (++sx == p.nx) { sx = 0; px ^= 1; }
    }
  } else if (warp < 10) {
    // ===================== epilogue 1: h = act(acc1 + b1) -> swizzled shared operand =====================
    // warps 2..5 own GEMM1 tile 0 (halo rows 0..127), warps 6..9 tile 1 (rows 128..)
    const int quarter = warp & 3;
    const int t128 = quarter * 32 + lane;                 // TMEM lane = row inside the 128-row MMA tile
    const int mt = (warp - 2) >> 2;
    const int q = mt * 128 + t128;
    const int yy = q / p.pitch, xx = q - yy * p.pitch;
    const bool warp_live = mt * 128 + quarter * 32 < p.halo_rows + 2;   // (warp-uniform) rows some tap of a real output reads
    const bool stored = q < p.halo_rows + 2;
    const uint32_t rowoff = (uint32_t)q * (uint32_t)(C * 2);
    // canonical K-major layout: the 16-byte chunk index is XOR-ed with address bits [7, 7 + log2(mask + 1)) of the row
    const uint32_t xr = (rowoff >> 7) & (C == 64 ? 7u : (C == 32 ? 3u : 1u));
    constexpr bool silu_tanh1 = SILU && !FP16;      // compile-time: no activation dispatch (indirect branch) per chunk
    for (int it = 0; it < n_my; ++it) {
      const int t = t_begin + it;
      const int b = fast_div(t, p.mul_tpi, tiles_per_img);
      const int r = t - b * tiles_per_img;
      const int ty = fast_div(r, p.mul_tw, p.tiles_w);
      const int tx = r - ty * p.tiles_w;
      const int st = it & 1;
      const uint32_t ph = (uint32_t)((it >> 1) & 1);
      mbar_wait(&sh->a1full[st], ph);
      tc_fence_after();
      // the first TMEM loads are issued before the wait for the hidden-tile slot: that wait (a shared-memory round trip of
      // ~170 clk even when the phase completed long ago) overlaps their latency
      constexpr int KH = KS >= 2 ? 2 : 1;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc1_col + (uint32_t)((st * 2 + mt) * p.Cpad);
      uint32_t raw[KH][16];
      if (warp_live) {
#pragma unroll
        for (int k = 0; k < KH; ++k) tmem_ld_x16(taddr + (uint32_t)(16 * k), raw[k]);
      }
      mbar_wait(&sh->hempty[st], ph ^ 1);
      uint8_t* hslot = hs + (size_t)st * p.h_slot_bytes;
      if (warp_live) {
        const int iy = ty * p.th - 1 + yy, ix = tx * p.tw - 1 + xx;
        const bool inside = (q < p.halo_rows) && iy >= 0 && iy < p.H && ix >= 0 && ix < p.W && b < p.batch;
        // 16 hidden channels of this thread's halo pixel: bias + act -> two swizzled 16-byte chunks
        auto emit = [&](const uint32_t (&raw)[16], int c) {
          uint32_t w[8];
          if (inside) {
            float v[16];
            if constexpr (silu_tanh1) {
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const float4 bb = *reinterpret_cast<const float4*>(sbias1 + c + j);
                const float hb[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float h = fmaf(__uint_as_float(raw[j + u]), 0.5f, hb[u]);
                  float tt;
                  asm("tanh.approx.f32 %0, %1;" : "=f"(tt) : "f"(h));
                  v[j + u] = fmaf(h, tt, h);
                }
              }
            } else if constexpr (SILU && FP16) {
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const float4 bb = *reinterpret_cast<const float4*>(sbias1 + c + j);
                v[j + 0] = silu_exp(__uint_as_float(raw[j + 0]) + bb.x);
                v[j + 1] = silu_exp(__uint_as_float(raw[j + 1]) + bb.y);
                v[j + 2] = silu_exp(__uint_as_float(raw[j + 2]) + bb.z);
                v[j + 3] = silu_exp(__uint_as_float(raw[j + 3]) + bb.w);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = act_f<false>(__uint_as_float(raw[j]) + sbias1[c + j], p.act1);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) w[j] = pack16_t<FP16>(v[2 * j], v[2 * j + 1]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) w[j] = 0u;
          }
#pragma unroll
          for (int hch = 0; hch < 2; ++hch) {
            // chunk index inside the row: (c/8 + hch); rows of 32/64 bytes share a 128-byte line with their neighbours,
            // so the XOR acts on the full in-line chunk position
            const uint32_t a = rowoff + (uint32_t)(c * 2 + hch * 16);
            const uint32_t phys = (a & ~0x70u) | ((((a >> 4) & 7u) ^ xr) << 4);
            if (stored) *reinterpret_cast<uint4*>(hslot + phys) = make_uint4(w[4 * hch], w[4 * hch + 1], w[4 * hch + 2], w[4 * hch + 3]);
          }
        };
        // up to 32 channels (two TMEM loads) in flight at a time: with all four loads of a 64-channel row live next to the
        // 16 activations of a chunk the kernel needs > 96 registers (the cap at 608 threads) and ptxas spills loop invariants
        // to local memory, whose reloads are L2 round trips here (the L1 is carved out for shared memory)
#pragma unroll
        for (int k0 = 0; k0 < KS; k0 += KH) {
          if (k0) {
#pragma unroll
            for (int k = 0; k < KH; ++k) tmem_ld_x16(taddr + (uint32_t)(16 * (k0 + k)), raw[k]);
          }
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < KH; ++k) emit(raw[k], 16 * (k0 + k));
        }
      }
      tc_fence_before();
      mbar_arrive(&sh->a1empty[st]);
      fence_proxy_async();                     // generic-proxy stores -> visible to the tensor core
      mbar_arrive(&sh->hfull[st]);
    }
  } else {
    // ===================== epilogue 2: y = act(acc2 + b2) (+ x) =====================
    pdl_wait();
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int hl0 = row / p.pitch, wl0 = row - hl0 * p.pitch;
    const bool row_ok = hl0 < p.th && wl0 < p.tw;
    const int grp = (warp - 10) >> 2;                     // tiles alternate between the two groups; group g owns acc2 stage g
    for (int it = grp; it < n_my; it += 2) {
      const int t = t_begin + it;
      const int b = fast_div(t, p.mul_tpi, tiles_per_img);
      const int r = t - b * tiles_per_img;
      const int ty = fast_div(r, p.mul_tw, p.tiles_w);
      const int tx = r - ty * p.tiles_w;
      const int ho = ty * p.th + hl0, wo = tx * p.tw + wl0;
      const bool valid = row_ok && ho < p.H && wo < p.W && b < p.batch;
      const long long pix = ((long long)b * p.H + ho) * p.W + wo;
      const int st = it & 1;
      mbar_wait(&sh->a2full[st], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc2_col + (uint32_t)(st * p.Cpad);
      uint16_t* orow = (uint16_t*)p.epi.out + pix * p.epi.out_ld;
      const uint16_t* rrow = p.epi.res ? (const uint16_t*)p.epi.res + pix * p.epi.res_ld : nullptr;
#pragma unroll
      for (int c = 0; c < C; c += 32) {
        const bool two = (C % 32 == 0) || (c + 16 < C);
        uint32_t ra[16], rb[16];
        tmem_ld_x16(taddr + (uint32_t)c, ra);
        if (two) tmem_ld_x16(taddr + (uint32_t)(c + 16), rb);
        uint32_t qa[8], qb[8];
        if (rrow && valid) {
          ld_global_256(rrow + c, qa);
          if (two) ld_global_256(rrow + c + 16, qb);
        }
        tmem_ld_wait();
        if (valid) {
          epi_tc_chunk<FP16, SILU>(p.epi, ra, sbias2 + c, rrow ? qa : nullptr, orow + c, b, ho, wo, c);
          if (two) epi_tc_chunk<FP16, SILU>(p.epi, rb, sbias2 + c + 16, rrow ? qb : nullptr, orow + c + 16, b, ho, wo, c + 16);
        }
      }
      tc_fence_before();
      mbar_arrive(&sh->a2empty[st]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
#undef tmem_base
#undef tiles_per_img
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct BneckLaunch {
  CUtensorMap map_x, map_w1, map_w2;
  BneckParams p;
  int grid;
  size_t smem;
};

BneckLaunch* bneck_alloc() { return new (std::nothrow) BneckLaunch(); }
void bneck_free(BneckLaunch* p) { delete p; }

bool bneck_supported(const yx_bneck_desc* d) {
  return d && (d->c == 16 || d->c == 32 || d->c == 64) && (d->dtype == YX_BF16 || d->dtype == YX_FP16);
}

int bneck_prepare(const yx_bneck_desc* d, BneckLaunch* L) {
  YX_REQUIRE(d != nullptr, YX_ERR_INVALID_ARG, "bottleneck: null descriptor");
  YX_REQUIRE(d->c == 16 || d->c == 32 || d->c == 64, YX_ERR_UNSUPPORTED, "bottleneck: c=%d (fused kernel: 16, 32 or 64)", d->c);
  YX_REQUIRE(d->dtype == YX_BF16 || d->dtype == YX_FP16, YX_ERR_INVALID_ARG, "bottleneck: dtype must be bf16/fp16");
  YX_REQUIRE(d->batch > 0 && d->h > 0 && d->w > 0, YX_ERR_INVALID_ARG, "bottleneck: empty input");
  YX_REQUIRE(d->x && d->w1 && d->w2 && d->bias1 && d->bias2 && d->out, YX_ERR_INVALID_ARG, "bottleneck: null pointer");
  YX_REQUIRE(d->x_ld % 16 == 0 && d->out_ld % 16 == 0 && d->x_ld >= d->c && d->out_ld >= d->c, YX_ERR_INVALID_ARG,
             "bottleneck: x_ld/out_ld must be multiples of 16 and >= c");
  YX_REQUIRE(((uintptr_t)d->x & 31) == 0 && ((uintptr_t)d->out & 31) == 0 && ((uintptr_t)d->w1 & 15) == 0 &&
                 ((uintptr_t)d->w2 & 15) == 0 && ((uintptr_t)d->bias1 & 15) == 0 && ((uintptr_t)d->bias2 & 15) == 0,
             YX_ERR_INVALID_ARG, "bottleneck: pointer alignment");
  {
    // the halo of a tile is read while other tiles are written: in-place operation is not possible
    const char* x0 = (const char*)d->x; const char* o0 = (const char*)d->out;
    const long long span_x = ((long long)d->batch * d->h * d->w - 1) * d->x_ld * 2 + d->c * 2;
    const long long span_o = ((long long)d->batch * d->h * d->w - 1) * d->out_ld * 2 + d->c * 2;
    const bool disjoint_range = (o0 + span_o <= x0) || (x0 + span_x <= o0);
    // two channel slices of the same buffer interleave in memory; they are disjoint iff the slices do not overlap
    bool ok = disjoint_range;
    if (!ok && d->x_ld == d->out_ld) {
      const long long delta = (o0 - x0) / 2;
      const long long m = ((delta % d->x_ld) + d->x_ld) % d->x_ld;
      ok = (m >= d->c) && (m + d->c <= d->x_ld);
    }
    YX_REQUIRE(ok, YX_ERR_INVALID_ARG, "bottleneck: out must not alias x (the fused kernel cannot run in place)");
  }
  BneckParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.C = d->c; p.Cpad = d->c < 32 ? 32 : d->c;
  p.batch = d->batch; p.H = d->h; p.W = d->w;
  p.ksteps = d->c / 16;
  p.row_bytes = (unsigned)d->c * 2u;
  p.swz_mask = d->c == 64 ? 7u : (d->c == 32 ? 3u : 1u);
  long long best = -1; int btw = 1, bth = 1;
  for (int tw = 1; tw <= d->w && tw + 2 <= 128; ++tw) {
    int th = 128 / (tw + 2);
    if (th > d->h) th = d->h;
    if (th < 1) continue;
    if ((th + 2) * (tw + 2) + 2 > 256) continue;          // the halo must fit the two 128-row GEMM1 tiles
    const long long tiles = ceil_div64(d->w, tw) * ceil_div64(d->h, th);
    const long long cost = tiles * 4096 + (long long)(th + 2) * (tw + 2);
    if (best < 0 || cost < best) { best = cost; btw = tw; bth = th; }
  }
  p.tw = btw; p.th = bth; p.pitch = btw + 2;
  p.halo_rows = (p.th + 2) * p.pitch;
  p.tiles_w = (int)ceil_div64(d->w, p.tw); p.tiles_h = (int)ceil_div64(d->h, p.th);
  p.num_tiles = d->batch * p.tiles_w * p.tiles_h;
  p.tiles_per_img = p.tiles_w * p.tiles_h;
  p.mul_tpi = fast_div_mul(p.tiles_w * p.tiles_h); p.mul_tw = fast_div_mul(p.tiles_w);
  // GEMM1 reads 256 rows from the slot start and GEMM2 rows up to 127 + 2*pitch + 2: 256 rows cover both
  // GEMM1's second tile reads rows 128..255 from the slot start: rows past the slot are the next slot / the H
  // region (garbage accumulator rows that nothing reads); GEMM2 reads rows <= 127 + 2*pitch + 2 < halo_rows + 2
  p.x_slot_bytes = ((unsigned)(p.halo_rows + 2) * p.row_bytes + 1023u) & ~1023u;
  p.h_slot_bytes = p.x_slot_bytes;
  p.x_tx_bytes = (unsigned)p.halo_rows * p.row_bytes;
  p.w_tile_bytes = ((unsigned)d->c * p.row_bytes + 1023u) & ~1023u;   // [N = c rows x c channels]
  p.w_tx_bytes = (unsigned)d->c * p.row_bytes;
  p.bias_bytes = 1024u;
  p.tmem_cols = 32; while (p.tmem_cols < (unsigned)(6 * p.Cpad)) p.tmem_cols <<= 1;
  p.desc_hi = umma_desc_hi(p.row_bytes);
  p.idesc = umma_idesc(d->dtype, d->c);
  p.act1 = d->act; p.bias1 = d->bias1;
  EpiParams& e = p.epi;
  e.out_h = d->h; e.out_w = d->w; e.out_c = d->c; e.act = d->act; e.dtype = d->dtype; e.epilogue = YX_EPI_STORE;
  e.bias = d->bias2; e.out = d->out; e.out_ld = d->out_ld;
  e.res = d->use_add ? d->x : nullptr; e.res_ld = d->x_ld;
  const int max_smem = max_smem_optin();
  const long long fixed = 2048 + 2 * (long long)p.bias_bytes + 2 * (long long)p.h_slot_bytes + 10 * (long long)p.w_tile_bytes;
  p.nx = (int)((max_smem - fixed) / p.x_slot_bytes);
  if (p.nx > kBnX) p.nx = kBnX;
  YX_REQUIRE(p.nx >= 2, YX_ERR_UNSUPPORTED, "bottleneck: shared memory too small (%lld fixed bytes)", fixed);
  L->smem = (size_t)fixed + (size_t)p.nx * p.x_slot_bytes;

  const CUtensorMapDataType tdt = tma_dtype(d->dtype);
  const CUtensorMapSwizzle sw = tma_swizzle(p.row_bytes);
  {
    cuuint64_t dims[4] = {(cuuint64_t)d->c, (cuuint64_t)d->w, (cuuint64_t)d->h, (cuuint64_t)d->batch};
    cuuint64_t strides[3] = {(cuuint64_t)d->x_ld * 2, (cuuint64_t)d->x_ld * 2 * d->w, (cuuint64_t)d->x_ld * 2 * d->w * d->h};
    cuuint32_t box[4] = {(cuuint32_t)d->c, (cuuint32_t)p.pitch, (cuuint32_t)(p.th + 2), 1};
    const int rc = encode_tma(&L->map_x, tdt, 4, d->x, dims, strides, box, nullptr, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              "bottleneck x");
    if (rc) return rc;
  }
  for (int which = 0; which < 2; ++which) {
    const cuuint64_t K = (cuuint64_t)(which ? 9 : 1) * d->c;
    cuuint64_t dims[2] = {K, (cuuint64_t)d->c};
    cuuint64_t strides[1] = {K * 2};
    cuuint32_t box[2] = {(cuuint32_t)d->c, (cuuint32_t)d->c};
    const int rc = encode_tma(which ? &L->map_w2 : &L->map_w1, tdt, 2, which ? d->w2 : d->w1, dims, strides, box, nullptr, sw,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, which ? "bottleneck W2" : "bottleneck W1");
    if (rc) return rc;
  }
  const int sms = num_sms();
  L->grid = p.num_tiles < sms ? p.num_tiles : sms;
  return YX_OK;
}

// [fp16][KS = 1, 2, 4][SiLU]
static decltype(&bneck_tc_kernel<false, 1, false>) const kBneckKernels[2][3][2] = {
    {{bneck_tc_kernel<false, 1, false>, bneck_tc_kernel<false, 1, true>},
     {bneck_tc_kernel<false, 2, false>, bneck_tc_kernel<false, 2, true>},
     {bneck_tc_kernel<false, 4, false>, bneck_tc_kernel<false, 4, true>}},
    {{bneck_tc_kernel<true, 1, false>, bneck_tc_kernel<true, 1, true>},
     {bneck_tc_kernel<true, 2, false>, bneck_tc_kernel<true, 2, true>},
     {bneck_tc_kernel<true, 4, false>, bneck_tc_kernel<true, 4, true>}}};

int bneck_launch(const BneckLaunch* L, cudaStream_t stream) {
  static bool smem_set[kMaxDevices] = {};
  YX_CUDA(opt_in_smem(smem_set, kBneckKernels, [](int) { return max_smem_optin(); }));
  const auto kernel = kBneckKernels[L->p.epi.dtype == YX_FP16][L->p.ksteps / 2][L->p.act1 == YX_ACT_SILU];
  YX_CUDA(launch_pdl(kernel, dim3((unsigned)L->grid), dim3((unsigned)kBnThreads), L->smem, stream, L->map_x, L->map_w1, L->map_w2,
                     L->p));
  return YX_OK;
}

}  // namespace yx
