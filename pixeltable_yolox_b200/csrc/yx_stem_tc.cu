// Fused Focus + stem conv for sm_100a: space-to-depth, 3x3 conv, folded BN and SiLU in ONE kernel.
//   reference: Focus.forward (yolox/models/network_blocks.py:186-208) followed by its BaseConv
//   (network_blocks.py:27-52).
// The raw NCHW image (fp32 or uint8, 0..255) is read once and the NHWC 16-bit stem output written
// once; nothing else touches HBM.
//
// GEMM view: the 3x3 conv runs on the space-to-depth grid (H/2 x W/2, 12 channels padded to K = 16 per tap).
// Per tile of 7 x 16 output pixels:
//   warp 9      TMA-loads the tile's 3 x 18 x 36 raw patch (one 4-D box of the NCHW image, zero filled outside
//               the image = Conv2d padding) into a 4-deep ring;
//   warps 0-7   two groups of "builders" (alternating tiles) turn it into the space-to-depth HALO tile: 9 x 18
//               pixels x 16 channels (32-byte rows, canonical K-major SWIZZLE_32B layout). Every raw pixel is
//               converted exactly once (the first version built the im2col operand, 9x the conversions and 32 KB
//               of shared-memory stores per tile; ncu/roofline: shared-memory bandwidth bound at ~2x the HBM time);
//   warp 8      issues nine tcgen05.mma per tile, one per filter tap: the A descriptor of tap (r, s) is the SAME
//               halo tile with its start address shifted by r*18 + s rows (accumulator row m = y*18 + x; columns
//               x >= 16 are garbage and dropped by the epilogue), B = the tap's [out_c x 16] weight tile resident
//               in shared memory; accumulators in TMEM (4 stages);
//   warps 10-17 two epilogue groups (bias + SiLU + 256-bit stores).
// K order inside a tap: k = 2*(2*c + py) + px for image channel c and pixel parity (py, px), i.e. Focus channel
// 3*(2*px + py) + c (network_blocks.py:199-207: TL, BL, TR, BR); k = 12..15 are zero.
#include <string.h>

#include <new>

#include "yx_tc_epilogue.cuh"

namespace yx {

static constexpr int kStemBuilders = 128;            // threads per builder group
static constexpr int kStemMaxRing = 4;               // barrier arrays are sized for the largest variant
// Variant V: 0 = one CTA per SM (two builder groups, two issuing warps, four epilogue groups, 4-deep rings);
//            1 = two co-resident CTAs per SM with half of everything each (one builder group, one issuing warp, two
//                epilogue groups, 2-deep rings).
// The single-CTA kernel is bound by the hand-off latency of its TMA -> builder -> MMA -> epilogue pipeline (~1 000 clk per
// 120-pixel tile with no unit saturated, section 4.4 of DESIGN.md); two independent pipelines per SM overlap that latency.
template <int V> struct StemCfg {
  static constexpr int kBuilderGroups = V == 0 ? 2 : 1;       // tiles alternate between the groups
  static constexpr int kMmaWarps = V == 0 ? 2 : 1;            // tiles alternate between the issuing warps
  static constexpr int kEpiGroups = V == 0 ? 4 : 2;
  static constexpr int kStages = V == 0 ? 4 : 2;              // halo-tile (A operand) stages
  static constexpr int kAcc = V == 0 ? 4 : 2;
  static constexpr int kPatchStages = V == 0 ? 4 : 2;
  static constexpr int kWarpMma = kStemBuilders * kBuilderGroups / 32, kWarpTma = kWarpMma + 1, kWarpEpi = kWarpMma + 2;
  static constexpr int kWarpMma2 = kWarpEpi + 4 * kEpiGroups;
  static constexpr int kThreads = kStemBuilders * kBuilderGroups + 64 + 128 * kEpiGroups + (kMmaWarps == 2 ? 32 : 0);
  static constexpr int kCtasPerSm = V == 0 ? 1 : 2;
  // A parity wait can only tell "this phase" from "the previous one": every waiter must stay within one phase of its
  // barrier. That holds when all uses of a ring slot belong to ONE group of warps working through its tiles in order, i.e.
  // when the group count divides the slot count (three epilogue groups on four accumulator slots let a group reach tile
  // t + 8 of a slot whose tile t + 4 was still in flight with the other issuing warp: wrong accumulators, then a deadlock).
  static_assert(kAcc % kEpiGroups == 0 && kStages % kBuilderGroups == 0 && kStages % kMmaWarps == 0 && kAcc % kMmaWarps == 0 &&
                kPatchStages % kBuilderGroups == 0, "ring slots must map to one warp group each (mbarrier parity aliasing)");
  static_assert(kStages <= kStemMaxRing && kAcc <= kStemMaxRing && kPatchStages <= kStemMaxRing, "ring depth");
};
// The output tile (th x tw, accumulator row m = y * (tw + 2) + x, th * (tw + 2) <= 128) is chosen per image width
// on the host: the raw patch arrives as 3 * (2*th + 4) TMA rows and the TMA unit's cost is per ROW (fp32 160-byte and
// uint8 64-byte rows of the first 7 x 16 tile took the same 250 us), so wide, flat tiles (3 x 40 at 640^2: 30 rows of
// 352 bytes per 120 pixels instead of 54 rows per 112) are what brings the kernel to the HBM roofline.

struct StemParams {
  const void* img; int img_dtype;
  int batch, h, w;            // image size
  int out_h, out_w;           // h/2, w/2
  int tiles_w, tiles_h, num_tiles;
  int tw, th, pitch, halo_pix;        // output tile, accumulator row pitch tw + 2, (th + 2) * pitch halo pixels
  int patch_rows, patch_pitch, lead;  // raw patch: 2*th + 4 rows of patch_pitch elements; the patch starts `lead` elements in
  unsigned patch_stage_bytes, a_stage_bytes;
  unsigned mul_tpi, mul_tw;           // fast_div multipliers for tiles per image / tiles per row
  int BN, BNpad;              // out_c (multiple of 16) and its TMEM pitch
  unsigned idesc, desc_hi, tmem_cols;
  unsigned bias_bytes, b_bytes, w_tile_bytes, patch_tx;
  EpiParams epi;
};

struct __align__(8) StemShared {
  uint64_t full[kStemMaxRing];
  uint64_t empty[kStemMaxRing];
  uint64_t tmem_full[kStemMaxRing];
  uint64_t tmem_empty[kStemMaxRing];
  uint64_t w_full;
  uint64_t patch_full[kStemMaxRing];
  uint64_t patch_empty[kStemMaxRing];
  uint32_t tmem_base;
};

__device__ __forceinline__ void bar_sync_named(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <typename TI>
__device__ __forceinline__ void load_pair(const TI* p, float& a, float& b);
template <>
__device__ __forceinline__ void load_pair<float>(const float* p, float& a, float& b) {
  const float2 v = *reinterpret_cast<const float2*>(p);
  a = v.x; b = v.y;
}
template <>
__device__ __forceinline__ void load_pair<uint8_t>(const uint8_t* p, float& a, float& b) {
  // u8 -> fp32 without I2F (conversions issue on the quarter-rate XU pipe, 108 of them per operand row):
  // 0x4B000000 | u is the float 2^23 + u, one FADD removes the 2^23
  const uint32_t v = *reinterpret_cast<const uint16_t*>(p);
  a = __uint_as_float(0x4B000000u | (v & 0xffu)) - 8388608.0f;
  b = __uint_as_float(0x4B000000u | (v >> 8)) - 8388608.0f;
}

template <typename TI, bool FP16, bool SILU, int V>
__global__ void __launch_bounds__(StemCfg<V>::kThreads, StemCfg<V>::kCtasPerSm)
stem_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_img,
               const StemParams p) {
  using Cfg = StemCfg<V>;
  constexpr int kStemStages = Cfg::kStages, kStemAcc = Cfg::kAcc, kPatchStages = Cfg::kPatchStages;
  constexpr int kStemBuilderGroups = Cfg::kBuilderGroups, kStemEpiGroups = Cfg::kEpiGroups, kMmaWarps = Cfg::kMmaWarps;
  constexpr int kWarpMma = Cfg::kWarpMma, kWarpTma = Cfg::kWarpTma, kWarpEpi = Cfg::kWarpEpi, kWarpMma2 = Cfg::kWarpMma2;
  extern __shared__ uint8_t smem_raw[];
  // pointer arithmetic on the __shared__ array (not an integer round trip) keeps the address space known to the
  // compiler: LDS/STS instead of generic loads for every bias / staging access
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  StemShared* sh = reinterpret_cast<StemShared*>(smem);
  float* sbias = reinterpret_cast<float*>(smem + 1024);
  uint8_t* patch = smem + 1024 + p.bias_bytes;                                         // [kPatchStages] raw patches
  uint8_t* wsm = patch + kPatchStages * p.patch_stage_bytes;                           // [9][BN x 16] weights
  wsm += (1024u - (smem_u32(wsm) & 1023u)) & 1023u;
  uint8_t* astage = wsm + ((p.b_bytes + 1023u) & ~1023u);                              // [stages] s2d halo tiles

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr bool fp16 = FP16;

  {
    const float bscale = epi_half_bias(p.epi) ? 0.5f : 1.0f;
    for (int i = threadIdx.x; i < p.epi.out_c; i += blockDim.x) sbias[i] = p.epi.bias[i] * bscale;
  }
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_w);
    // consumer-side barriers count WARPS: one elected lane arrives after __syncwarp(). A per-thread arrive is 32 serialized
    // shared-memory operations per warp; at 3 x 4 warps per tile they were ~380 of the ~1000 shared-memory wavefronts
    // of a tile, on the data pipe the tensor core reads its operands through (ncu: LSU + TC wavefronts at 81 %)
    for (int i = 0; i < kStemStages; ++i) { mbar_init(&sh->full[i], kStemBuilders / 32); mbar_init(&sh->empty[i], 1); }
    for (int i = 0; i < kStemAcc; ++i) { mbar_init(&sh->tmem_full[i], 1); mbar_init(&sh->tmem_empty[i], 4); }
    mbar_init(&sh->w_full, 1);
    for (int i = 0; i < kPatchStages; ++i) { mbar_init(&sh->patch_full[i], 1); mbar_init(&sh->patch_empty[i], kStemBuilders / 32); }
    tma_prefetch_desc(&map_img);
    fence_barrier_init();
  }
  if (warp == kWarpMma) {
    tmem_alloc(&sh->tmem_base, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch, bias copy) touches only
  // constants and overlaps the tail of the previous kernel; activations are read/written after the wait
  pdl_launch_dependents();
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp < kWarpMma) {
    // ===================== halo-tile builders =====================
    const int m = threadIdx.x & (kStemBuilders - 1);
    const int bgrp = threadIdx.x / kStemBuilders;
    const int kPitch = p.patch_pitch;                       // raw patch row pitch (elements)
    const int plane = p.patch_rows * kPitch;                // one image channel of the patch
    // halo pixel q = Y*pitch + X of the space-to-depth grid <- raw[c][2Y + py][2X + px]; one 32-byte operand row.
    // Everything that depends on q only is computed once (the division by the runtime pitch costs ~20 instructions).
    int src_off[2];
    uint32_t row0[2], row1[2];
    bool live[2];
#pragma unroll
    for (int rep = 0; rep < 2; ++rep) {
      const int q = m + rep * kStemBuilders;
      live[rep] = q < p.halo_pix;
      const int Y = q / p.pitch, X = q - Y * p.pitch;
      src_off[rep] = (2 * Y) * kPitch + p.lead + 2 * X;
      // SWIZZLE_32B: the 16-byte chunk index of a row is XOR-ed with address bit 7 (= bit 2 of the row index)
      const uint32_t sw = ((uint32_t)q >> 2) & 1u;
      row0[rep] = (uint32_t)q * 32u + ((0u ^ sw) << 4);
      row1[rep] = (uint32_t)q * 32u + ((1u ^ sw) << 4);
    }
    for (int it = bgrp;; it += kStemBuilderGroups) {
      const long long tl = (long long)blockIdx.x + (long long)it * gridDim.x;
      if (tl >= p.num_tiles) break;
      const int stage = it % kStemStages, ps = it % kPatchStages;
      const uint32_t phase = (uint32_t)((it / kStemStages) & 1), pphase = (uint32_t)((it / kPatchStages) & 1);
      mbar_wait(&sh->patch_full[ps], pphase);
      const TI* pt = reinterpret_cast<const TI*>(patch + (size_t)ps * p.patch_stage_bytes);
      mbar_wait(&sh->empty[stage], phase ^ 1);
      uint8_t* a0 = astage + (size_t)stage * p.a_stage_bytes;
      float fa[2][6], fb[2][6];
#pragma unroll
      for (int rep = 0; rep < 2; ++rep) {
        if (live[rep]) {
          const TI* src = pt + src_off[rep];
#pragma unroll
          for (int i = 0; i < 6; ++i) load_pair<TI>(src + (i >> 1) * plane + (i & 1) * kPitch, fa[rep][i], fb[rep][i]);
        }
      }
#pragma unroll
      for (int rep = 0; rep < 2; ++rep) {
        if (live[rep]) {
          uint32_t wd[6];
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            // fp16: pixels are fed as x/256 (exact) and the host packs 256*W: BN-folded stem weights (~W/300 for raw
            // 0..255 inputs) would otherwise fall into fp16's subnormal range and lose most of their mantissa
            if (FP16) { fa[rep][i] *= 0.00390625f; fb[rep][i] *= 0.00390625f; }
            wd[i] = pack16_t<FP16>(fa[rep][i], fb[rep][i]);
          }
          *reinterpret_cast<uint4*>(a0 + row0[rep]) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
          *reinterpret_cast<uint4*>(a0 + row1[rep]) = make_uint4(wd[4], wd[5], 0u, 0u);
        }
      }
      fence_proxy_async();                    // this thread's generic-proxy stores -> visible to the tensor core
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&sh->patch_empty[ps]);    // the warp is done with the raw patch
        mbar_arrive(&sh->full[stage]);
      }
    }
  } else if (warp == kWarpMma || (kMmaWarps == 2 && warp == kWarpMma2)) {
    // ===================== MMA issuers =====================
    // A [128 x 16] x [16 x 32] MMA is bound by the tensor core's shared-memory read of A (128 rows x 32 B at ~64 B/clk =
    // 64 clk, the math needs 16) and the issuing thread stays in tcgen05.mma for about that long, so its barrier waits
    // (~150 clk each even when the phase is already complete) were dead time of the tensor pipe: a clock64 trace
    // showed 780 clk of issue + 420 clk of waits per tile. Two warps issue alternate tiles.
    const int g = warp == kWarpMma ? 0 : 1;
    if (lane == 0) {
      if (g == 0) {
        // resident weights: nine [BN x 16] K-major tiles
        mbar_arrive_expect_tx(&sh->w_full, p.b_bytes);
        for (int tap = 0; tap < 9; ++tap) tma_load_2d(&map_w, &sh->w_full, wsm + (size_t)tap * p.w_tile_bytes, tap * 16, 0);
      }
      mbar_wait(&sh->w_full, 0);
      const uint64_t hi = ((uint64_t)p.desc_hi << 32) | (1u << 16);
      const uint32_t w16 = smem_u32(wsm) >> 4, wt16 = p.w_tile_bytes >> 4;
      const uint32_t pitch2 = (uint32_t)p.pitch * 2u;
      for (int mit = g;; mit += kMmaWarps) {
        const long long tl = (long long)blockIdx.x + (long long)mit * gridDim.x;
        if (tl >= p.num_tiles) break;
        const int stage = mit % kStemStages, as = mit % kStemAcc;
        const uint32_t phase = (uint32_t)((mit / kStemStages) & 1), aphase = (uint32_t)((mit / kStemAcc) & 1);
        mbar_wait(&sh->tmem_empty[as], aphase ^ 1);
        mbar_wait(&sh->full[stage], phase);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.BNpad);
        const uint32_t a16 = smem_u32(astage + (size_t)stage * p.a_stage_bytes) >> 4;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          // tap (r, s): halo rows shifted by r*pitch + s (32-byte rows = 2 units of 16 bytes)
          const uint64_t adesc = hi | (uint64_t)(a16 + (uint32_t)(tap / 3) * pitch2 + (uint32_t)((tap % 3) * 2));
          const uint64_t bdesc = hi | (uint64_t)(w16 + (uint32_t)tap * wt16);
          umma_f16(d_tmem, adesc, bdesc, p.idesc, (uint32_t)(tap != 0));
        }
        umma_commit(&sh->empty[stage]);
        umma_commit(&sh->tmem_full[as]);
      }
    }
  } else if (warp == kWarpTma) {
    // ===================== patch producer (TMA) =====================
    if (lane == 0) {
      pdl_wait();
      int ps = 0;
      uint32_t pphase = 0;
      for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x) {
        const int b = t / tiles_per_img;
        const int r = t - b * tiles_per_img;
        const int ty = r / p.tiles_w, tx = r - ty * p.tiles_w;
        mbar_wait(&sh->patch_empty[ps], pphase ^ 1);
        mbar_arrive_expect_tx(&sh->patch_full[ps], p.patch_tx);
        tma_load_4d(&map_img, &sh->patch_full[ps], patch + (size_t)ps * p.patch_stage_bytes,
                    2 * tx * p.tw - 2 - p.lead, 2 * ty * p.th - 2, 0, b);
        if (++ps == kPatchStages) { ps = 0; pphase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue groups =====================
    pdl_wait();
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int grp = (warp - kWarpEpi) >> 2;
    const int hl = row / p.pitch, wl = row - hl * p.pitch;
    const bool row_ok = hl < p.th && wl < p.tw;
    for (int it = grp;; it += kStemEpiGroups) {
      const long long tl = (long long)blockIdx.x + (long long)it * gridDim.x;
      if (tl >= p.num_tiles) break;
      const int t = (int)tl;
      const int as = it % kStemAcc;
      const uint32_t aphase = (uint32_t)((it / kStemAcc) & 1);
      const int b = fast_div(t, p.mul_tpi, tiles_per_img);
      const int r = t - b * tiles_per_img;
      const int ty = fast_div(r, p.mul_tw, p.tiles_w), tx = r - ty * p.tiles_w;
      const int ho = ty * p.th + hl, wo = tx * p.tw + wl;
      const bool valid = row_ok && ho < p.out_h && wo < p.out_w;
      mbar_wait(&sh->tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * p.BNpad);
      const long long pix = ((long long)b * p.out_h + ho) * p.out_w + wo;
      uint16_t* orow = (uint16_t*)p.epi.out + pix * p.epi.out_ld;
      for (int c = 0; c < p.BN; c += 32) {
        const bool two = (c + 16 < p.BN);
        uint32_t ra[16], rb[16];
        tmem_ld_x16(taddr + (uint32_t)c, ra);
        if (two) tmem_ld_x16(taddr + (uint32_t)(c + 16), rb);
        tmem_ld_wait();
        if (valid) {
          epi_tc_chunk<FP16, SILU>(p.epi, ra, sbias + c, nullptr, orow + c, b, ho, wo, c);
          if (two) epi_tc_chunk<FP16, SILU>(p.epi, rb, sbias + c + 16, nullptr, orow + c + 16, b, ho, wo, c + 16);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sh->tmem_empty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWarpMma) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct StemLaunch {
  CUtensorMap map_w, map_img;
  StemParams p;
  int grid;
  size_t smem;
  int variant;            // StemCfg<V>
};

// Two co-resident CTAs (variant 1) when they fit. Measured at 64 x 640^2 (tools/gpu_time_stem.py): 210 -> 202 us
// (fp32 image), 214 -> 201 us (uint8); a variant with one epilogue group per CTA measured 216 us. The gain is small because
// the kernel is not latency-bound after all: ncu (profiles/r2_stem.md) has the L1 data pipe saturated -- LSU wavefronts 68 %
// (shared loads of the builders and epilogues 39 %, stores 9 %) + tensor-core operand reads 34 % of the same pipe.

StemLaunch* stem_alloc() { return new (std::nothrow) StemLaunch(); }
void stem_free(StemLaunch* p) { delete p; }

int stem_prepare(const void* img, int img_dtype, const void* w, const float* bias, void* out, long long out_ld,
                 int batch, int h, int wd, int out_c, int act, int dtype, StemLaunch* L) {
  YX_REQUIRE(img && w && bias && out, YX_ERR_INVALID_ARG, "stem: null pointer");
  YX_REQUIRE(img_dtype == YX_FP32 || img_dtype == YX_U8, YX_ERR_INVALID_ARG, "stem: image dtype must be fp32 or uint8");
  YX_REQUIRE(dtype == YX_BF16 || dtype == YX_FP16, YX_ERR_INVALID_ARG, "stem: output dtype must be bf16/fp16");
  YX_REQUIRE(batch > 0 && h > 0 && wd > 0 && h % 2 == 0 && wd % 2 == 0, YX_ERR_INVALID_ARG, "stem: H, W must be even");
  YX_REQUIRE(out_c % 16 == 0 && out_c >= 16 && out_c <= 128, YX_ERR_UNSUPPORTED, "stem: out_c=%d (16..128, multiple of 16)", out_c);
  YX_REQUIRE(out_ld % 16 == 0 && out_ld >= out_c && ((uintptr_t)out & 31) == 0, YX_ERR_INVALID_ARG, "stem: out misaligned");
  YX_REQUIRE(((uintptr_t)img & 15) == 0 && ((uintptr_t)w & 15) == 0 && ((uintptr_t)bias & 15) == 0, YX_ERR_INVALID_ARG, "stem: pointer alignment");
  StemParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.img = img; p.img_dtype = img_dtype; p.batch = batch; p.h = h; p.w = wd;
  p.out_h = h / 2; p.out_w = wd / 2;
  {
    // tile choice: fewest TMA rows per image (3 * (2*th + 4) per tile), th >= 3 bounds the vertical re-read of the patch
    // rows; the box must start 16-byte aligned for every tile: 2*tw*es % 16 == 0
    const int es0 = img_dtype == YX_FP32 ? 4 : 1;
    long long best = -1;
    for (int tw = 8; tw <= 40; ++tw) {
      if ((2 * tw * es0) % 16) continue;
      const int th = 128 / (tw + 2);
      if (th < 3 && tw > 8) continue;
      const long long tiles = (long long)((p.out_w + tw - 1) / tw) * ((p.out_h + th - 1) / th);
      const long long cost = tiles * 3 * (2 * th + 4);
      if (best < 0 || cost < best) { best = cost; p.tw = tw; p.th = th; }
    }
  }
  p.pitch = p.tw + 2; p.halo_pix = (p.th + 2) * p.pitch;
  YX_REQUIRE(p.halo_pix <= 2 * kStemBuilders, YX_ERR_UNSUPPORTED, "stem: halo of %d pixels exceeds the builder groups", p.halo_pix);
  p.patch_rows = 2 * p.th + 4;
  p.tiles_w = (p.out_w + p.tw - 1) / p.tw; p.tiles_h = (p.out_h + p.th - 1) / p.th;
  p.num_tiles = batch * p.tiles_w * p.tiles_h;
  p.mul_tpi = fast_div_mul(p.tiles_w * p.tiles_h); p.mul_tw = fast_div_mul(p.tiles_w);
  p.BN = out_c;
  p.BNpad = 32; while (p.BNpad < p.BN) p.BNpad <<= 1;
  int V = 1;
  {
    // two CTAs per SM need <= 112 KB each; otherwise fall back to the single-CTA variant
    const unsigned es1 = img_dtype == YX_FP32 ? 4u : 1u;
    const unsigned per16 = 16u / es1, lead1 = per16 - 2u;
    const unsigned pitch1 = (lead1 + 2u * (unsigned)p.tw + 4u + per16 - 1u) / per16 * per16;
    const size_t patch1 = ((size_t)(3 * p.patch_rows) * pitch1 * es1 + 127u) & ~(size_t)127u;
    const size_t a1 = ((size_t)(128 + 2 * p.pitch + 2) * 32u + 1023u) & ~(size_t)1023u;
    const size_t need = 2048 + ((size_t)out_c * 4u + 1023u) / 1024u * 1024u + 2 * patch1 + 1024 + (((size_t)out_c * 32u * 9u + 1023u) & ~(size_t)1023u) + 2 * a1;
    if (need > 112 * 1024) V = 0;
  }
  L->variant = V;
  const int n_acc = V == 0 ? StemCfg<0>::kAcc : StemCfg<1>::kAcc;
  const int n_stages = V == 0 ? StemCfg<0>::kStages : StemCfg<1>::kStages;
  const int n_patch = V == 0 ? StemCfg<0>::kPatchStages : StemCfg<1>::kPatchStages;
  p.tmem_cols = (unsigned)(n_acc * p.BNpad);
  p.idesc = umma_idesc(dtype, p.BN);
  p.desc_hi = umma_desc_hi(32);                                      // 16 channels per tap: 32-byte rows
  p.bias_bytes = ((unsigned)out_c * 4u + 1023u) & ~1023u;
  p.w_tile_bytes = (unsigned)out_c * 32u;                            // one tap: [out_c x 16], a multiple of 512 B
  p.b_bytes = 9u * p.w_tile_bytes;
  EpiParams& e = p.epi;
  e.out_h = p.out_h; e.out_w = p.out_w; e.out_c = out_c; e.act = act; e.dtype = dtype; e.epilogue = YX_EPI_STORE;
  e.bias = bias; e.out = out; e.out_ld = out_ld;
  {
    const int es0 = img_dtype == YX_FP32 ? 4 : 1;
    p.lead = 16 / es0 - 2;                                          // (2 + lead) * es == 16: 16-byte aligned box start
    const int per16 = 16 / es0;
    p.patch_pitch = (p.lead + 2 * p.tw + 4 + per16 - 1) / per16 * per16;   // box width: a multiple of 16 bytes
    YX_REQUIRE(p.patch_pitch <= 256, YX_ERR_UNSUPPORTED, "stem: TMA box of %d elements", p.patch_pitch);
    p.patch_stage_bytes = ((unsigned)(3 * p.patch_rows * p.patch_pitch * es0) + 127u) & ~127u;
    p.a_stage_bytes = ((unsigned)(128 + 2 * p.pitch + 2) * 32u + 1023u) & ~1023u;   // rows addressed by the nine shifted taps
  }
  L->smem = 2048 + p.bias_bytes + (size_t)n_patch * p.patch_stage_bytes + 1024 + ((p.b_bytes + 1023u) & ~1023u) +
            (size_t)n_stages * p.a_stage_bytes;
  YX_REQUIRE(V == 0 || L->smem <= 112 * 1024, YX_ERR_UNSUPPORTED, "stem: %zu bytes of shared memory do not allow two CTAs per SM", L->smem);
  {
    // the NCHW image as a 4-D tensor [W, H, 3, B]; one box = the 40 (u8: 64) x 18 x 3 window holding a tile's patch
    const int es = img_dtype == YX_FP32 ? 4 : 1;
    const cuuint32_t bw = (cuuint32_t)p.patch_pitch;        // the box starts 16-byte aligned, `lead` pixels left of the patch
    YX_REQUIRE(((long long)wd * es) % 16 == 0, YX_ERR_UNSUPPORTED, "stem: image row pitch must be a multiple of 16 bytes");
    cuuint64_t idims[4] = {(cuuint64_t)wd, (cuuint64_t)h, 3, (cuuint64_t)batch};
    cuuint64_t istr[3] = {(cuuint64_t)wd * es, (cuuint64_t)wd * h * es, (cuuint64_t)wd * h * 3 * es};
    cuuint32_t ibox[4] = {bw, (cuuint32_t)p.patch_rows, 3, 1};
    const int rc = encode_tma(&L->map_img, tma_dtype(img_dtype), 4, img, idims, istr, ibox, nullptr, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "stem image");
    if (rc) return rc;
    p.patch_tx = bw * (cuuint32_t)p.patch_rows * 3 * es;
  }
  cuuint64_t dims[2] = {144, (cuuint64_t)out_c};
  cuuint64_t strides[1] = {288};
  cuuint32_t box[2] = {16, (cuuint32_t)out_c};
  const int rc = encode_tma(&L->map_w, tma_dtype(dtype), 2, w, dims, strides, box, nullptr, tma_swizzle(32),
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "stem W");
  if (rc) return rc;
  const int sms = num_sms() * (V == 0 ? 1 : 2);
  L->grid = p.num_tiles < sms ? p.num_tiles : sms;
  return YX_OK;
}

// [variant][uint8 image][fp16 output][SiLU]
static decltype(&stem_tc_kernel<float, false, false, 0>) const kStemKernels[2][2][2][2] = {
    {{{stem_tc_kernel<float, false, false, 0>, stem_tc_kernel<float, false, true, 0>},
      {stem_tc_kernel<float, true, false, 0>, stem_tc_kernel<float, true, true, 0>}},
     {{stem_tc_kernel<uint8_t, false, false, 0>, stem_tc_kernel<uint8_t, false, true, 0>},
      {stem_tc_kernel<uint8_t, true, false, 0>, stem_tc_kernel<uint8_t, true, true, 0>}}},
    {{{stem_tc_kernel<float, false, false, 1>, stem_tc_kernel<float, false, true, 1>},
      {stem_tc_kernel<float, true, false, 1>, stem_tc_kernel<float, true, true, 1>}},
     {{stem_tc_kernel<uint8_t, false, false, 1>, stem_tc_kernel<uint8_t, false, true, 1>},
      {stem_tc_kernel<uint8_t, true, false, 1>, stem_tc_kernel<uint8_t, true, true, 1>}}}};

int stem_launch(const StemLaunch* L, cudaStream_t stream) {
  static bool smem_set[kMaxDevices] = {};
  // the first 8 kernels are variant 0 (one CTA per SM), the other 8 variant 1 (two CTAs per SM)
  YX_CUDA(opt_in_smem(smem_set, kStemKernels, [](int i) { return i < 8 ? 200 * 1024 : 112 * 1024; }));
  const int V = L->variant;
  const auto kernel = kStemKernels[V][L->p.img_dtype != YX_FP32][L->p.epi.dtype == YX_FP16][L->p.epi.act == YX_ACT_SILU];
  YX_CUDA(launch_pdl(kernel, dim3((unsigned)L->grid), dim3((unsigned)(V == 0 ? StemCfg<0>::kThreads : StemCfg<1>::kThreads)),
                     L->smem, stream, L->map_w, L->map_img, L->p));
  return YX_OK;
}

}  // namespace yx
