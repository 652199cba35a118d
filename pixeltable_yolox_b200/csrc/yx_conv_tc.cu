// tcgen05/TMEM/TMA implicit-GEMM convolution for sm_100a.
//
// Replaces BaseConv.forward (yolox/models/network_blocks.py:27-52: conv -> BN -> SiLU) and the
// biased 1x1 prediction convs of YoloxHead (yolox/models/yolo_head.py:94-120, 140-211).
//
// GEMM view   D[M=pixels, N=out_c] = A[M, K] * W[N, K]^T,   K = taps * in_c
//   A is never materialised: for every filter tap (r, s) a TMA *tiled* 4-D load of the NHWC
//   activation tensor [C, W, H, B] with box [KC, tw, th, 1] starting at
//   (c, w0*stride + s - pad, h0*stride + r - pad, b) lands a [128 pixel rows x KC channels]
//   K-major, hardware-swizzled operand tile in shared memory. TMA zero-fills out-of-bounds
//   elements, which is exactly Conv2d's zero padding; stride-2 convs use elementStrides = 2.
//   1x1 convs use the same code with the tensor viewed as [C, M, 1, 1] (flat 128-pixel tiles).
//   W is a plain 2-D tensor [K, N] (K contiguous) loaded with box [KC, BN].
//
// One persistent CTA per SM, 6 warps:
//   warp 0      TMA producer (one elected lane): fills a ring of `stages` {A,B} slots
//   warp 1      TMEM allocator + MMA issuer (one lane): tcgen05.mma 128 x BN x 16, fp32
//               accumulators in TMEM, `acc_stages`-deep so tile i+1 is multiplied while
//               tile i is drained
//   warps 2..5  epilogue: tcgen05.ld (each warp owns the 32 TMEM lanes of its quarter),
//               bias + activation (+ residual, + 2x upsample copy, or head decode), 16-byte stores
// Synchronisation is mbarrier-only: full/empty per smem slot, tmem_full/tmem_empty per
// accumulator stage; tcgen05.commit releases slots and publishes accumulators.
#include <stdlib.h>
#include <string.h>

#include <new>

#include "yx_tc_epilogue.cuh"

namespace yx {

struct ConvTcParams {
  int tw, th;            // spatial tile; tw*th <= 128 (flat mode: tw = 128, th = 1)
  int tiles_w, tiles_h;  // tiles per image (flat mode: tiles_w = ceil(M/128), tiles_h = 1)
  int n_tiles;           // out_c / BN
  int num_tiles;         // total work items
  int BN, BNpad;         // N tile and its TMEM column pitch
  int KC;                // channels per pipeline stage (16 / 32 / 64)
  int kchunks;           // in_c / KC
  int ksize, stride, pad;
  int in_c;
  int batch;
  int flat;
  long long M;           // batch*out_h*out_w
  int stages, acc_stages;
  unsigned a_stage_bytes, stage_bytes, tx_bytes;
  unsigned desc_hi;      // upper 32 bits of the UMMA smem descriptor (SBO, version, layout)
  unsigned idesc;
  unsigned tmem_cols;
  unsigned bias_bytes;   // shared-memory copy of the bias vector (out_c floats, rounded to 1 KB)
  unsigned head_bytes;   // YX_EPI_HEAD: per-warp [32][5+nc] fp32 staging for coalesced row stores
  int epi_groups;        // 1..kMaxEpiGroups
  // ---- halo mode (3x3 stride 1): one TMA halo tile per channel chunk, the 9 taps are row-shifted
  //      UMMA descriptors into it; weights resident in smem or shared by G consecutive M tiles
  int halo;              // 1: taps x shifted descriptors (3x3 s1 with taps = 9, 1x1 with taps = 1); 2: stride-2 planes
  int taps;
  int pitch;             // accumulator rows per tile row (= tw + 2 in halo mode, = tw otherwise)
  int G;                 // M tiles per weight stage
  int m_tiles;           // real M tiles; m_tiles_pad = ceil(m_tiles / G) * G
  int a_slots;           // halo ring depth
  unsigned a_slot_bytes, a_tx_bytes, row_bytes;
  int b_resident;        // all 9*kchunks weight tiles stay in smem (n_tiles == 1)
  unsigned b_tile_bytes, b_tx_bytes, b_region_bytes;
  unsigned mul_tpi, mul_tw, mul_ntiles, mul_ohw, mul_ow;   // floor(2^32 / d) + 1 for tiles_per_img, tiles_w, n_tiles, out_h*out_w, out_w
  // ---- halo == 2 (3x3 stride 2): input viewed as [2C, W/2, H, B] (x parity folded into the channels), one
  //      halo tile per (channel chunk, y parity) "plane kind"; each kind runs a short list of MMA ops
  int s2_kinds, s2_cchunks;
  struct S2Kind {
    int ch_off;            // channel coordinate of the plane in the folded view (+ cc * 64)
    int row_off;           // first input row = 2 * y0 + row_off
    int nops;
    unsigned a_off16[4];   // (row shift * row_bytes + byte offset inside the row) >> 4
    int bk[4];             // K coordinate of the weight box (+ cc * 64)
    int ks[4];             // k-steps (16 channels each)
  } s2[4];
  EpiParams epi;
};

static constexpr int kMaxStages = 12;
static constexpr int kMaxASlots = 8;
static constexpr int kMaxAcc = 4;
static constexpr int kMaxEpiGroups = 3;           // epilogue warpgroups (4 warps each); tiles alternate between them
static constexpr int kMaxThreads = 64 + 128 * kMaxEpiGroups;

struct __align__(8) TcShared {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t tmem_full[kMaxAcc];
  uint64_t tmem_empty[kMaxAcc];
  uint64_t afull[kMaxASlots];
  uint64_t aempty[kMaxASlots];
  uint64_t bres_full;
  uint32_t tmem_base;
};


__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- halo-mode MMA issue helpers (run by the one elected lane of the MMA warp) ----
// resident weights, one M tile: 9 taps x KS k-steps, descriptors advance by compile-time constants
template <int KS, int TAPS>
__device__ __forceinline__ void halo_issue_res(uint64_t ad, uint32_t dt, uint64_t bd, uint32_t btile16, uint32_t idesc,
                                               uint32_t acc0, uint32_t rb16, uint32_t prb16) {
#pragma unroll
  for (int tap = 0; tap < TAPS; ++tap) {
    const uint64_t a = ad + (uint64_t)((uint32_t)(tap / 3) * prb16 + (uint32_t)(tap % 3) * rb16);
    const uint64_t b = bd + (uint64_t)((uint32_t)tap * btile16);
#pragma unroll
    for (int j = 0; j < KS; ++j) umma_f16(dt, a + 2 * j, b + 2 * j, idesc, (tap | j) ? 1u : acc0);
  }
}
// streamed weights (ring of `n_bs` stages), one or two M tiles sharing every weight stage
template <int KS, bool TWO, int TAPS>
__device__ __forceinline__ void halo_issue_ring(TcShared* sh, uint64_t ad0, uint64_t ad1, uint32_t dt0, uint32_t dt1,
                                                uint64_t bd0, uint32_t btile16, uint32_t idesc, uint32_t acc0,
                                                uint32_t rb16, uint32_t prb16, int& sb, uint32_t& pb, int n_bs) {
#pragma unroll
  for (int tap = 0; tap < TAPS; ++tap) {
    mbar_wait(&sh->full[sb], pb);
    tc_fence_after();
    const uint64_t sh16 = (uint64_t)((uint32_t)(tap / 3) * prb16 + (uint32_t)(tap % 3) * rb16);
    const uint64_t b = bd0 + (uint64_t)((uint32_t)sb * btile16);
    const uint32_t accf = tap ? 1u : acc0;
#pragma unroll
    for (int j = 0; j < KS; ++j) umma_f16(dt0, ad0 + sh16 + 2 * j, b + 2 * j, idesc, j ? 1u : accf);
    if (TWO) {
#pragma unroll
      for (int j = 0; j < KS; ++j) umma_f16(dt1, ad1 + sh16 + 2 * j, b + 2 * j, idesc, j ? 1u : accf);
    }
    umma_commit(&sh->empty[sb]);
    if (++sb == n_bs) { sb = 0; pb ^= 1; }
  }
}


// SILU: the activation is SiLU (compile-time: the generic activation code and its per-chunk dispatch disappear)
// HEAD: the YX_EPI_HEAD epilogue (decode + optional score filter) is its own instantiation, so its ~1 000 SASS
// instructions do not sit in the instruction cache footprint / register allocation of the activation-store kernels
template <bool FP16, bool SILU, bool HEAD>
__global__ void __launch_bounds__(kMaxThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // operand tiles need 1024-byte alignment for the 128-byte swizzle atom
  // pointer arithmetic on the __shared__ array (not an integer round trip) keeps the address space known to the
  // compiler: LDS/STS instead of generic loads for every bias / staging access
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  TcShared* sh = reinterpret_cast<TcShared*>(smem);
  float* sbias = reinterpret_cast<float*>(smem + 1024);
  float* shead = reinterpret_cast<float*>(smem + 1024 + p.bias_bytes);
  uint8_t* tiles = smem + 1024 + p.bias_bytes + p.head_bytes;
  // bias lives in shared memory: with ~200 KB of operand stages the L1 carve-out is ~0, so a
  // global bias load in the epilogue would be an L2 round trip per 16 columns
  {
    const float bscale = (epi_half_bias(p.epi) && p.epi.epilogue == YX_EPI_STORE) ? 0.5f : 1.0f;
    // head: the sigmoid channels (obj, classes) stage -log2e * bias (see the head epilogue)
    const float hscale = (HEAD && (p.epi.head_decode & 2)) ? -1.4426950408889634f : 1.0f;
    for (int i = threadIdx.x; i < p.epi.out_c; i += blockDim.x)
      sbias[i] = p.epi.bias[i] * (HEAD ? (i >= 4 ? hscale : 1.0f) : bscale);
  }

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&sh->full[i], 1);
      mbar_init(&sh->empty[i], 1);
    }
    for (int i = 0; i < p.acc_stages; ++i) {
      mbar_init(&sh->tmem_full[i], 1);
      mbar_init(&sh->tmem_empty[i], 128);
    }
    for (int i = 0; i < p.a_slots; ++i) {
      mbar_init(&sh->afull[i], 1);
      mbar_init(&sh->aempty[i], 1);
    }
    mbar_init(&sh->bres_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&sh->tmem_base, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch, bias copy) touches only
  // constants and overlaps the tail of the previous kernel; activations are read/written after the wait
  // resident weights are constants: their loads are issued BEFORE griddepcontrol.wait (each role waits itself,
  // right before its first access to activations), so they overlap the previous kernel's tail as well
  pdl_launch_dependents();

  const int num_k = p.ksize * p.ksize * p.kchunks;
  const int tiles_per_img = p.tiles_w * p.tiles_h;
  // halo mode: the CTA owns the contiguous unit range [t_begin, t_end) of the order
  //   t = (mblock * n_tiles + n_tile) * G + i,   m_tile = mblock * G + i
  // so that up to G consecutive units share one weight tile; all three roles walk it identically
  const long long T_units = (long long)p.num_tiles;
  const int t_begin = (int)(T_units * blockIdx.x / gridDim.x);
  const int t_end = (int)(T_units * (blockIdx.x + 1) / gridDim.x);
  uint8_t* const bregion = tiles;                       // weight ring or resident weights
  uint8_t* const aregion = tiles + p.b_region_bytes;    // halo ring

  if (p.halo == 2 && warp == 0) {
    // ===================== TMA producer (stride-2 planes) =====================
    if (lane == 0) {
      if (p.b_resident) {
        int nb = 0;
        for (int cc = 0; cc < p.s2_cchunks; ++cc)
          for (int k = 0; k < p.s2_kinds; ++k) nb += p.s2[k].nops;
        mbar_arrive_expect_tx(&sh->bres_full, p.b_tx_bytes * (unsigned)nb);
        nb = 0;
        for (int cc = 0; cc < p.s2_cchunks; ++cc)
          for (int k = 0; k < p.s2_kinds; ++k)
            for (int o = 0; o < p.s2[k].nops; ++o, ++nb)
              tma_load_2d(&map_b, &sh->bres_full, bregion + (size_t)nb * p.b_tile_bytes, p.s2[k].bk[o] + cc * 64, 0);
      }
      pdl_wait();
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      for (int t = t_begin; t < t_end; ++t) {
        const int n_tile = t % p.n_tiles;
        const int m_tile = t / p.n_tiles;
        const int b = m_tile / tiles_per_img;
        const int r = m_tile - b * tiles_per_img;
        const int ty = r / p.tiles_w;
        const int tx = r - ty * p.tiles_w;
        for (int cc = 0; cc < p.s2_cchunks; ++cc) {
          for (int k = 0; k < p.s2_kinds; ++k) {
            mbar_wait(&sh->aempty[sa], pa ^ 1);
            mbar_arrive_expect_tx(&sh->afull[sa], p.a_tx_bytes);
            tma_load_4d(&map_a, &sh->afull[sa], aregion + (size_t)sa * p.a_slot_bytes, p.s2[k].ch_off + cc * 64,
                        tx * p.tw - 1, 2 * ty * p.th + p.s2[k].row_off, b);
            if (++sa == p.a_slots) { sa = 0; pa ^= 1; }
            if (!p.b_resident) {
              for (int o = 0; o < p.s2[k].nops; ++o) {
                mbar_wait(&sh->empty[sb], pb ^ 1);
                mbar_arrive_expect_tx(&sh->full[sb], p.b_tx_bytes);
                tma_load_2d(&map_b, &sh->full[sb], bregion + (size_t)sb * p.b_tile_bytes, p.s2[k].bk[o] + cc * 64,
                            n_tile * p.BN);
                if (++sb == p.stages) { sb = 0; pb ^= 1; }
              }
            }
          }
        }
      }
    }
  } else if (p.halo == 2 && warp == 1) {
    // ===================== MMA issuer (stride-2 planes) =====================
    const uint32_t a0 = smem_u32(aregion) >> 4, aslot16 = p.a_slot_bytes >> 4;
    const uint32_t b0 = smem_u32(bregion) >> 4, btile16 = p.b_tile_bytes >> 4;
    const uint64_t dhi = ((uint64_t)p.desc_hi << 32) | (1u << 16);
    const uint32_t idesc = p.idesc;
    const int n_acc = p.acc_stages, n_as = p.a_slots, n_bs = p.stages;
    const bool ring = !p.b_resident;
    int sa = 0, sb = 0, as = 0;
    uint32_t pa = 0, pb = 0, pacc = 0;
    if (!ring) mbar_wait(&sh->bres_full, 0);
    for (int t = t_begin; t < t_end; ++t) {
      mbar_wait(&sh->tmem_empty[as], pacc ^ 1);
      tc_fence_after();
      const uint32_t dt = tmem_base + (uint32_t)(as * p.BNpad);
      uint32_t bres = b0;
      uint32_t accf = 0;
      for (int cc = 0; cc < p.s2_cchunks; ++cc) {
        for (int k = 0; k < p.s2_kinds; ++k) {
          mbar_wait(&sh->afull[sa], pa);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t abase = a0 + (uint32_t)sa * aslot16;
            const int nops = p.s2[k].nops;
            for (int o = 0; o < nops; ++o) {
              uint32_t bl;
              if (ring) {
                mbar_wait(&sh->full[sb], pb);
                tc_fence_after();
                bl = b0 + (uint32_t)sb * btile16;
              } else {
                bl = bres;
                bres += btile16;
              }
              const uint64_t ad = dhi | (uint64_t)(abase + p.s2[k].a_off16[o]), bd = dhi | (uint64_t)bl;
              const int ks = p.s2[k].ks[o];
              umma_f16(dt, ad, bd, idesc, accf);
              accf = 1;
              if (ks > 1) umma_f16(dt, ad + 2, bd + 2, idesc, 1u);
              if (ks > 2) { umma_f16(dt, ad + 4, bd + 4, idesc, 1u); umma_f16(dt, ad + 6, bd + 6, idesc, 1u); }
              if (ring) {
                umma_commit(&sh->empty[sb]);
                if (++sb == n_bs) { sb = 0; pb ^= 1; }
              }
            }
            umma_commit(&sh->aempty[sa]);
          }
          __syncwarp();
          accf = 1;
          if (++sa == n_as) { sa = 0; pa ^= 1; }
        }
      }
      if (elect_one_sync()) umma_commit(&sh->tmem_full[as]);
      __syncwarp();
      if (++as == n_acc) { as = 0; pacc ^= 1; }
    }
  } else if (p.halo && warp == 0) {
    // ===================== TMA producer (halo mode) =====================
    if (lane == 0) {
      if (p.b_resident) {
        mbar_arrive_expect_tx(&sh->bres_full, p.b_tx_bytes * (unsigned)(p.taps * p.kchunks));
        for (int tap = 0; tap < p.taps; ++tap)
          for (int c = 0; c < p.kchunks; ++c)
            tma_load_2d(&map_b, &sh->bres_full, bregion + (size_t)(c * p.taps + tap) * p.b_tile_bytes,
                        tap * p.in_c + c * p.KC, 0);
      }
      pdl_wait();
      int ca = 0, sb = 0;
      uint32_t pb = 0;
      for (int t = t_begin; t < t_end;) {
        const int i0 = t % p.G;
        const int u = t / p.G;
        const int n_tile = u % p.n_tiles;
        const int mblock = u / p.n_tiles;
        int g = p.G - i0;
        if (g > t_end - t) g = t_end - t;
        for (int c = 0; c < p.kchunks; ++c) {
          for (int i = 0; i < g; ++i, ++ca) {
            const int m_tile = mblock * p.G + i0 + i;
            const int b = m_tile / tiles_per_img;          // >= batch for padding tiles: TMA zero-fills
            const int r = m_tile - b * tiles_per_img;
            const int ty = r / p.tiles_w;
            const int tx = r - ty * p.tiles_w;
            const int slot = ca % p.a_slots;
            mbar_wait(&sh->aempty[slot], (uint32_t)(((ca / p.a_slots) & 1) ^ 1));
            mbar_arrive_expect_tx(&sh->afull[slot], p.a_tx_bytes);
            if (p.flat)
              tma_load_4d(&map_a, &sh->afull[slot], aregion + (size_t)slot * p.a_slot_bytes, c * p.KC, m_tile * 128, 0, 0);
            else
              tma_load_4d(&map_a, &sh->afull[slot], aregion + (size_t)slot * p.a_slot_bytes, c * p.KC,
                          tx * p.tw - 1, ty * p.th - 1, b);
          }
          if (!p.b_resident) {
            for (int tap = 0; tap < p.taps; ++tap) {
              mbar_wait(&sh->empty[sb], pb ^ 1);
              mbar_arrive_expect_tx(&sh->full[sb], p.b_tx_bytes);
              tma_load_2d(&map_b, &sh->full[sb], bregion + (size_t)sb * p.b_tile_bytes, tap * p.in_c + c * p.KC,
                          n_tile * p.BN);
              if (++sb == p.stages) { sb = 0; pb ^= 1; }
            }
          }
        }
        t += g;
      }
    }
  } else if (p.halo && warp == 1) {
    // ===================== MMA issuer (halo mode) =====================
    // The whole warp walks the (warp-uniform) loop and one elected lane issues: a divergent single-thread
    // loop costs ~5 cycles per scalar instruction, which is more than a 128xNx16 MMA for N <= 64.
    const uint32_t rb16 = p.row_bytes >> 4;
    const uint32_t prb16 = (uint32_t)p.pitch * rb16;
    const uint32_t a0 = smem_u32(aregion) >> 4, aslot16 = p.a_slot_bytes >> 4;
    const uint32_t b0 = smem_u32(bregion) >> 4, btile16 = p.b_tile_bytes >> 4;
    const uint64_t dhi = ((uint64_t)p.desc_hi << 32) | (1u << 16);   // LBO = 1 in the low word
    const uint32_t idesc = p.idesc;
    const int ksteps = p.KC >> 4;
    const int G = p.G, n_acc = p.acc_stages, n_as = p.a_slots, n_bs = p.stages, kch = p.kchunks, taps = p.taps;
    const bool ring = !p.b_resident;
    int sa = 0, sb = 0, as = 0, i0 = t_begin % G;
    uint32_t pa = 0, pb = 0, pacc = 0;
    if (!ring) mbar_wait(&sh->bres_full, 0);
    for (int t = t_begin; t < t_end;) {
      int g = G - i0;
      if (g > t_end - t) g = t_end - t;
      i0 = 0;
      uint32_t dt0, dt1 = 0;
      const int st0 = as;
      mbar_wait(&sh->tmem_empty[as], pacc ^ 1);
      dt0 = tmem_base + (uint32_t)(as * p.BNpad);
      if (++as == n_acc) { as = 0; pacc ^= 1; }
      const int st1 = as;
      if (g > 1) {
        mbar_wait(&sh->tmem_empty[as], pacc ^ 1);
        dt1 = tmem_base + (uint32_t)(as * p.BNpad);
        if (++as == n_acc) { as = 0; pacc ^= 1; }
      }
      tc_fence_after();
      uint32_t bres = b0;
      for (int c = 0; c < kch; ++c) {
        const int sl0 = sa;
        mbar_wait(&sh->afull[sa], pa);
        const uint32_t al0 = a0 + (uint32_t)sa * aslot16;
        if (++sa == n_as) { sa = 0; pa ^= 1; }
        const int sl1 = sa;
        uint32_t al1 = 0;
        if (g > 1) {
          mbar_wait(&sh->afull[sa], pa);
          al1 = a0 + (uint32_t)sa * aslot16;
          if (++sa == n_as) { sa = 0; pa ^= 1; }
        }
        if (elect_one_sync()) {
          // one straight-line block per chunk: descriptors advance by constants, no branches between MMAs
          const uint64_t ad0 = dhi | (uint64_t)al0, ad1 = dhi | (uint64_t)al1;
          const uint32_t acc0 = (uint32_t)(c != 0);
          if (ring) {
#define YX_RING(KS, TWO, TAPS) halo_issue_ring<KS, TWO, TAPS>(sh, ad0, ad1, dt0, dt1, dhi | (uint64_t)b0, btile16, idesc, acc0, rb16, prb16, sb, pb, n_bs)
#define YX_RING_T(TWO, TAPS) do { if (ksteps == 4) YX_RING(4, TWO, TAPS); else if (ksteps == 2) YX_RING(2, TWO, TAPS); else YX_RING(1, TWO, TAPS); } while (0)
            if (taps == 9) { if (g > 1) YX_RING_T(true, 9); else YX_RING_T(false, 9); }
            else { if (g > 1) YX_RING_T(true, 1); else YX_RING_T(false, 1); }
#undef YX_RING_T
#undef YX_RING
          } else {
            const uint64_t bd = dhi | (uint64_t)bres;
#define YX_RES(KS, TAPS) halo_issue_res<KS, TAPS>(ad0, dt0, bd, btile16, idesc, acc0, rb16, prb16)
            if (taps == 9) { if (ksteps == 4) YX_RES(4, 9); else if (ksteps == 2) YX_RES(2, 9); else YX_RES(1, 9); }
            else { if (ksteps == 4) YX_RES(4, 1); else if (ksteps == 2) YX_RES(2, 1); else YX_RES(1, 1); }
#undef YX_RES
          }
          umma_commit(&sh->aempty[sl0]);
          if (g > 1) umma_commit(&sh->aempty[sl1]);
        }
        __syncwarp();
        bres += (uint32_t)taps * btile16;
      }
      if (elect_one_sync()) {
        umma_commit(&sh->tmem_full[st0]);
        if (g > 1) umma_commit(&sh->tmem_full[st1]);
      }
      __syncwarp();
      t += g;
    }
  } else if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      pdl_wait();
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x) {
        const int n_tile = t % p.n_tiles;
        const int m_tile = t / p.n_tiles;
        int b, x0, y0;
        if (p.flat) {
          b = 0; y0 = 0; x0 = m_tile * 128;
        } else {
          b = m_tile / tiles_per_img;
          const int r = m_tile - b * tiles_per_img;
          const int ty = r / p.tiles_w;
          const int tx = r - ty * p.tiles_w;
          x0 = tx * p.tw * p.stride - p.pad;
          y0 = ty * p.th * p.stride - p.pad;
        }
        // taps and channel chunks as nested loops (no division per stage)
        for (int fr = 0, kb = 0; fr < p.ksize; ++fr) {
          for (int fs = 0; fs < p.ksize; ++fs, kb += p.in_c) {
            for (int cc = 0; cc < p.kchunks; ++cc) {
              mbar_wait(&sh->empty[stage], phase ^ 1);
              mbar_arrive_expect_tx(&sh->full[stage], p.tx_bytes);
              uint8_t* sa = tiles + (size_t)stage * p.stage_bytes;
              tma_load_4d(&map_a, &sh->full[stage], sa, cc * p.KC, x0 + fs, y0 + fr, b);
              tma_load_2d(&map_b, &sh->full[stage], sa + p.a_stage_bytes, kb + cc * p.KC, n_tile * p.BN);
              if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (per-tap ring) =====================
    // warp-uniform loop, one elected lane issues; ~12 instructions + KC/16 MMAs per stage
    const uint64_t dhi = ((uint64_t)p.desc_hi << 32) | (1u << 16);
    const uint32_t t16 = smem_u32(tiles) >> 4, stage16 = p.stage_bytes >> 4, boff16 = p.a_stage_bytes >> 4;
    const uint32_t idesc = p.idesc;
    const int ksteps = p.KC / 16, n_st = p.stages, n_acc = p.acc_stages;
    int stage = 0, as = 0;
    uint32_t phase = 0, aphase = 0;
    for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x) {
      mbar_wait(&sh->tmem_empty[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.BNpad);
      for (int kt = 0; kt < num_k; ++kt) {
        mbar_wait(&sh->full[stage], phase);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint64_t ad = dhi | (uint64_t)(t16 + (uint32_t)stage * stage16);
          const uint64_t bd = ad + boff16;
          const uint32_t acc0 = (uint32_t)(kt != 0);
          umma_f16(d_tmem, ad, bd, idesc, acc0);
          if (ksteps > 1) umma_f16(d_tmem, ad + 2, bd + 2, idesc, 1u);
          if (ksteps > 2) { umma_f16(d_tmem, ad + 4, bd + 4, idesc, 1u); umma_f16(d_tmem, ad + 6, bd + 6, idesc, 1u); }
          umma_commit(&sh->empty[stage]);  // slot is free once these MMAs have read it
        }
        __syncwarp();
        if (++stage == n_st) { stage = 0; phase ^= 1; }
      }
      if (elect_one_sync()) umma_commit(&sh->tmem_full[as]);   // accumulator complete -> epilogue
      __syncwarp();
      if (++as == n_acc) { as = 0; aphase ^= 1; }
    }
  } else {
    // ===================== epilogue (warps 2.., in groups of 4) =====================
    // With one epilogue warp per scheduler every dependent instruction stalls the SM sub-partition;
    // group g drains the tiles it, it+G, ... of this CTA so that G tiles are in the epilogue at once.
    pdl_wait();                               // residual reads / output writes must follow the previous kernel
    const int quarter = warp & 3;            // TMEM lanes [32*quarter, 32*quarter+32)
    const int row = quarter * 32 + lane;     // accumulator row = pixel inside the tile
    const int grp = (warp - 2) >> 2;
    const int out_hw = p.epi.out_h * p.epi.out_w;
    // everything that does not depend on the tile is decoded once; per tile there is no integer division
    int hl0 = 0, wl0 = 0;
    if (!p.flat) { hl0 = row / p.pitch; wl0 = row - hl0 * p.pitch; }
    const bool row_ok = p.flat || (hl0 < p.th && wl0 < p.tw);
    const bool need_coords = (p.flat && (p.epi.ups != nullptr || HEAD)) || p.epi.shuf_c != 0;
    int as = grp % p.acc_stages;
    uint32_t aphase = (uint32_t)((grp / p.acc_stages) & 1);
    for (int it = grp;; it += p.epi_groups) {
      int n_tile, m_tile;
      if (p.halo) {
        const int t = t_begin + it;
        if (t >= t_end) break;
        const int u = p.G == 2 ? (t >> 1) : t;
        const int mb = fast_div(u, p.mul_ntiles, p.n_tiles);
        n_tile = u - mb * p.n_tiles;
        m_tile = p.G == 2 ? (mb * 2 + (t & 1)) : mb;
      } else {
        const long long tl = (long long)blockIdx.x + (long long)it * gridDim.x;
        if (tl >= p.num_tiles) break;
        m_tile = fast_div((int)tl, p.mul_ntiles, p.n_tiles);
        n_tile = (int)tl - m_tile * p.n_tiles;
      }
      int b = 0, ho = 0, wo = 0;
      long long pix;
      bool valid;
      if (p.flat) {
        const long long m = (long long)m_tile * 128 + row;
        valid = m < p.M;
        pix = valid ? m : 0;
        if (need_coords) {
          b = fast_div((int)pix, p.mul_ohw, out_hw);
          const int r = (int)pix - b * out_hw;
          ho = fast_div(r, p.mul_ow, p.epi.out_w);
          wo = r - ho * p.epi.out_w;
        }
      } else {
        b = fast_div(m_tile, p.mul_tpi, tiles_per_img);
        const int r = m_tile - b * tiles_per_img;
        const int ty = fast_div(r, p.mul_tw, p.tiles_w);
        const int tx = r - ty * p.tiles_w;
        ho = ty * p.th + hl0;
        wo = tx * p.tw + wl0;
        valid = row_ok && (ho < p.epi.out_h) && (wo < p.epi.out_w) && (b < p.batch);
        pix = ((long long)b * p.epi.out_h + ho) * p.epi.out_w + wo;
      }
      mbar_wait(&sh->tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * p.BNpad);
      const float* tbias = sbias + n_tile * p.BN;
      if constexpr (HEAD) {
        // ---- head: decode/sigmoid in registers, stage the warp's 32 rows in shared memory, then
        //      write each [5+nc] fp32 row with coalesced 128-byte stores
        const int nch = 5 + p.epi.head_nc;
        float* wstage = shead + (size_t)(warp - 2) * 32 * nch;   // one staging slab per epilogue warp
        // sigmoid(x) = 1 / (1 + 2^(-x*log2e)): the staged bias of the sigmoid channels is pre-multiplied by
        // -log2e, so each element is FFMA + EX2 + FADD + RCP (ex2/rcp.approx: ~1e-7 relative) + one shared store
        const bool dec_box = (p.epi.head_decode & 1) != 0, dec_sig = (p.epi.head_decode & 2) != 0;
        const float sgn = dec_sig ? -1.4426950408889634f : 1.0f;
        float* wrow = wstage + lane * nch;
        // 16 channels at a time: the biases are read first (four LDS.128) and all 16 values are finished before the
        // first store. Interleaving `wrow[j] = ...` with `tbias[j]` reads made every element a serial
        // LDS -> FFMA -> EX2 -> FADD -> RCP -> STS chain (shared stores and loads may alias, so they are kept in
        // order): ncu showed the epilogue warps ~95 % stalled on the short scoreboard at ~9 clk per instruction.
        // fused score filter (stage 1 of yx_postprocess, filter_kernel in yx_postprocess.cu). Arg-max over the class
        // confidences with torch.max's rule (first maximum wins; a NaN wins and the first NaN is reported): sigmoid
        // outputs are +0..1 or the canonical NaN, so their bit patterns compared as signed integers order exactly that way
        // and a pairwise tree that keeps the LEFT operand on ties reports the first index. Since score = obj * conf <= obj,
        // a warp none of whose anchors has obj >= conf_thre skips the arg-max altogether (the usual case).
        const bool filt = p.epi.head_cand != nullptr;
        bool need = false;              // warp-uniform
        float obj = 0.0f;
        int best_bits = -1, best_i = 0;
        auto sig16 = [&](const uint32_t (&r)[16], int cc, int lo) {
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 bb = *reinterpret_cast<const float4*>(tbias + cc + j);
            v[j + 0] = fmaf(__uint_as_float(r[j + 0]), sgn, bb.x);
            v[j + 1] = fmaf(__uint_as_float(r[j + 1]), sgn, bb.y);
            v[j + 2] = fmaf(__uint_as_float(r[j + 2]), sgn, bb.z);
            v[j + 3] = fmaf(__uint_as_float(r[j + 3]), sgn, bb.w);
          }
          if (dec_sig) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = ex2_approx(v[j]);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = rcp_approx(1.0f + v[j]);
          }
          const bool full = cc + 16 <= nch;
          if (full) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (j >= lo) wrow[cc + j] = v[j];
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (j >= lo && cc + j < nch) wrow[cc + j] = v[j];
          }
          if (filt) {
            if (lo) {                            // first chunk: channel 4 is the objectness
              obj = v[4];
              need = __any_sync(0xffffffffu, valid && !(obj < p.epi.head_conf));
            }
            if (need) {
              const int first = lo ? 5 : 0;      // classes start at channel 5
              int kb[16], ki[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                kb[j] = (j >= first && (full || cc + j < nch)) ? __float_as_int(v[j]) : -1;
                ki[j] = j;
              }
#pragma unroll
              for (int st = 1; st < 16; st <<= 1) {
#pragma unroll
                for (int j = 0; j < 16; j += 2 * st) {
                  const bool t = kb[j + st] > kb[j];
                  kb[j] = t ? kb[j + st] : kb[j];
                  ki[j] = t ? ki[j + st] : ki[j];
                }
              }
              if (kb[0] > best_bits) { best_bits = kb[0]; best_i = cc - 5 + ki[0]; }
            }
          }
        };
        float x0, x1, x2, x3;
        {
          // channels 0..15: box (cx, cy, w, h) then obj / first classes
          uint32_t raw[16];
          tmem_ld_x16(taddr, raw);
          tmem_ld_wait();
          const float4 b0 = *reinterpret_cast<const float4*>(tbias);
          x0 = __uint_as_float(raw[0]) + b0.x; x1 = __uint_as_float(raw[1]) + b0.y;
          x2 = __uint_as_float(raw[2]) + b0.z; x3 = __uint_as_float(raw[3]) + b0.w;
          if (dec_box) {
            x0 = (x0 + (float)wo) * p.epi.head_stride;
            x1 = (x1 + (float)ho) * p.epi.head_stride;
            x2 = __expf(x2) * p.epi.head_stride;
            x3 = __expf(x3) * p.epi.head_stride;
          }
          sig16(raw, 0, 4);
        }
        for (int c = 16; c < p.BN; c += 32) {
          const bool two = (c + 16 < p.BN);
          uint32_t ra[16], rb[16];
          tmem_ld_x16(taddr + (uint32_t)c, ra);
          if (two) tmem_ld_x16(taddr + (uint32_t)(c + 16), rb);
          tmem_ld_wait();
          if (c < nch) sig16(ra, c, 0);
          if (two && c + 16 < nch) sig16(rb, c + 16, 0);
        }
        const long long arow = valid ? ((long long)b * p.epi.head_anchors + p.epi.head_anchor_off +
                                        (long long)ho * p.epi.out_w + wo) : -1;
        if (filt || p.epi.head_xyxy) {
          // boxes.py:32-37 and :44-50 in the filter kernel's arithmetic (round-to-nearest intrinsics: no FMA contraction)
          const float hw2 = __fdiv_rn(x2, 2.0f), hh2 = __fdiv_rn(x3, 2.0f);
          const float4 box = make_float4(__fsub_rn(x0, hw2), __fsub_rn(x1, hh2), __fadd_rn(x0, hw2), __fadd_rn(x1, hh2));
          if (p.epi.head_xyxy) { x0 = box.x; x1 = box.y; x2 = box.z; x3 = box.w; }
          if (filt && need) {
            const float best = __int_as_float(best_bits);
            const float score = __fmul_rn(obj, best);
            const bool pass = valid && score >= p.epi.head_conf;
            if (pass) {          // rows of anchors below the threshold are never read by the NMS stage
              float4* crow = reinterpret_cast<float4*>(p.epi.head_cand + arow * 8);
              crow[0] = box;
              crow[1] = make_float4(obj, best, (float)best_i, score);
            }
            // a warp's rows may straddle two images (flat 1x1 tiles): aggregate per image of the first passing lane,
            // the rare lanes of the other image append on their own
            const unsigned bal = __ballot_sync(0xffffffffu, pass);
            if (bal) {
              const int leader = __ffs(bal) - 1;
              const int bl = __shfl_sync(0xffffffffu, b, leader);
              const unsigned same = __ballot_sync(0xffffffffu, pass && b == bl);
              int base = 0;
              if (lane == leader) base = atomicAdd(&p.epi.head_counts[bl], __popc(same));
              base = __shfl_sync(0xffffffffu, base, leader);
              if (pass) {
                const int a = (int)(arow - (long long)b * p.epi.head_anchors);
                const float sc = (score == 0.0f) ? 0.0f : score;  // -0 -> +0
                const unsigned long long key = ((unsigned long long)(~orderable_f32(sc)) << 32) | (unsigned long long)(unsigned)a;
                const int pos = (b == bl) ? base + __popc(same & ((1u << lane) - 1)) : atomicAdd(&p.epi.head_counts[b], 1);
                p.epi.head_keys[(long long)b * p.epi.head_anchors + pos] = key;
              }
            }
          }
        }
        wrow[0] = x0; wrow[1] = x1; wrow[2] = x2; wrow[3] = x3;
        // accumulators are in registers/smem now: hand the TMEM stage back before the slow stores
        tc_fence_before();
        mbar_arrive(&sh->tmem_empty[as]);
        __syncwarp();
        const long long a0 = __shfl_sync(0xffffffffu, arow, 0);
        const bool contiguous = __all_sync(0xffffffffu, arow == a0 + lane) && ((a0 * nch) & 3) == 0 && ((32 * nch) & 3) == 0;
        if (contiguous) {
          // the warp's 32 rows are one contiguous, 16-byte aligned block of 32*(5+nc) floats
          float4* dst = reinterpret_cast<float4*>(p.epi.head_out + a0 * nch);
          const float4* src = reinterpret_cast<const float4*>(wstage);
          // four 16-byte rows in flight per lane (loads first, then stores)
          const int n4 = 8 * nch;
          int i = lane;
          for (; i + 96 < n4; i += 128) {
            const float4 t0 = src[i], t1 = src[i + 32], t2 = src[i + 64], t3 = src[i + 96];
            dst[i] = t0; dst[i + 32] = t1; dst[i + 64] = t2; dst[i + 96] = t3;
          }
          for (; i < n4; i += 32) dst[i] = src[i];
        } else {
          for (int r = 0; r < 32; ++r) {
            const long long ar = __shfl_sync(0xffffffffu, arow, r);
            if (ar < 0) continue;
            float* dst = p.epi.head_out + ar * nch;
            const float* src = wstage + r * nch;
            for (int ch = lane; ch < nch; ch += 32) dst[ch] = src[ch];
          }
        }
        __syncwarp();
        as += p.epi_groups;
        while (as >= p.acc_stages) { as -= p.acc_stages; aphase ^= 1; }
      } else {
      // ---- activation store: two 16-column TMEM loads in flight, residual prefetched before the
      //      wait, one 256-bit store per thread per 16 columns (a full 32-byte sector)
      uint16_t* orow = (uint16_t*)p.epi.out + pix * p.epi.out_ld + n_tile * p.BN;
      // second destination: channels >= out2_begin (the stacked CSP GEMM writes x_1 and x_2 to two dense buffers)
      uint16_t* orow2 = p.epi.out2 ? (uint16_t*)p.epi.out2 + pix * p.epi.out2_ld + (n_tile * p.BN - p.epi.out2_begin) : nullptr;
      const int split = orow2 ? p.epi.out2_begin - n_tile * p.BN : 0x7fffffff;
      const uint16_t* rrow = p.epi.res ? (const uint16_t*)p.epi.res + pix * p.epi.res_ld + n_tile * p.BN : nullptr;
      // depth-to-space store (dgrad of a stride-2 conv as one sub-pixel conv): channel block q goes to pixel (2y + q/2, 2x + q%2)
      const int sc = p.epi.shuf_c;
      auto dst_of = [&](int c) -> uint16_t* {
        if (!sc) return (c >= split ? orow2 : orow) + c;
        const int cg = n_tile * p.BN + c;
        const int q = cg >= 2 * sc ? (cg >= 3 * sc ? 3 : 2) : (cg >= sc ? 1 : 0);
        const long long up = ((long long)b * 2 * p.epi.out_h + 2 * ho + (q >> 1)) * (2 * p.epi.out_w) + 2 * wo + (q & 1);
        return (uint16_t*)p.epi.out + up * p.epi.out_ld + (cg - q * sc);
      };
      for (int c = 0; c < p.BN; c += 32) {
        const bool two = (c + 16 < p.BN);
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
          epi_tc_chunk<FP16, SILU>(p.epi, ra, tbias + c, rrow ? qa : nullptr, dst_of(c), b, ho, wo, n_tile * p.BN + c);
          if (two)
            epi_tc_chunk<FP16, SILU>(p.epi, rb, tbias + c + 16, rrow ? qb : nullptr, dst_of(c + 16), b, ho, wo, n_tile * p.BN + c + 16);
        }
      }
      tc_fence_before();
      mbar_arrive(&sh->tmem_empty[as]);
      as += p.epi_groups;
      while (as >= p.acc_stages) { as -= p.acc_stages; aphase ^= 1; }
      }   // !HEAD
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct ConvTcLaunch {
  CUtensorMap map_a, map_b;
  ConvTcParams p;
  int grid;
  int ctas;              // co-resident CTAs per SM the launch was sized for
  size_t smem;
};

int fill_epi_params(const yx_conv_desc* d, EpiParams* e) {
  YX_REQUIRE(d->out_c % 16 == 0, YX_ERR_INVALID_ARG, "conv: out_c=%d must be a multiple of 16", d->out_c);
  e->out_h = d->out_h; e->out_w = d->out_w; e->out_c = d->out_c;
  e->act = d->act; e->dtype = d->dtype; e->epilogue = d->epilogue;
  e->bias = d->bias;
  YX_REQUIRE(d->bias != nullptr, YX_ERR_INVALID_ARG, "conv: bias is null");
  YX_REQUIRE(((uintptr_t)d->bias & 15) == 0, YX_ERR_INVALID_ARG, "conv: bias must be 16-byte aligned");
  e->out = d->out; e->out_ld = d->out_ld;
  e->res = d->res; e->res_ld = d->res_ld;
  e->ups = d->ups; e->ups_ld = d->ups_ld;
  e->out2 = d->out2; e->out2_ld = d->out2_ld; e->out2_begin = d->out2_begin;
  e->head_out = d->head_out;
  e->head_anchors = d->head_anchors; e->head_anchor_off = d->head_anchor_off;
  e->head_nc = d->head_nc; e->head_decode = d->head_decode; e->head_stride = d->head_stride;
  e->head_cand = d->head_cand; e->head_keys = (unsigned long long*)d->head_keys; e->head_counts = d->head_counts;
  e->head_conf = d->head_conf_thre; e->head_xyxy = d->head_xyxy;
  e->shuf_c = d->shuffle2_c;
  if (d->epilogue == YX_EPI_HEAD) {
    YX_REQUIRE(d->head_out != nullptr, YX_ERR_INVALID_ARG, "conv(head): head_out is null");
    YX_REQUIRE(5 + d->head_nc <= d->out_c, YX_ERR_INVALID_ARG, "conv(head): out_c=%d < 5+nc=%d", d->out_c, 5 + d->head_nc);
    if (d->head_cand || d->head_xyxy) {
      YX_REQUIRE(d->dtype != YX_FP32, YX_ERR_UNSUPPORTED, "conv(head): the fused score filter exists on the tcgen05 path only");
      YX_REQUIRE(d->head_decode == 3, YX_ERR_INVALID_ARG, "conv(head): the fused score filter needs head_decode == 3");
      YX_REQUIRE(d->head_nc >= 1, YX_ERR_INVALID_ARG, "conv(head): the fused score filter needs at least one class");
      if (d->head_cand)
        YX_REQUIRE(d->head_keys && d->head_counts && ((uintptr_t)d->head_cand & 15) == 0, YX_ERR_INVALID_ARG,
                   "conv(head): head_cand needs head_keys, head_counts and 16-byte alignment");
    }
  } else {
    YX_REQUIRE(d->epilogue == YX_EPI_STORE, YX_ERR_INVALID_ARG, "conv: unknown epilogue %d", d->epilogue);
    YX_REQUIRE(d->out != nullptr, YX_ERR_INVALID_ARG, "conv: out is null");
    const int al = d->dtype == YX_FP32 ? 4 : 8;
    YX_REQUIRE(d->out_ld % al == 0 && ((uintptr_t)d->out & 15) == 0, YX_ERR_INVALID_ARG,
               "conv: out must be 16-byte aligned with out_ld %% %d == 0", al);
    if (d->shuffle2_c) {
      YX_REQUIRE(d->dtype != YX_FP32, YX_ERR_UNSUPPORTED, "conv: the depth-to-space store exists on the tcgen05 path only");
      YX_REQUIRE(d->shuffle2_c > 0 && d->shuffle2_c % 16 == 0 && d->out_c == 4 * d->shuffle2_c && d->out_ld >= d->shuffle2_c &&
                     !d->res && !d->ups && !d->out2,
                 YX_ERR_INVALID_ARG, "conv: shuffle2_c must be a multiple of 16 with out_c == 4 * shuffle2_c, no res / ups / out2");
    } else
    YX_REQUIRE(d->out_ld >= (d->out2 ? d->out2_begin : d->out_c), YX_ERR_INVALID_ARG, "conv: out_ld < out_c");
    if (d->out2) YX_REQUIRE(d->out2_ld >= d->out_c - d->out2_begin, YX_ERR_INVALID_ARG, "conv: out2_ld too small");
    if (d->res) YX_REQUIRE(d->res_ld % al == 0 && ((uintptr_t)d->res & 15) == 0, YX_ERR_INVALID_ARG, "conv: res misaligned");
    if (d->ups) YX_REQUIRE(d->ups_ld % al == 0 && ((uintptr_t)d->ups & 15) == 0, YX_ERR_INVALID_ARG, "conv: ups misaligned");
    if (d->out2)
      YX_REQUIRE(d->out2_ld % 16 == 0 && ((uintptr_t)d->out2 & 31) == 0 && d->out2_begin % 16 == 0 && d->out2_begin > 0 &&
                     d->out2_begin < d->out_c && !d->ups && !d->res,
                 YX_ERR_INVALID_ARG, "conv: out2 needs 32-byte alignment, out2_begin %% 16 == 0 inside (0, out_c), no res/ups");
  }
  return YX_OK;
}

int validate_conv_geometry(const yx_conv_desc* d) {
  YX_REQUIRE(d != nullptr, YX_ERR_INVALID_ARG, "conv: null descriptor");
  YX_REQUIRE(d->ksize == 1 || d->ksize == 3, YX_ERR_UNSUPPORTED, "conv: ksize=%d (only 1 and 3)", d->ksize);
  YX_REQUIRE(d->stride == 1 || d->stride == 2, YX_ERR_UNSUPPORTED, "conv: stride=%d (only 1 and 2)", d->stride);
  YX_REQUIRE(d->batch > 0 && d->in_h > 0 && d->in_w > 0, YX_ERR_INVALID_ARG, "conv: empty input");
  const int pad = (d->ksize - 1) / 2;
  const int oh = (d->in_h + 2 * pad - d->ksize) / d->stride + 1;
  const int ow = (d->in_w + 2 * pad - d->ksize) / d->stride + 1;
  YX_REQUIRE(oh == d->out_h && ow == d->out_w, YX_ERR_INVALID_ARG,
             "conv: out %dx%d inconsistent with in %dx%d k%d s%d (expected %dx%d)", d->out_h, d->out_w,
             d->in_h, d->in_w, d->ksize, d->stride, oh, ow);
  YX_REQUIRE(d->in_c % 16 == 0 && d->in_c > 0, YX_ERR_INVALID_ARG, "conv: in_c=%d must be a multiple of 16", d->in_c);
  YX_REQUIRE(d->in != nullptr && d->w != nullptr, YX_ERR_INVALID_ARG, "conv: null in/w");
  YX_REQUIRE(d->in_ld >= d->in_c, YX_ERR_INVALID_ARG, "conv: in_ld < in_c");
  return YX_OK;
}

// CTAs per SM for this layer. Measured on the yolox_s step (B = 64, us per launch, 1 -> 2 CTAs):
// two co-resident CTAs pay off where a tile is a handful of MMAs followed by a long epilogue and the single CTA's pipeline
// is latency-bound -- the stride-2 plane layers with few input channels (32->64 @160: 142 -> 117, 64->128 @80: 78 -> 74) and
// the 3x3 layers on the 20x20 maps (256->256: 43 -> 39, 128->256: 29 -> 27). They lose where one CTA already keeps the
// tensor pipe busy (head 3x3 @80x80: 178 -> 203, 3x3 128->128 @40x40: 37 -> 41) or where halving the shared memory evicts the
// resident weights (1x1 1024->512: 31 -> 37). YX_CTAS_PER_SM=1|2 forces a setting (a test hook).
static int conv_ctas_per_sm(const yx_conv_desc* d) {
  if (d->epilogue == YX_EPI_HEAD) return 1;                   // the head staging slabs need the shared memory
  if (const char* e = getenv("YX_CTAS_PER_SM")) { const int v = atoi(e); if (v == 1 || v == 2) return v; }
  if (d->ksize == 3 && d->stride == 2 && d->in_c <= 64) return 2;
  if (d->ksize == 3 && d->stride == 1 && d->out_h * d->out_w <= 400 && d->in_c >= 128) return 2;
  return 1;
}

static int largest_divisor_tile(int n, int cap) {
  // largest multiple-of-16 divisor of n that is <= cap
  for (int t = cap - cap % 16; t >= 16; t -= 16)
    if (n % t == 0) return t;
  return 16;
}

static int conv_tc_prepare_mode(const yx_conv_desc* d, ConvTcLaunch* L, bool allow_s2, bool allow_flat = true) {
  int rc = validate_conv_geometry(d);
  if (rc) return rc;
  YX_REQUIRE(d->dtype == YX_BF16 || d->dtype == YX_FP16, YX_ERR_INVALID_ARG, "conv_tc: dtype must be bf16/fp16");
  YX_REQUIRE(d->in_ld % 8 == 0 && ((uintptr_t)d->in & 15) == 0 && ((uintptr_t)d->w & 15) == 0,
             YX_ERR_INVALID_ARG, "conv_tc: in/w must be 16-byte aligned, in_ld %% 8 == 0");
  if (d->epilogue == YX_EPI_STORE) {
    // the epilogue moves 16 channels (32 bytes) per instruction
    YX_REQUIRE(d->out_ld % 16 == 0 && ((uintptr_t)d->out & 31) == 0, YX_ERR_INVALID_ARG,
               "conv_tc: out must be 32-byte aligned with out_ld %% 16 == 0");
    if (d->res) YX_REQUIRE(d->res_ld % 16 == 0 && ((uintptr_t)d->res & 31) == 0, YX_ERR_INVALID_ARG, "conv_tc: res must be 32-byte aligned");
    if (d->ups) YX_REQUIRE(d->ups_ld % 16 == 0 && ((uintptr_t)d->ups & 31) == 0, YX_ERR_INVALID_ARG, "conv_tc: ups must be 32-byte aligned");
  }
  ConvTcParams& p = L->p;
  memset(&p, 0, sizeof(p));
  rc = fill_epi_params(d, &p.epi);
  if (rc) return rc;

  p.ksize = d->ksize; p.stride = d->stride; p.pad = (d->ksize - 1) / 2;
  p.in_c = d->in_c; p.batch = d->batch;
  p.M = (long long)d->batch * d->out_h * d->out_w;
  p.KC = (d->in_c % 64 == 0) ? 64 : (d->in_c % 32 == 0 ? 32 : 16);
  p.kchunks = d->in_c / p.KC;
  p.BN = largest_divisor_tile(d->out_c, 256);
  p.n_tiles = d->out_c / p.BN;
  p.BNpad = 32;
  while (p.BNpad < p.BN) p.BNpad <<= 1;
  // Two co-resident CTAs per SM for the small layers (few tiles per SM: the kernel is fill / drain latency, not throughput):
  // each CTA takes half the shared memory and half of TMEM and one epilogue warpgroup (192 threads x ~120 registers), so that
  // one CTA's loads and MMAs overlap the other's epilogue and, with programmatic dependent launch, the next kernel's
  // prologue (barriers, TMEM, resident weights) starts in the slot a finished CTA frees while its neighbour still drains.
  int ctas = conv_ctas_per_sm(d);
  const int tmem_budget = 512 / ctas;
  p.acc_stages = tmem_budget / p.BNpad;
  if (p.acc_stages < 1) { ctas = 1; p.acc_stages = 512 / p.BNpad; }
  if (p.acc_stages > kMaxAcc) p.acc_stages = kMaxAcc;
  p.tmem_cols = (unsigned)(p.acc_stages * p.BNpad);  // power of two >= 32 by construction

  p.flat = (d->ksize == 1 && d->stride == 1) ? 1 : 0;
  p.halo = (d->ksize == 3 && d->stride == 1) ? 1 : 0;
  p.taps = p.flat ? 1 : 9;
  if (p.flat && allow_flat) p.halo = 1;
  // stride 2: the x parity folds into the channel dimension only when pixel pairs are contiguous
  if (allow_s2 && d->ksize == 3 && d->stride == 2 && d->in_ld == d->in_c && d->in_w % 2 == 0 && (d->in_c == 32 || d->in_c % 64 == 0))
    p.halo = 2;
  if (p.halo == 2) { p.KC = 64; p.kchunks = 2 * d->in_c / 64; }
  const unsigned row_bytes = (unsigned)p.KC * 2;             // 128 / 64 / 32 = swizzle span
  p.row_bytes = row_bytes;
  p.G = 1; p.a_slots = 0; p.b_region_bytes = 0;
  int max_smem = max_smem_optin();
  if (ctas == 2 && max_smem > 112 * 1024) max_smem = 112 * 1024;       // 228 KB per SM, 1 KB reserved per CTA
  p.bias_bytes = ((unsigned)d->out_c * 4u + 1023u) & ~1023u;

  if (p.halo) {
    const int hx = p.halo == 2 ? 1 : 2;     // halo columns / rows per tile
    if (p.flat) {
      p.tw = 128; p.th = 1; p.pitch = 128;
      p.tiles_w = (int)ceil_div64(p.M, 128); p.tiles_h = 1;
      p.m_tiles = p.tiles_w;
      p.a_slot_bytes = (128u * row_bytes + 1023u) & ~1023u;
      p.a_tx_bytes = 128u * row_bytes;
    } else {
      // spatial tile: th rows of (tw + hx) accumulator rows each (the halo columns of every row are discarded)
      long long best_cost = -1; int btw = 1, bth = 1;
      for (int tw = 1; tw <= d->out_w && tw + hx <= 128; ++tw) {
        int th = 128 / (tw + hx);
        if (th > d->out_h) th = d->out_h;
        if (th < 1 || (th + hx) * d->stride > 256) continue;
        const long long tiles = ceil_div64(d->out_w, tw) * ceil_div64(d->out_h, th);
        const long long cost = tiles * 4096 + (long long)(th + hx) * (tw + hx);   // fewest tiles, then least halo traffic
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; btw = tw; bth = th; }
      }
      p.tw = btw; p.th = bth; p.pitch = btw + hx;
      p.tiles_w = (int)ceil_div64(d->out_w, p.tw);
      p.tiles_h = (int)ceil_div64(d->out_h, p.th);
      p.m_tiles = d->batch * p.tiles_w * p.tiles_h;
      // rows touched by the last tap of accumulator row 127, rounded to the swizzle atom
      const unsigned slot_rows = p.halo == 2 ? 127u + (unsigned)p.pitch + 2u : 127u + 2u * (unsigned)p.pitch + 3u;
      p.a_slot_bytes = (slot_rows * row_bytes + 1023u) & ~1023u;
      p.a_tx_bytes = (unsigned)((p.th + hx) * p.pitch) * row_bytes;
    }
    // short K loops are epilogue-bound: three tiles in the epilogue at once (MMA cycles per tile ~ k-steps * N / 2)
    p.epi_groups = (p.taps * p.kchunks * (p.KC / 16) * d->out_c <= 4096 && d->out_c <= 128) ? 3 : 2;
    if (d->epilogue == YX_EPI_HEAD) p.epi_groups = 2;                            // staging slabs are 10.9 KB per warp
    YX_REQUIRE(d->epilogue == YX_EPI_STORE || p.flat, YX_ERR_UNSUPPORTED, "conv_tc: the head epilogue needs a 1x1 conv");
    p.head_bytes = d->epilogue == YX_EPI_HEAD ? (((unsigned)p.epi_groups * 4u * 32u * (unsigned)(5 + d->head_nc) * 4u + 1023u) & ~1023u) : 0u;
    const unsigned fixed_bytes = 2048u + p.bias_bytes + p.head_bytes;
    const long long avail = (long long)max_smem - fixed_bytes;
    long long n_btiles = (long long)p.taps * p.kchunks;
    if (p.halo == 2) {
      // op tables; a_off16 = (row shift * row_bytes + byte offset in the row) / 16, P = pitch
      const unsigned rb16 = row_bytes >> 4, P = (unsigned)p.pitch;
      const int C = d->in_c;
      auto tapk = [&](int r, int sx) { return (r * 3 + sx) * C; };
      memset(p.s2, 0, sizeof(p.s2));
      if (C == 32) {
        // one mixed chunk per row: [x-even 32 ch | x-odd 32 ch]; taps (r,1),(r,2) are one K = 64 GEMM at column
        // x, tap (r,0) is a K = 32 GEMM on the x-odd half of column x-1
        p.s2_kinds = 2; p.s2_cchunks = 1;
        p.s2[0] = {0, -1, 4, {1u * rb16, 0u * rb16 + 4u, (P + 1u) * rb16, P * rb16 + 4u},
                   {tapk(0, 1), tapk(0, 0), tapk(2, 1), tapk(2, 0)}, {4, 2, 4, 2}};
        p.s2[1] = {0, 0, 2, {1u * rb16, 0u * rb16 + 4u, 0, 0}, {tapk(1, 1), tapk(1, 0), 0, 0}, {4, 2, 0, 0}};
      } else {
        p.s2_kinds = 4; p.s2_cchunks = C / 64;
        p.s2[0] = {0, -1, 2, {1u * rb16, (P + 1u) * rb16, 0, 0}, {tapk(0, 1), tapk(2, 1), 0, 0}, {4, 4, 0, 0}};
        p.s2[1] = {0, 0, 1, {1u * rb16, 0, 0, 0}, {tapk(1, 1), 0, 0, 0}, {4, 0, 0, 0}};
        p.s2[2] = {C, -1, 4, {0u, 1u * rb16, P * rb16, (P + 1u) * rb16},
                   {tapk(0, 0), tapk(0, 2), tapk(2, 0), tapk(2, 2)}, {4, 4, 4, 4}};
        p.s2[3] = {C, 0, 2, {0u, 1u * rb16, 0, 0}, {tapk(1, 0), tapk(1, 2), 0, 0}, {4, 4, 0, 0}};
      }
      n_btiles = 0;
      for (int k = 0; k < p.s2_kinds; ++k) n_btiles += p.s2[k].nops;
      n_btiles *= p.s2_cchunks;
    }
    // N tile: the whole out_c (<= 256) when its weights can stay resident next to >= 3 halo slots, otherwise
    // <= 128 so that two accumulator pairs fit TMEM and two M tiles share every streamed weight stage
    long long b_all = 0;
    for (int cap = 256; cap >= 128; cap -= 128) {
      p.BN = largest_divisor_tile(d->out_c, cap);
      p.n_tiles = d->out_c / p.BN;
      p.BNpad = 32;
      while (p.BNpad < p.BN) p.BNpad <<= 1;
      p.acc_stages = tmem_budget / p.BNpad;
      if (p.acc_stages < 1) p.acc_stages = 1;
      if (p.acc_stages > kMaxAcc) p.acc_stages = kMaxAcc;
      p.tmem_cols = (unsigned)(p.acc_stages * p.BNpad);
      p.b_tile_bytes = ((unsigned)p.BN * row_bytes + 1023u) & ~1023u;
      p.b_tx_bytes = (unsigned)p.BN * row_bytes;
      b_all = n_btiles * p.b_tile_bytes;
      p.b_resident = (p.n_tiles == 1 && avail - b_all >= 3ll * p.a_slot_bytes) ? 1 : 0;
      if (p.b_resident) break;
    }
    if (p.epi_groups > p.acc_stages) p.epi_groups = p.acc_stages;
    if (ctas == 2) p.epi_groups = 1;
    // stride-2 planes only pay off with resident weights (streamed weights are not shared between M tiles there)
    if (p.halo == 2 && !p.b_resident) return conv_tc_prepare_mode(d, L, false);
    // 1x1 with weights too large to stay resident: the per-tap ring with N up to 256 streams fewer bytes
    if (p.flat && !p.b_resident) return conv_tc_prepare_mode(d, L, allow_s2, false);
    if (p.b_resident) {
      p.G = 1;
      p.b_region_bytes = (unsigned)b_all;
      p.stages = 1;
      p.a_slots = (int)((avail - b_all) / p.a_slot_bytes);
    } else {
      p.G = (p.acc_stages >= 4 && p.halo == 1) ? 2 : 1;
      p.a_slots = 2 * p.G;
      long long rest = avail - (long long)p.a_slots * p.a_slot_bytes;
      YX_REQUIRE(rest >= 2ll * p.b_tile_bytes, YX_ERR_UNSUPPORTED, "conv_tc(halo): shared memory too small");
      p.stages = (int)(rest / p.b_tile_bytes);
      if (p.stages > kMaxStages) p.stages = kMaxStages;
      p.b_region_bytes = (unsigned)p.stages * p.b_tile_bytes;
      // leftover shared memory deepens the halo ring
      rest = avail - p.b_region_bytes;
      p.a_slots = (int)(rest / p.a_slot_bytes);
    }
    if (p.a_slots > kMaxASlots) p.a_slots = kMaxASlots;
    YX_REQUIRE(p.a_slots >= p.G, YX_ERR_UNSUPPORTED, "conv_tc(halo): halo ring does not fit shared memory");
    const int m_pad = (int)ceil_div64(p.m_tiles, p.G) * p.G;
    p.num_tiles = m_pad * p.n_tiles;
    L->smem = fixed_bytes + p.b_region_bytes + (size_t)p.a_slots * p.a_slot_bytes;
  } else {
  if (p.flat) {
    p.tw = 128; p.th = 1;
    p.tiles_w = (int)ceil_div64(p.M, 128); p.tiles_h = 1;
    p.num_tiles = p.tiles_w * p.n_tiles;
  } else {
    // choose the spatial tile (tw x th <= 128 pixels) that wastes the fewest accumulator rows
    long long best_cost = -1; int btw = 1, bth = 1;
    for (int tw = 1; tw <= d->out_w && tw <= 128; ++tw) {
      int th = 128 / tw;
      if (th > d->out_h) th = d->out_h;
      if (th < 1) continue;
      if (th * d->stride > 256 || tw * d->stride > 256) continue;
      const long long tiles = ceil_div64(d->out_w, tw) * ceil_div64(d->out_h, th);
      // cost: number of tiles; tie -> wider rows (longer contiguous runs for TMA)
      const long long cost = tiles * 1024 - tw;
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; btw = tw; bth = th; }
    }
    p.tw = btw; p.th = bth;
    p.tiles_w = (int)ceil_div64(d->out_w, p.tw);
    p.tiles_h = (int)ceil_div64(d->out_h, p.th);
    p.num_tiles = d->batch * p.tiles_w * p.tiles_h * p.n_tiles;
  }
  p.pitch = p.tw;
  p.m_tiles = p.num_tiles / p.n_tiles;

  const unsigned a_bytes = 128u * row_bytes;
  const unsigned b_bytes = (unsigned)p.BN * row_bytes;
  p.a_stage_bytes = (a_bytes + 1023u) & ~1023u;
  p.stage_bytes = p.a_stage_bytes + ((b_bytes + 1023u) & ~1023u);
  p.tx_bytes = (unsigned)(p.tw * p.th) * row_bytes + b_bytes;  // bytes TMA actually delivers
  // epilogue groups: memory-bound layers (short K loops) need several tiles in the epilogue at once
  {
    const int num_k_total = d->ksize * d->ksize * (d->in_c / p.KC);
    p.epi_groups = num_k_total * (p.KC / 16) * p.BN <= 4096 ? 3 : 2;   // MMA cycles per tile ~ k-steps * BN / 2
    if (p.epi_groups > p.acc_stages) p.epi_groups = p.acc_stages;
    if (d->epilogue == YX_EPI_HEAD && p.epi_groups > 2) p.epi_groups = 2;   // staging slabs are 10.9 KB per warp
    if (ctas == 2) p.epi_groups = 1;
  }
  p.head_bytes = d->epilogue == YX_EPI_HEAD ? (((unsigned)p.epi_groups * 4u * 32u * (unsigned)(5 + d->head_nc) * 4u + 1023u) & ~1023u) : 0u;
  const unsigned fixed_bytes = 2048u + p.bias_bytes + p.head_bytes;
  int stages = (int)((max_smem - (int)fixed_bytes) / p.stage_bytes);
  if (stages > 8) stages = 8;
  YX_REQUIRE(stages >= 2, YX_ERR_UNSUPPORTED, "conv_tc: stage of %u bytes does not fit shared memory", p.stage_bytes);
  p.stages = stages;
  L->smem = fixed_bytes + (size_t)stages * p.stage_bytes;
  }

  p.desc_hi = umma_desc_hi(row_bytes);
  p.idesc = umma_idesc(d->dtype, p.BN);
  const CUtensorMapDataType tdt = tma_dtype(d->dtype);
  const CUtensorMapSwizzle sw = tma_swizzle(row_bytes);
  {
    cuuint64_t dims[4], strides[3];
    cuuint32_t box[4], estr[4];
    if (p.flat) {
      dims[0] = (cuuint64_t)d->in_c; dims[1] = (cuuint64_t)p.M; dims[2] = 1; dims[3] = 1;
      strides[0] = (cuuint64_t)d->in_ld * 2;
      strides[1] = strides[0] * (cuuint64_t)p.M;
      strides[2] = strides[1];
      box[0] = (cuuint32_t)p.KC; box[1] = 128; box[2] = 1; box[3] = 1;
      estr[0] = estr[1] = estr[2] = estr[3] = 1;
    } else {
      dims[0] = (cuuint64_t)d->in_c; dims[1] = (cuuint64_t)d->in_w; dims[2] = (cuuint64_t)d->in_h; dims[3] = (cuuint64_t)d->batch;
      strides[0] = (cuuint64_t)d->in_ld * 2;
      strides[1] = strides[0] * (cuuint64_t)d->in_w;
      strides[2] = strides[1] * (cuuint64_t)d->in_h;
      box[0] = (cuuint32_t)p.KC; box[1] = (cuuint32_t)(p.tw * d->stride); box[2] = (cuuint32_t)(p.th * d->stride); box[3] = 1;
      estr[0] = 1; estr[1] = (cuuint32_t)d->stride; estr[2] = (cuuint32_t)d->stride; estr[3] = 1;
      if (p.halo == 1) { box[1] = (cuuint32_t)p.pitch; box[2] = (cuuint32_t)(p.th + 2); }
      if (p.halo == 2) {
        dims[0] = (cuuint64_t)(2 * d->in_c); dims[1] = (cuuint64_t)(d->in_w / 2);
        strides[0] = (cuuint64_t)d->in_ld * 4;
        box[0] = 64; box[1] = (cuuint32_t)p.pitch; box[2] = (cuuint32_t)((p.th + 1) * 2);
        estr[1] = 1;
      }
    }
    rc = encode_tma(&L->map_a, tdt, 4, d->in, dims, strides, box, estr, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "A");
    if (rc) return rc;
  }
  {
    const cuuint64_t K = (cuuint64_t)d->ksize * d->ksize * d->in_c;
    cuuint64_t dims[2] = {K, (cuuint64_t)d->out_c};
    cuuint64_t strides[1] = {K * 2};
    cuuint32_t box[2] = {(cuuint32_t)p.KC, (cuuint32_t)p.BN};
    rc = encode_tma(&L->map_b, tdt, 2, d->w, dims, strides, box, nullptr, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "W");
    if (rc) return rc;
  }
  p.mul_tpi = fast_div_mul(p.tiles_w * p.tiles_h);
  p.mul_tw = fast_div_mul(p.tiles_w);
  p.mul_ntiles = fast_div_mul(p.n_tiles);
  p.mul_ohw = fast_div_mul(d->out_h * d->out_w);
  p.mul_ow = fast_div_mul(d->out_w);
  const int sms = num_sms() * ctas;
  L->ctas = ctas;
  L->grid = p.num_tiles < sms ? p.num_tiles : sms;
  if (p.halo) {
    const int groups = p.num_tiles / p.G;     // never split a weight-sharing group when there is less than one per SM
    L->grid = groups < sms ? groups : sms;
  }
  return YX_OK;
}

int conv_tc_prepare(const yx_conv_desc* d, ConvTcLaunch* L) { return conv_tc_prepare_mode(d, L, true); }

ConvTcLaunch* conv_tc_alloc() { return new (std::nothrow) ConvTcLaunch(); }
void conv_tc_free(ConvTcLaunch* p) { delete p; }

// The launch selection of conv_tc_prepare, without a launch (yx_conv_schedule): tests use it to show which mode, ring
// depths and per-CTA tile ranges a shape exercises.
int conv_tc_schedule(const yx_conv_desc* d, int32_t* info, int capacity) {
  ConvTcLaunch L = {};
  const int rc = conv_tc_prepare(d, &L);
  if (rc) return rc;
  const ConvTcParams& p = L.p;
  const int32_t v[] = {p.halo, p.flat, p.b_resident, p.G, L.ctas, p.epi_groups, p.acc_stages, p.a_slots,
                       p.stages, p.BN, p.n_tiles, p.m_tiles, p.num_tiles, L.grid, p.tw, p.th};
  int n = 0;
  for (; n < (int)(sizeof(v) / sizeof(v[0])) && n < capacity; ++n) info[n] = v[n];
  return n;
}

// [fp16][store, store + SiLU, head]: the head epilogue has no SiLU instantiation
static decltype(&conv_tc_kernel<false, false, false>) const kConvKernels[2][3] = {
    {conv_tc_kernel<false, false, false>, conv_tc_kernel<false, true, false>, conv_tc_kernel<false, false, true>},
    {conv_tc_kernel<true, false, false>, conv_tc_kernel<true, true, false>, conv_tc_kernel<true, false, true>}};

int conv_tc_launch(const ConvTcLaunch* L, cudaStream_t stream) {
  static bool smem_set[kMaxDevices] = {};
  YX_CUDA(opt_in_smem(smem_set, kConvKernels, [](int) { return max_smem_optin(); }));
  const EpiParams& e = L->p.epi;
  const int epi = e.epilogue == YX_EPI_HEAD ? 2 : (e.act == YX_ACT_SILU ? 1 : 0);
  const auto kernel = kConvKernels[e.dtype == YX_FP16][epi];
  YX_CUDA(launch_pdl(kernel, dim3((unsigned)L->grid), dim3((unsigned)(64 + 128 * L->p.epi_groups)), L->smem, stream, L->map_a,
                     L->map_b, L->p));
  return YX_OK;
}

}  // namespace yx
