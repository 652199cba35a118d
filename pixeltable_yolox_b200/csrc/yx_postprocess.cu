// postprocess = score filter + class-aware NMS, batched over images, no host synchronisation.
//   reference: yolox/utils/boxes.py:31-75 (postprocess) and the third-party
//   torchvision.ops.batched_nms / nms it calls at boxes.py:56-67 (torchvision 0.17.2 pinned in
//   poetry.lock:2084-2085; semantics restated in oracle/postprocess_oracle.py and pinned against
//   the installed torchvision by tests/golden/make_golden.py).
//
// Stage 1  filter_kernel      warp per anchor: coalesced read of the 5+nc floats, warp arg-max over
//                             the classes (first index wins ties, like torch.max), score =
//                             obj*class_conf (one fp32 multiply), cxcywh->xyxy exactly as
//                             boxes.py:32-37, dense candidate row + 64-bit sort key for anchors with
//                             score >= conf_thre (warp-aggregated append).
// Stage 2  sort_nms_kernel    one CTA per image, or one thread-block cluster of 2 / 4 / 8 CTAs per image:
//                             merge sort of the keys (descending score, ascending anchor = torch's stable
//                             descending sort) in shared memory, then greedy NMS: groups of 512 sorted
//                             candidates are tested against the boxes already kept (phase A, per-class
//                             lists in shared memory); the survivors of several groups form a batch whose
//                             512x512 suppression bitmask is built in shared memory (phase B) and scanned
//                             by one warp that hops from kept box to kept box (phase C). Keys, mask and
//                             kept list never touch HBM. DESIGN.md 4.9 has the phase clocks.
// IoU arithmetic follows torchvision's nms kernel operation by operation in fp32 (round-to-nearest
// intrinsics so that nvcc cannot contract multiplies and adds into FMAs):
//   inter = max(0, min(x2) - max(x1)) * max(0, min(y2) - max(y1));
//   suppressed iff inter / (area_i + area_j - inter) > thr   (the division itself only runs within 2^-20 of
//   the threshold; outside that band a multiply decides with the same result, see suppresses()).
#include <stdlib.h>
#include <string.h>
#include <math.h>

#include "yx_common.cuh"

namespace yx {

static constexpr int kChunk = 512;
static constexpr int kChunkWords = kChunk / 32;
static constexpr int kNmsThreads = 512;
static constexpr int kMaxSmemKeys = 16384;  // 128 KB of 64-bit keys
static constexpr int kMaskPitch = kChunkWords + 1;   // words per mask row: odd pitch, column reads are bank-conflict free
static constexpr int kChunkBytes = kChunk * 24 + kChunk * kMaskPitch * 4;
static constexpr int kClassCap = 512;       // class ids below this get a linked list of kept boxes
static constexpr int kNmsFixedBytes = kChunkBytes + kChunk * 4 + 3 * kClassCap * 4;   // + survivors, list heads, two bounds per class
static constexpr int kKeptEntryBytes = 20;  // box 16 + (class | next << 10) 4; the area is recomputed (3 flops)
static constexpr int kNmsSmemBudget = 224 * 1024;   // dynamic shared memory (+ ~3.5 KB static <= 228 KB per CTA): 8 704 kept entries, i.e. every anchor of a 640^2 image

static constexpr int kFlushRows = 192;               // survivor batch: resolved once it holds this many of its 512 rows (measured sweep 128..512: flat within 3 %, profiles/r2_nms_flush_sweep.jsonl)
static constexpr int kNmsMaxCluster = 8;             // CTAs of one image's thread-block cluster (sort_nms_kernel<true>)

__device__ __forceinline__ uint32_t orderable(float f) { return orderable_f32(f); }

__device__ __forceinline__ uint32_t nms_cluster_ctarank() {
  uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r;
}
__device__ __forceinline__ uint32_t nms_cluster_nctarank() {
  uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r;
}
// every thread of every CTA of the cluster; release / acquire at cluster scope (orders shared memory of the own CTA,
// distributed shared memory and the global workspace before / after it); also a CTA barrier
__device__ __forceinline__ void nms_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// generic address of the same shared-memory object in CTA `rank` of the cluster
template <typename T>
__device__ __forceinline__ T* nms_peer(T* local, int rank) {
  unsigned long long out;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"(reinterpret_cast<unsigned long long>(local)), "r"(rank));
  return reinterpret_cast<T*>(out);
}

// ------------------------------------------------------------------------------------------
// Stage 1
// ------------------------------------------------------------------------------------------
static constexpr int kFilterAnchors = 128;   // anchors per CTA (one per thread)

// One CTA stages 128 consecutive rows of [5+nc] floats in shared memory with coalesced (128-bit when
// aligned) loads; then every thread owns one anchor: sequential arg-max over its row (row pitch 5+nc is
// odd for nc = 80, so the strided shared reads are conflict free), box conversion, score, and one
// warp-aggregated append of the passing anchors' sort keys.
__global__ void __launch_bounds__(kFilterAnchors)
filter_kernel(float* __restrict__ pred, int batch, int anchors, int nc, float conf_thre, int inplace_xyxy,
              float* __restrict__ cand, unsigned long long* __restrict__ keys, int* __restrict__ counts) {
  extern __shared__ __align__(128) float frows[];         // [kFilterAnchors][5+nc]
  __shared__ uint64_t fbar;
  const int nch = 5 + nc;
  const int chunks = (anchors + kFilterAnchors - 1) / kFilterAnchors;
  const int b = blockIdx.x / chunks;
  const int a0 = (blockIdx.x - b * chunks) * kFilterAnchors;
  const int na = min(kFilterAnchors, anchors - a0);
  const int tid = threadIdx.x, lane = tid & 31;
  float* g = pred + ((long long)b * anchors + a0) * nch;
  const int total = na * nch;
  if (tid == 0) { mbar_init(&fbar, 1); fence_barrier_init(); }
  __syncthreads();
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0 && (total & 3) == 0) {
    // one bulk copy (TMA, no register staging) brings the CTA's rows in; 5 CTAs per SM keep ~200 KB in flight
    if (tid == 0) {
      mbar_arrive_expect_tx(&fbar, (uint32_t)total * 4u);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(frows)),
                   "l"(g), "r"((uint32_t)total * 4u), "r"(smem_u32(&fbar))
                   : "memory");
    }
    mbar_wait(&fbar, 0);
  } else if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* s4 = reinterpret_cast<float4*>(frows);
    for (int i = tid; i < total / 4; i += kFilterAnchors) s4[i] = g4[i];
    for (int i = (total & ~3) + tid; i < total; i += kFilterAnchors) frows[i] = g[i];
  } else {
    for (int i = tid; i < total; i += kFilterAnchors) frows[i] = g[i];
  }
  __syncthreads();
  bool pass = false;
  unsigned long long key = 0;
  if (tid < na) {
    const float* row = frows + tid * nch;
    // torch.max(dim): first occurrence of the maximum; a NaN wins and the first NaN is reported
    float best = row[5];
    int best_i = 0;
    for (int c = 1; c < nc; ++c) {
      const float v = row[5 + c];
      if (!(best != best) && (v > best || v != v)) { best = v; best_i = c; }
    }
    const float cx = row[0], cy = row[1], w = row[2], h = row[3], obj = row[4];
    const float hw = __fdiv_rn(w, 2.0f), hh = __fdiv_rn(h, 2.0f);
    float4 box;
    box.x = __fsub_rn(cx, hw); box.y = __fsub_rn(cy, hh);
    box.z = __fadd_rn(cx, hw); box.w = __fadd_rn(cy, hh);
    const float score = __fmul_rn(obj, best);
    const int a = a0 + tid;
    if (inplace_xyxy) {
      float* grow = g + (long long)tid * nch;
      grow[0] = box.x; grow[1] = box.y; grow[2] = box.z; grow[3] = box.w;
    }
    float4* crow = reinterpret_cast<float4*>(cand + ((long long)b * anchors + a) * 8);
    crow[0] = box;
    crow[1] = make_float4(obj, best, (float)best_i, score);
    pass = score >= conf_thre;
    const float sc = (score == 0.0f) ? 0.0f : score;  // -0 -> +0
    key = ((unsigned long long)(~orderable(sc)) << 32) | (unsigned long long)(unsigned)a;
  }
  const unsigned bal = __ballot_sync(0xffffffffu, pass);
  if (bal) {
    int base = 0;
    if (lane == (__ffs(bal) - 1)) base = atomicAdd(&counts[b], __popc(bal));
    base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
    if (pass) keys[(long long)b * anchors + base + __popc(bal & ((1u << lane) - 1))] = key;
  }
}

// Ordered compaction for yx_score_filter_compact: one CTA per image walks the dense candidate
// rows in anchor order with a block-wide exclusive scan of the pass flags.
__global__ void __launch_bounds__(1024)
compact_kernel(const float* __restrict__ cand_dense, int anchors, float conf_thre, float* __restrict__ cand,
               int* __restrict__ cand_idx, int* __restrict__ cand_count) {
  __shared__ int warp_sums[32];
  __shared__ int base;
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  for (int a0 = 0; a0 < anchors; a0 += blockDim.x) {
    const int a = a0 + threadIdx.x;
    const float4* row = reinterpret_cast<const float4*>(cand_dense + ((long long)b * anchors + a) * 8);
    float4 r0 = make_float4(0, 0, 0, 0), r1 = make_float4(0, 0, 0, -INFINITY);
    bool pass = false;
    if (a < anchors) { r0 = row[0]; r1 = row[1]; pass = r1.w >= conf_thre; }
    const unsigned bal = __ballot_sync(0xffffffffu, pass);
    const int wprefix = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) warp_sums[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
      int v = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += n;
      }
      warp_sums[lane] = v;  // inclusive
    }
    __syncthreads();
    const int woff = warp == 0 ? 0 : warp_sums[warp - 1];
    if (pass) {
      const int dst = base + woff + wprefix;
      float4* orow = reinterpret_cast<float4*>(cand + ((long long)b * anchors + dst) * 8);
      orow[0] = r0; orow[1] = r1;
      cand_idx[(long long)b * anchors + dst] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) base += warp_sums[(blockDim.x >> 5) - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) cand_count[b] = base;
}

// ------------------------------------------------------------------------------------------
// Stage 2
// ------------------------------------------------------------------------------------------
struct NmsSource {
  const float* boxes; int box_stride;      // xyxy, floats per candidate
  const float* scores; int score_stride;
  const void* cls; int cls_stride; int cls_is_float;
  long long per_image;                      // candidates per image in the dense arrays
  int cand_rows;                            // 1: boxes / scores / cls are the 8-float candidate rows of the score filter
};

struct NmsArgs {
  NmsSource src;
  const unsigned long long* keys;  // [B, per_image] (filter path) or null (build from scores)
  const int* counts;               // [B]
  float thr;                       // largest float f with (double)f <= nms_thre: x > f <=> x > nms_thre
  int variant;                     // 0 offset trick, 1 per-class, 2 class-agnostic,
                                   // 3/4: torchvision's own choice on CUDA / CPU (by candidate count)
  // scratch [B, per_image]
  unsigned long long* gkeys;       // used when the key list does not fit shared memory
  long long gkeys_stride;          // keys per image in gkeys (next_pow2(per_image))
  int smem_keys_cap;               // number of 64-bit keys the dynamic shared memory can hold
  int smem_bytes;                  // dynamic shared memory of the launch
  int kept_cap;                    // kept boxes that fit the shared-memory kept list
  float4* sorted_box;              // boxes as NMS sees them (offset applied for variant 0)
  int* sorted_cls;
  int* sorted_idx;
  int* kept_pos;                   // positions (in sorted order) of the kept candidates
  // outputs
  int* keep; int* keep_count;      // yx_batched_nms
  float* dets; long long* det_idx; int* det_count; int max_det;  // yx_postprocess (from cand rows)
  int no_small;                    // YX_NMS_NO_SMALL: never take the single-warp path (tests compare the two paths)
};

__device__ __forceinline__ bool suppresses(const float4 a, float area_a, const float4 b, float area_b, float thr) {
  const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
  const float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
  const float w = fmaxf(0.0f, __fsub_rn(xx2, xx1));
  const float h = fmaxf(0.0f, __fsub_rn(yy2, yy1));
  const float inter = __fmul_rn(w, h);
  // disjoint boxes: 0 / x is 0 (or NaN for 0 / 0), never > thr for thr >= 0 -- skip the IEEE division
  if (inter == 0.0f && thr >= 0.0f) return false;
  const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  // The IEEE division only decides pairs within 2^-20 of the threshold. Rounding is monotone, so with q = inter / uni (real):
  // inter > rn(rn(thr * uni) * (1 + 2^-20)) implies q > thr * (1 + 2^-21) >= thr + ulp(thr), hence rn(q) > thr; and
  // inter < rn(rn(thr * uni) * (1 - 2^-20)) implies q < thr, hence rn(q) <= thr. (Ranges keep thr * uni a normal number; NaNs
  // fail both compares and take the division.)
  if (uni > 1e-18f && uni < 1e18f && thr > 1e-6f && thr < 1e6f) {
    const float p = __fmul_rn(thr, uni);
    if (inter > __fmul_rn(p, 1.00000095367431640625f)) return true;
    if (inter < __fmul_rn(p, 0.99999904632568359375f)) return false;
  }
  const float ovr = __fdiv_rn(inter, uni);
  return ovr > thr;
}
__device__ __forceinline__ float box_area(const float4 b) {
  return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}

// n <= 32 candidates (the common case at the default thresholds: ~20 per image): one warp does the whole image in
// registers -- key sort by 15 shuffle compare-exchanges, 32 x 32 suppression bits with the same arithmetic as the chunked
// path, the fixed 32-step greedy resolution -- and writes the outputs; no shared memory, no block barriers.
__device__ __forceinline__ void nms_small_warp(const NmsArgs& g, int b, int n, int variant, long long base) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  unsigned long long k = ~0ull;
  if (lane < n) {
    if (g.keys) k = g.keys[base + lane];
    else {
      float sc = g.src.scores[(base + lane) * g.src.score_stride];
      if (sc == 0.0f) sc = 0.0f;
      k = ((unsigned long long)(~orderable(sc)) << 32) | (unsigned long long)(unsigned)lane;
    }
  }
#pragma unroll
  for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const unsigned long long o = __shfl_xor_sync(full, k, stride);
      const bool keep_min = (((lane & stride) == 0) == ((lane & size) == 0));
      k = keep_min ? (k < o ? k : o) : (k > o ? k : o);
    }
  }
  const bool valid = lane < n;
  const int idx = valid ? (int)(unsigned)(k & 0xffffffffull) : 0;
  float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
  int c = 0;
  float mx = -INFINITY;
  if (valid) {
    const float* bp = g.src.boxes + (base + idx) * g.src.box_stride;
    bx = make_float4(bp[0], bp[1], bp[2], bp[3]);
    if (g.src.cls_is_float) c = (int)reinterpret_cast<const float*>(g.src.cls)[(base + idx) * g.src.cls_stride];
    else c = reinterpret_cast<const int*>(g.src.cls)[(base + idx) * g.src.cls_stride];
    mx = fmaxf(fmaxf(bx.x, bx.y), fmaxf(bx.z, bx.w));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(full, mx, o));
  if (variant == 0) {
    const float off = __fmul_rn((float)c, __fadd_rn(mx, 1.0f));
    bx.x = __fadd_rn(bx.x, off); bx.y = __fadd_rn(bx.y, off);
    bx.z = __fadd_rn(bx.z, off); bx.w = __fadd_rn(bx.w, off);
  }
  const float area = box_area(bx);
  unsigned row = 0u;                                   // bit j: this lane's box suppresses the later box j
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float4 ob;
    ob.x = __shfl_sync(full, bx.x, j); ob.y = __shfl_sync(full, bx.y, j);
    ob.z = __shfl_sync(full, bx.z, j); ob.w = __shfl_sync(full, bx.w, j);
    const float oa = __shfl_sync(full, area, j);
    const int oc = __shfl_sync(full, c, j);
    if (valid && j > lane && j < n && (variant != 1 || oc == c) && suppresses(bx, area, ob, oa, g.thr)) row |= 1u << j;
  }
  unsigned alive = n >= 32 ? full : ((1u << n) - 1u), keptw = 0u;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const unsigned di = __shfl_sync(full, row, i);
    if ((alive >> i) & 1u) { keptw |= 1u << i; alive &= ~di; }
  }
  const int nk = __popc(keptw);
  const bool mine = (keptw >> lane) & 1u;
  const int pos = __popc(keptw & ((1u << lane) - 1u));
  if (g.keep) {
    if (mine) g.keep[base + pos] = idx;
    if (lane == 0) g.keep_count[b] = nk;
  }
  if (g.dets) {
    if (mine && pos < g.max_det) {
      const float4* crow = reinterpret_cast<const float4*>(g.src.boxes + (base + idx) * 8);
      const float4 r0 = crow[0], r1 = crow[1];
      float* d = g.dets + ((long long)b * g.max_det + pos) * 7;
      d[0] = r0.x; d[1] = r0.y; d[2] = r0.z; d[3] = r0.w; d[4] = r1.x; d[5] = r1.y; d[6] = r1.z;
      if (g.det_idx) g.det_idx[(long long)b * g.max_det + pos] = idx;
    }
    if (lane == 0) g.det_count[b] = nk;
  }
}

// Ascending sort of keys[0, n) (unique 64-bit keys) by all threads of the CTA: bitonic network in its all-ascending
// form -- for every block size one "flip" step (i against i ^ (size-1)) followed by half-cleaners (i against i ^ j,
// j = size/4 .. 1). Because every compare-exchange is ascending, the slots >= n behave like +inf padding that never
// moves, so pairs with a partner >= n are simply not enumerated: n = 8 400 costs about half of the padded 16 384
// network. Four independent pairs are loaded before the first compare so that the shared-memory latency of a step
// overlaps. Ends with a CTA barrier.
__device__ __forceinline__ void sort_keys_asc(unsigned long long* keys, const int n, const int tid, const int max_lg = 31) {
  for (int lg = 1; (1 << (lg - 1)) < n && lg <= max_lg; ++lg) {      // max_lg: stop at sorted blocks of 2^max_lg keys
    const int size = 1 << lg, half = size >> 1;
    {
      const int fb = n >> lg, rem = n & (size - 1);
      const int full = fb << (lg - 1);                       // pairs of the complete blocks
      const int cnt = full + max(0, rem - half);             // + pairs of the last, partial block whose partner is < n
      for (int q0 = tid; q0 < cnt; q0 += 4 * kNmsThreads) {
        unsigned long long a[4], c[4];
        int lo[4], hi[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int q = q0 + u * kNmsThreads;
          if (q < cnt) {
            const int blk = q < full ? (q >> (lg - 1)) : fb;
            const int t = q < full ? (q & (half - 1)) : (size - rem) + (q - full);
            lo[u] = (blk << lg) + t; hi[u] = (blk << lg) + size - 1 - t;
            a[u] = keys[lo[u]]; c[u] = keys[hi[u]];
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (q0 + u * kNmsThreads < cnt && a[u] > c[u]) { keys[lo[u]] = c[u]; keys[hi[u]] = a[u]; }
      }
      __syncthreads();
    }
    for (int lgj = lg - 2; lgj >= 0; --lgj) {
      const int j = 1 << lgj;
      const int cnt = ((n >> (lgj + 1)) << lgj) + max(0, (n & (2 * j - 1)) - j);
      for (int q0 = tid; q0 < cnt; q0 += 4 * kNmsThreads) {
        unsigned long long a[4], c[4];
        int lo[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int q = q0 + u * kNmsThreads;
          if (q < cnt) {
            lo[u] = ((q & ~(j - 1)) << 1) | (q & (j - 1));
            a[u] = keys[lo[u]]; c[u] = keys[lo[u] | j];
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (q0 + u * kNmsThreads < cnt && a[u] > c[u]) { keys[lo[u]] = c[u]; keys[lo[u] | j] = a[u]; }
      }
      __syncthreads();
    }
  }
}

// Merge sort of keys[0, n) (unique keys, all below ~0) with a second buffer of n keys: blocks of 16 by the bitonic network
// above, then log2(n / 16) merge passes. In a pass every thread produces D = 17 (n <= 4 096) or 33 consecutive outputs of
// one pair of runs: merge-path binary search for its starting point, then a sequential two-way merge out of shared
// memory. D is odd so that the threads of a warp, D keys apart, stream through different banks (a power of two put all 32
// lanes on one bank: 190k clk for n = 8 400 instead of the network's 230k). A pass reads and writes every key once; the
// 10 passes for n = 8 400 replace 95 steps of the network.
// Returns the buffer that holds the result (keys after an even number of passes, tmp after an odd one: see
// merge_sorted_in_tmp). Ends with a CTA barrier.
__device__ __forceinline__ int merge_passes(int n) { return n > 16 ? (32 - __clz(n - 1)) - 4 : 0; }
__device__ __forceinline__ bool merge_sorted_in_tmp(int n) { return merge_passes(n) & 1; }
__device__ __forceinline__ unsigned long long* merge_sort_keys(unsigned long long* keys, unsigned long long* tmp, const int n,
                                                               const int tid) {
  sort_keys_asc(keys, n, tid, 4);
  unsigned long long* src = keys;
  unsigned long long* dst = tmp;
  const int D = n <= 4096 ? 17 : 33;
  for (int lgL = 4; (1 << lgL) < n; ++lgL) {
    const int L = 1 << lgL;
    const int ipp = (2 * L + D - 1) / D;                      // items per pair of runs (the last one is shorter)
    const int items = ((n + 2 * L - 1) >> (lgL + 1)) * ipp;
    for (int it = tid; it < items; it += kNmsThreads) {
      const int pr = it / ipp;
      const int d = (it - pr * ipp) * D;                      // first output of the item inside its pair
      const int a0 = pr << (lgL + 1);
      const int lenA = min(L, n - a0), b0 = a0 + lenA, lenB = min(L, n - b0);
      const int cnt = min(D, lenA + lenB - d);
      if (cnt <= 0) continue;                                 // the pair at the end of the list is incomplete
      const unsigned long long* A = src + a0;
      const unsigned long long* B = src + b0;
      int lo = max(0, d - lenB), hi = min(d, lenA);          // merge path: how many of the first d outputs come from A
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (A[mid] < B[d - 1 - mid]) lo = mid + 1; else hi = mid;
      }
      int i = lo, j = d - lo;
      unsigned long long ka = i < lenA ? A[i] : ~0ull, kb = j < lenB ? B[j] : ~0ull;
      unsigned long long* out = dst + a0 + d;
      for (int t = 0; t < cnt; ++t) {                         // branch-free step: one shared-memory load, no divergence
        const bool ta = ka < kb;
        out[t] = ta ? ka : kb;
        i += ta ? 1 : 0; j += ta ? 0 : 1;
        const int nx = ta ? i : j;
        const unsigned long long* P = ta ? A : B;
        const unsigned long long v = nx < (ta ? lenA : lenB) ? P[nx] : ~0ull;
        ka = ta ? v : ka; kb = ta ? kb : v;
      }
    }
    __syncthreads();
    unsigned long long* sw = src; src = dst; dst = sw;
  }
  return src;
}

__device__ __forceinline__ void nms_load_row(const NmsArgs& g, long long base, int idx, float4& bx, int& c) {
  if (g.src.cand_rows) {
    // candidate rows of the score filter: 8 floats (x1, y1, x2, y2, obj, class_conf, class, score), 32-byte aligned
    float o, cc, cl, sc;                      // one 256-bit load (sm_100: LDG.256)
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(bx.x), "=f"(bx.y), "=f"(bx.z), "=f"(bx.w), "=f"(o), "=f"(cc), "=f"(cl), "=f"(sc)
                 : "l"(g.src.boxes + (base + idx) * 8));
    c = (int)cl;
    return;
  }
  const float* bp = g.src.boxes + (base + idx) * g.src.box_stride;
  bx = make_float4(bp[0], bp[1], bp[2], bp[3]);
  if (g.src.cls_is_float) c = (int)reinterpret_cast<const float*>(g.src.cls)[(base + idx) * g.src.cls_stride];
  else c = reinterpret_cast<const int*>(g.src.cls)[(base + idx) * g.src.cls_stride];
}

__device__ __forceinline__ unsigned long long nms_key(const NmsArgs& g, long long base, int i) {
  if (g.keys) return g.keys[base + i];
  float sc = g.src.scores[(base + i) * g.src.score_stride];
  if (sc == 0.0f) sc = 0.0f;
  return ((unsigned long long)(~orderable(sc)) << 32) | (unsigned long long)(unsigned)i;
}

// CL = false: one CTA per image (grid = batch). CL = true: one thread-block cluster of R = 2 / 4 / 8 CTAs per image
// (grid = batch * R, cluster dimension R), chosen by the host when batch * R CTAs are co-resident:
//   sort     every CTA sorts one contiguous 1/R run of the key list in its own shared memory; the final position of a
//            key is its index in its run plus its lower bounds in the other runs (binary searches through distributed
//            shared memory; keys are unique), and the CTA scatters box / class / index there
//   phase A  the kept list is dealt round-robin over the CTAs (entry e lives in CTA e % R): every CTA tests the whole
//            group against its share, the 512 dead bits are OR-ed through distributed shared memory
//   phase B  the (row, word) items of the batch's suppression mask are dealt round-robin; every CTA stores its words
//            into the mask of CTA 0
//   phase C  greedy scan by one warp of CTA 0; the other CTAs read its survivor list and every CTA appends its share
// One cluster barrier per group and two per batch. The arithmetic of every IoU test and the greedy order are those of
// CL = false: kept rows are bit-identical for every R.
template <bool CL>
__global__ void __launch_bounds__(kNmsThreads, 1) sort_nms_kernel(const NmsArgs g) {
  extern __shared__ __align__(16) uint8_t nsm[];
  __shared__ float red[kNmsThreads / 32], red_mn[kNmsThreads / 32];
  __shared__ int red_cmax[kNmsThreads / 32], red_cmin[kNmsThreads / 32];
  __shared__ int s_nkept, s_ck;
  __shared__ unsigned s_removed[kChunkWords];
  __shared__ unsigned short s_cpos[kChunk];     // sorted position of every batch row, relative to the batch's first group
  __shared__ unsigned s_deadx[CL ? 2 * kNmsMaxCluster * kChunkWords : 1];   // [2][R][16] dead bits found by every CTA
  __shared__ float s_xf[CL ? kNmsMaxCluster * 2 : 1];                   // [R] (max, min) coordinate of every run
  __shared__ int s_xi[CL ? kNmsMaxCluster * 2 : 1];                     // [R] (max, min) class of every run

  const int R = CL ? (int)nms_cluster_nctarank() : 1;
  const int rank = CL ? (int)nms_cluster_ctarank() : 0;
  const int b = CL ? (int)(blockIdx.x / (unsigned)R) : (int)blockIdx.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const long long base = (long long)b * g.src.per_image;
  int n = g.counts[b];
  if (n > g.src.per_image) n = (int)g.src.per_image;

  float4* sbox = g.sorted_box + base;
  int* scls = g.sorted_cls + base;
  int* sidx = g.sorted_idx + base;
  int* kept = g.kept_pos + base;

  if (tid == 0) s_nkept = 0;
  // torchvision.ops.batched_nms: coordinate trick unless boxes.numel() > 100000 (CUDA, torchvision >= 0.19; the installed
  // 0.26 the goldens were generated with) / 4000 (CPU) / 20000 (CUDA, torchvision 0.17.2 = the reference's poetry.lock pin)
  int variant = g.variant;
  if (variant == 3) variant = (4LL * n > 100000) ? 1 : 0;
  if (variant == 4) variant = (4LL * n > 4000) ? 1 : 0;
  if (variant == 5) variant = (4LL * n > 20000) ? 1 : 0;     // torchvision 0.17.2 (the reference's pin) on CUDA

  // (n is the same in every CTA of a cluster: all exits and barrier counts below are uniform over the cluster)
  if (n > 0 && n <= 32 && !g.no_small) {
    if (warp == 0 && rank == 0) nms_small_warp(g, b, n, variant, base);
    return;
  }
  if (n > 0) {
    // ---------------- keys + extrema of the (unsorted) candidates: max coordinate for the offset trick, class window ----
    // run of this CTA: all n candidates, or with a cluster the contiguous 1/R share [lo_r, lo_r + m)
    const int seg = (n + R - 1) / R;
    const int lo_r = min(n, rank * seg), m = min(n, lo_r + seg) - lo_r;
    int P = 1;
    while (P < m) P <<= 1;
    unsigned long long* keys = (CL || P <= g.smem_keys_cap) ? reinterpret_cast<unsigned long long*>(nsm)
                                                           : (g.gkeys + (long long)b * g.gkeys_stride);
    float mx = -INFINITY, mn = INFINITY;
    int cmax = 0, cmin = 0;
    for (int i0 = tid; i0 < m; i0 += 4 * kNmsThreads) {      // four keys, then their four rows, in flight per thread
      unsigned long long k[4];
      float4 bx[4];
      int c[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * kNmsThreads < m) k[u] = nms_key(g, base, lo_r + i0 + u * kNmsThreads);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * kNmsThreads < m) {
          keys[i0 + u * kNmsThreads] = k[u];
          nms_load_row(g, base, (int)(unsigned)(k[u] & 0xffffffffull), bx[u], c[u]);
        }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * kNmsThreads < m) {
          mx = fmaxf(mx, fmaxf(fmaxf(bx[u].x, bx[u].y), fmaxf(bx[u].z, bx[u].w)));
          mn = fminf(mn, fminf(fminf(bx[u].x, bx[u].y), fminf(bx[u].z, bx[u].w)));
          cmax = max(cmax, c[u]); cmin = min(cmin, c[u]);
        }
    }
    {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
      }
      if (lane == 0) { red[warp] = mx; red_mn[warp] = mn; red_cmax[warp] = cmax; red_cmin[warp] = cmin; }
      __syncthreads();                                       // also: the keys are in place
      mx = red[0]; mn = red_mn[0]; cmax = red_cmax[0]; cmin = red_cmin[0];
      for (int i = 1; i < kNmsThreads / 32; ++i) {
        mx = fmaxf(mx, red[i]); mn = fminf(mn, red_mn[i]);
        cmax = max(cmax, red_cmax[i]); cmin = min(cmin, red_cmin[i]);
      }
    }
    if constexpr (CL) {
      // all-reduce of the four extrema over the cluster (max / min are exact in any order); lands with the barrier below
      if (tid < R) {
        float* xf = nms_peer(s_xf, tid);
        int* xi = nms_peer(s_xi, tid);
        xf[rank * 2] = mx; xf[rank * 2 + 1] = mn;
        xi[rank * 2] = cmax; xi[rank * 2 + 1] = cmin;
      }
    }
    // ---------------- sort ----------------
    // merge sort when two key buffers fit the shared memory of the launch (uniform over the cluster: decided on seg)
    const bool use_merge = (keys == reinterpret_cast<unsigned long long*>(nsm)) && (16LL * seg <= (long long)g.smem_bytes);
    unsigned long long* const keys0 = keys;
    if (use_merge) keys = merge_sort_keys(keys, keys + seg, m, tid);
    else sort_keys_asc(keys, m, tid);
    if constexpr (CL) {
      nms_cluster_sync();                                    // every run is final, extrema exchanged
      for (int rr = 0; rr < R; ++rr) {
        mx = fmaxf(mx, s_xf[rr * 2]); mn = fminf(mn, s_xf[rr * 2 + 1]);
        cmax = max(cmax, s_xi[rr * 2]); cmin = min(cmin, s_xi[rr * 2 + 1]);
      }
    }
    // ---------------- gather the sorted candidates (four rows in flight per thread) ----------------
    // boxes_for_nms = boxes + idxs.to(boxes) * (max_coordinate + 1)   (torchvision boxes.py) for the offset variant.
    // With a cluster the position of a key is its index in the own run plus its lower bounds in the other runs
    // (binary searches through distributed shared memory, four keys in lock-step; the keys are unique).
    const float step = __fadd_rn(mx, 1.0f);
    for (int i0 = tid; i0 < m; i0 += 4 * kNmsThreads) {
      unsigned long long k[4];
      int pos[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * kNmsThreads;
        pos[u] = i;
        k[u] = i < m ? keys[i] : 0ull;
      }
      if constexpr (CL) {
        for (int rr = 0; rr < R; ++rr) {
          if (rr == rank) continue;
          const int lo2 = min(n, rr * seg), m2 = min(n, lo2 + seg) - lo2;
          const unsigned long long* run = nms_peer(keys0, rr) + ((use_merge && merge_sorted_in_tmp(m2)) ? seg : 0);
          int l[4] = {0, 0, 0, 0}, h[4] = {m2, m2, m2, m2};
          for (int st = 32 - __clz(m2); st > 0; --st) {     // an interval of m2 closes in <= floor(log2 m2) + 1 halvings
            unsigned long long v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = l[u] < h[u] ? run[(l[u] + h[u]) >> 1] : 0ull;
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (l[u] < h[u]) {
                const int mid = (l[u] + h[u]) >> 1;
                if (v[u] < k[u]) l[u] = mid + 1; else h[u] = mid;
              }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) pos[u] += l[u];        // keys of run rr below k
        }
      }
      float4 bx[4];
      int c[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * kNmsThreads < m) nms_load_row(g, base, (int)(unsigned)(k[u] & 0xffffffffull), bx[u], c[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * kNmsThreads < m) {
          if (variant == 0) {
            const float off = __fmul_rn((float)c[u], step);
            bx[u].x = __fadd_rn(bx[u].x, off); bx[u].y = __fadd_rn(bx[u].y, off);
            bx[u].z = __fadd_rn(bx[u].z, off); bx[u].w = __fadd_rn(bx[u].w, off);
          }
          sbox[pos[u]] = bx[u]; scls[pos[u]] = c[u]; sidx[pos[u]] = (int)(unsigned)(k[u] & 0xffffffffull);
        }
    }
    if constexpr (CL) nms_cluster_sync(); else __syncthreads();   // sorted rows visible; runs no longer read

    // ---------------- greedy NMS: groups of 512 candidates, batches of survivors ----------------
    // Which pairs can interact?  per-class variant: equal classes only.  Offset variant: class c lives in
    // [c*s + min, c*s + max] with s = max+1, so classes a < b can only overlap when (b-a)*s < max-min+1,
    // i.e. |a-b| <= J with J = ceil((max-min+1)/s) - 1 (J = 0 when no coordinate is negative; J = 1 for
    // ordinary scenes with boxes sticking out of the image).  Pairs outside the window have IoU == 0 in
    // torchvision's own arithmetic, so skipping them is exact.  Class-agnostic: everything interacts.
    //
    // shared memory (the sort buffer is dead now):
    //   batch : box/area/class of up to 512 phase-A survivors, their 512x512 suppression bitmask, the rows kept by the scan
    //   kept  : boxes already kept (box, area, class) with a linked list per class; with a cluster, this CTA's share
    //           (global entry e = slot * R + rank)
    float4* cbox = reinterpret_cast<float4*>(nsm);                          // [kChunk]
    float* carea = reinterpret_cast<float*>(nsm + kChunk * 16);              // [kChunk]
    int* ccls = reinterpret_cast<int*>(nsm + kChunk * 20);                   // [kChunk]
    unsigned* cmask = reinterpret_cast<unsigned*>(nsm + kChunk * 24);        // [kChunk][kMaskPitch]
    int* ck = reinterpret_cast<int*>(nsm + kChunkBytes);                     // [kChunk] kept rows of the batch
    int* khead = ck + kChunk;                                                // [kClassCap] list heads
    // bounds of a class's kept boxes (orderable_f32): max over the list of min(x2, y2), min over the list of max(x1, y1).
    // A box whose min(x1, y1) is not below the first, or whose max(x2, y2) is not above the second, overlaps no entry in
    // x or in y -- its IoU with every entry is 0 in torchvision's own arithmetic -- and skips the list. With the offset
    // trick's class window J = 1 (any scene with a coordinate below zero) that removes the two neighbour lists.
    unsigned* kmaxlo = reinterpret_cast<unsigned*>(khead + kClassCap);       // [kClassCap]
    unsigned* kminhi = kmaxlo + kClassCap;                                   // [kClassCap]
    uint8_t* kbase = reinterpret_cast<uint8_t*>(kminhi + kClassCap);
    const int KC = g.kept_cap;
    float4* kbox = reinterpret_cast<float4*>(kbase);                          // [KC]
    int* kmeta = reinterpret_cast<int*>(kbase + (size_t)KC * 16);             // [KC] class, or class | (next + 1) << 10 with lists
    unsigned* cmask_w = (CL && rank != 0) ? nms_peer(cmask, 0) : cmask;       // phase B stores into CTA 0's mask

    int J = 0x3fffffff;                                   // class window; "infinite" = ungated
    if (variant == 1) J = 0;
    else if (variant == 0) {
      const float sft = mx + 1.0f;
      if (sft > 0.0f) {
        const float ratio = (mx - mn + 1.0f) / sft + 1e-3f;
        if (ratio < 64.0f) J = max(0, (int)ceilf(ratio) - 1);
      }
    }
    const bool use_lists = (J <= 4) && cmin >= 0 && cmax < kClassCap;
    for (int i = tid; i < kClassCap; i += kNmsThreads) { khead[i] = -1; kmaxlo[i] = 0u; kminhi[i] = 0xffffffffu; }

    // The sorted candidates are walked in groups of 512 (thread t owns candidate g0 + t). Phase A tests a group against
    // the boxes kept so far; its survivors are appended, in order, to a BATCH of up to 512 rows. Only a batch goes through
    // the suppression mask (phase B) and the greedy scan (phase C): in a dense scene most candidates die in phase A, so
    // one batch collects the survivors of several groups and B / C run a few times instead of once per group. This is
    // exact: the survivors of a later group were not tested against the keeps of the pending batch, but those keeps are
    // rows of the same batch and suppress them through the mask. A group whose survivors do not fit the batch is tested
    // again after the batch has been resolved (against the longer kept list).
    float4 cur_box = make_float4(0, 0, 0, 0), nx_box = cur_box;          // rows of this group / the next (loaded ahead)
    int cur_cls = -1, nx_cls = -1;
    if (tid < n) { cur_box = sbox[tid]; cur_cls = scls[tid]; }
    if (kChunk + tid < n) { nx_box = sbox[kChunk + tid]; nx_cls = scls[kChunk + tid]; }
    int g0 = 0;                       // first candidate of the group
    int nb = 0, cbase = 0;            // rows in the batch; sorted position of its first group (s_cpos is relative to it)
    unsigned turn = 0;                // phase-A executions so far: parity selects the dead-bit exchange buffer
    while (g0 < n || nb > 0) {
      __syncthreads();
      const int nk = s_nkept;
      const int nk_own = (nk + R - 1 - rank) / R;        // entries of the kept list this CTA holds
      bool flush = true;
      if (g0 < n) {
        const int gn = min(kChunk, n - g0);
        const float4 me = cur_box;
        const int my_cls = cur_cls;
        const float my_area = box_area(me);
        bool dead = (tid >= gn);
        // ---- phase A: against the boxes kept so far
        if (!dead) {
          const int nks = min(nk_own, KC);
          if (use_lists) {
            // (the next entry of a list is loaded while the IoU of the current one is computed)
            const unsigned my_lo = orderable(fminf(me.x, me.y)), my_hi = orderable(fmaxf(me.z, me.w));
            for (int c2 = max(my_cls - J, 0); c2 <= min(my_cls + J, kClassCap - 1) && !dead; ++c2) {
              if (g.thr >= 0.0f && (my_lo >= kmaxlo[c2] || my_hi <= kminhi[c2])) continue;
              int k = khead[c2];
              float4 kb = make_float4(0, 0, 0, 0);
              int meta = 0;
              if (k >= 0) { kb = kbox[k]; meta = kmeta[k]; }
              while (k >= 0) {
                const int kn = (meta >> 10) - 1;
                float4 kbn = kb;
                int metan = 0;
                if (kn >= 0) { kbn = kbox[kn]; metan = kmeta[kn]; }
                if (suppresses(kb, box_area(kb), me, my_area, g.thr)) { dead = true; break; }
                k = kn; kb = kbn; meta = metan;
              }
            }
          } else {
            for (int k = 0; k < nks; ++k) {
              if (abs(kmeta[k] - my_cls) > J) continue;
              const float4 kb = kbox[k];
              if (suppresses(kb, box_area(kb), me, my_area, g.thr)) { dead = true; break; }
            }
          }
          for (int k = KC; k < nk_own && !dead; ++k) {       // overflow of the shared-memory list
            const int kp = kept[k * R + rank];
            if (abs(scls[kp] - my_cls) > J) continue;
            const float4 kb = sbox[kp];
            if (suppresses(kb, box_area(kb), me, my_area, g.thr)) dead = true;
          }
        }
        {
          const unsigned bal = __ballot_sync(0xffffffffu, dead);
          if constexpr (CL) {
            // double buffered by turn: a CTA that runs ahead writes the next group's bits while this one still reads
            unsigned* dx = s_deadx + (turn & 1u) * (kNmsMaxCluster * kChunkWords);
            if (lane < R) nms_peer(dx, lane)[rank * kChunkWords + warp] = bal;
            nms_cluster_sync();                              // (1) every CTA's dead bits have arrived
            if (tid < kChunkWords) {
              unsigned u = 0u;
              for (int rr = 0; rr < R; ++rr) u |= dx[rr * kChunkWords + tid];
              s_removed[tid] = u;
            }
          } else {
            if (lane == 0) s_removed[warp] = bal;
          }
          ++turn;
        }
        __syncthreads();
        // survivors of the group and this thread's place among them (uniform counts: every thread reads the 16 words)
        int surv = 0, before = 0;
#pragma unroll
        for (int l = 0; l < kChunkWords; ++l) {
          const int pc = __popc(~s_removed[l]);
          surv += pc;
          before += l < warp ? pc : 0;
        }
        const bool alive = !((s_removed[warp] >> lane) & 1u);
        if (nb + surv <= kChunk) {
          if (nb == 0) cbase = g0;
          if (alive) {
            const int row = nb + before + __popc(~s_removed[warp] & ((1u << lane) - 1u));
            cbox[row] = me; carea[row] = my_area; ccls[row] = my_cls;
            s_cpos[row] = (unsigned short)(g0 + tid - cbase);
          }
          nb += surv;
          g0 += kChunk;
          cur_box = nx_box; cur_cls = nx_cls;
          if (g0 + kChunk + tid < n) { nx_box = sbox[g0 + kChunk + tid]; nx_cls = scls[g0 + kChunk + tid]; }
          // resolve the batch when it is nearly full, at the end of the list, or before its 16-bit positions run out
          flush = nb >= kFlushRows || g0 >= n || g0 - cbase > 60000;
        }
        // else: the batch is resolved first and the group tested again
      }
      if (!flush || nb == 0) continue;

      const int cn = nb;
      const int nw = (cn + 31) >> 5;
      // ---- phase B: suppression bitmask inside the batch (row i, bits j > i)
      {
        __syncthreads();
        // items (row, word): 16 per row, the words before the row's own are skipped; with a cluster the items are
        // dealt round-robin over the CTAs and stored into CTA 0's mask
        const int items = cn << 4;
        for (int q = rank * kNmsThreads + tid; q < items; q += R * kNmsThreads) {
          const int row = q >> 4;
          const int w = q & (kChunkWords - 1);
          if (w < (row >> 5) || w >= nw) continue;
          const float4 rbx = cbox[row];
          const float rar = carea[row];
          const int rcl = ccls[row];
          // columns of the word that come after the row and exist
          const int lo_bit = row + 1 - w * 32, hi_bit = cn - w * 32;
          unsigned m = (hi_bit >= 32 ? 0xffffffffu : ((1u << hi_bit) - 1u)) & (lo_bit <= 0 ? 0xffffffffu : (lo_bit >= 32 ? 0u : (0xffffffffu << lo_bit)));
          if (J != 0x3fffffff && __popc(m) > 8) {
            // class gate first, as a bit mask (the lanes of a warp hold up to 16 different words: column jb + w of
            // the word is read in step jb, so that the lanes hit different banks), ...
            unsigned gate = 0u;
#pragma unroll 8
            for (int jb = 0; jb < 32; ++jb) {
              const int jc = (jb + w) & 31;
              if (abs(ccls[w * 32 + jc] - rcl) <= J) gate |= (1u << jc);
            }
            m &= gate;
          }
          // ... then the IoU of the few pairs inside the class window only (a warp runs as many steps as its
          // fullest lane has pairs, instead of the IoU path in nearly every one of 32 steps)
          unsigned bits = 0u;
          while (m) {
            const int jb = __ffs(m) - 1;
            m &= m - 1u;
            const int j = w * 32 + jb;
            if (abs(ccls[j] - rcl) <= J && suppresses(rbx, rar, cbox[j], carea[j], g.thr)) bits |= (1u << jb);
          }
          cmask_w[row * kMaskPitch + w] = bits;
        }
        if constexpr (CL) nms_cluster_sync(); else __syncthreads();   // (2) CTA 0 holds the whole mask
      }
      // ---- phase C: one warp walks the batch word by word (32 rows); lane l owns word l of the removed set (at the
      //      start: the rows past the end of the batch). Inside a word the greedy order is resolved on the 32x32 diagonal
      //      block held in registers; the rows of the kept boxes are then OR-ed into the later words.
      if (warp == 0 && rank == 0) {
        unsigned removed = 0xffffffffu;
        if (lane < nw) removed = (cn - lane * 32 >= 32) ? 0u : (0xffffffffu << (cn - lane * 32));
        int cnt = 0;
        const int nwords = nw;
        for (int w = 0; w < nwords; ++w) {
          unsigned a = ~__shfl_sync(0xffffffffu, removed, w);          // alive candidates of word w
          if (a == 0u) continue;       // (a ballot that jumps to the next alive word measured slower: 104k vs 95k clk)
          if (__popc(a) <= 6) {
            // few alive candidates: hop from kept box to kept box; every lane reads the diagonal word of the kept row
            // (broadcast) and its own later word
            while (a) {
              const int i = __ffs(a) - 1;
              const unsigned* rowp = cmask + (w * 32 + i) * kMaskPitch;
              const unsigned diag = rowp[w];
              const unsigned r = (lane > w && lane < nwords) ? rowp[lane] : 0u;
              if (lane == 0) ck[cnt] = w * 32 + i;
              ++cnt;
              a &= ~(diag | (1u << i));
              removed |= r;
            }
            continue;
          }
          const unsigned dj = cmask[(w * 32 + lane) * kMaskPitch + w];  // row (w*32 + lane), bits of the same word
          unsigned keptw = a;
          // common case: no alive box of the word suppresses another alive box of the word
          if (__any_sync(0xffffffffu, ((a >> lane) & 1u) && (dj & a) != 0u)) {
            // 32 fixed steps: the shuffles do not depend on the chain, each step is a test + and-not
            keptw = 0u;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const unsigned di = __shfl_sync(0xffffffffu, dj, i);
              if ((a >> i) & 1u) { keptw |= 1u << i; a &= ~di; }
            }
          }
          const bool mine = (keptw >> lane) & 1u;
          if (mine) {
            const int slot = cnt + __popc(keptw & ((1u << lane) - 1u));
            ck[slot] = w * 32 + lane;
          }
          cnt += __popc(keptw);
          // rows of the kept boxes OR-ed into the later words. Few kept boxes: lane l walks the kept rows and ORs word
          // l of each (independent loads). Many: lane i contributes its row, one warp reduction per later word. Same
          // result either way.
          if (__popc(keptw) < nwords - 1 - w) {
            if (lane > w && lane < nwords) {
              unsigned r = 0u;
              for (unsigned mk = keptw; mk; mk &= mk - 1u) r |= cmask[(w * 32 + __ffs(mk) - 1) * kMaskPitch + lane];
              removed |= r;
            }
          } else {
            for (int l = w + 1; l < nwords; ++l) {
              const unsigned r = __reduce_or_sync(0xffffffffu, mine ? cmask[(w * 32 + lane) * kMaskPitch + l] : 0u);
              if (lane == l) removed |= r;
            }
          }
        }
        if (lane == 0) s_ck = cnt;
      }
      if constexpr (CL) nms_cluster_sync(); else __syncthreads();     // (3) CTA 0 has the batch's survivors
      // ---- append the batch's survivors to the kept list (parallel; list order is irrelevant)
      {
        // (the other CTAs read CTA 0's list: it is rewritten only after barrier (2) of the next batch)
        const int cnt = (CL && rank != 0) ? *nms_peer(&s_ck, 0) : s_ck;
        if (tid < cnt) {
          const int i = (CL && rank != 0) ? nms_peer(ck, 0)[tid] : ck[tid];
          const int e = nk + tid;
          if (rank == 0) kept[e] = cbase + (int)s_cpos[i];
          const int slot = e / R;
          if (e - slot * R == rank && slot < KC) {
            const int ci = ccls[i];
            kbox[slot] = cbox[i];
            kmeta[slot] = use_lists ? (ci | ((atomicExch(&khead[ci], slot) + 1) << 10)) : ci;
            if (use_lists) {
              const float4 kb = cbox[i];
              float lo = fminf(kb.z, kb.w), hi = fmaxf(kb.x, kb.y);
              if (!(kb.x == kb.x && kb.y == kb.y && kb.z == kb.z && kb.w == kb.w)) { lo = INFINITY; hi = -INFINITY; }   // NaN: never skipped
              atomicMax(&kmaxlo[ci], orderable(lo));
              atomicMin(&kminhi[ci], orderable(hi));
            }
          }
        }
        if (tid == 0) s_nkept = nk + cnt;
      }
      nb = 0;
      __syncthreads();
    }
    if constexpr (CL) nms_cluster_sync();   // the other CTAs have read the last batch's survivors from CTA 0
  }
  __syncthreads();
  if (rank != 0) return;

  // ---------------- outputs ----------------
  const int nk = s_nkept;
  if (g.keep) {
    for (int k = tid; k < nk; k += kNmsThreads) g.keep[base + k] = sidx[kept[k]];
    if (tid == 0) g.keep_count[b] = nk;
  }
  if (g.dets) {
    const int m = min(nk, g.max_det);
    for (int k = tid; k < m; k += kNmsThreads) {
      const int idx = sidx[kept[k]];
      const float4* crow = reinterpret_cast<const float4*>(g.src.boxes + (base + idx) * 8);
      const float4 r0 = crow[0], r1 = crow[1];
      float* d = g.dets + ((long long)b * g.max_det + k) * 7;
      d[0] = r0.x; d[1] = r0.y; d[2] = r0.z; d[3] = r0.w; d[4] = r1.x; d[5] = r1.y; d[6] = r1.z;
      if (g.det_idx) g.det_idx[(long long)b * g.max_det + k] = idx;
    }
    if (tid == 0) g.det_count[b] = nk;  // true number kept; rows beyond max_det are dropped
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static inline long long next_pow2_ll(long long v) { long long p = 1; while (p < v) p <<= 1; return p; }
static inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

struct PostWs {
  float* cand; unsigned long long* keys; unsigned long long* gkeys; float4* sbox;
  int* scls; int* sidx; int* kept; int* counts;
  size_t total;
};

static PostWs carve_ws(void* ws, int batch, long long per_image) {
  PostWs w;
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  size_t off = 0;
  const long long padded = per_image > kMaxSmemKeys ? next_pow2_ll(per_image) : per_image;
  w.counts = reinterpret_cast<int*>(p + off); off += align256((size_t)batch * 4);
  w.cand = reinterpret_cast<float*>(p + off); off += align256((size_t)batch * per_image * 32);
  w.keys = reinterpret_cast<unsigned long long*>(p + off); off += align256((size_t)batch * per_image * 8);
  w.gkeys = reinterpret_cast<unsigned long long*>(p + off);
  off += align256(per_image > kMaxSmemKeys ? (size_t)batch * padded * 8 : 256);
  w.sbox = reinterpret_cast<float4*>(p + off); off += align256((size_t)batch * per_image * 16);
  w.scls = reinterpret_cast<int*>(p + off); off += align256((size_t)batch * per_image * 4);
  w.sidx = reinterpret_cast<int*>(p + off); off += align256((size_t)batch * per_image * 4);
  w.kept = reinterpret_cast<int*>(p + off); off += align256((size_t)batch * per_image * 4);
  w.total = off;
  return w;
}

long long postprocess_ws_bytes(int batch, int anchors) {
  if (batch <= 0 || anchors <= 0) return 256;
  return (long long)carve_ws(nullptr, batch, anchors).total;
}

static float thr_for_strict_gt(double nms_thre) {
  // torchvision's CPU kernel compares the fp32 IoU with the double threshold:
  // x > thr  <=>  x > f, where f is the largest float that is <= thr
  float f = (float)nms_thre;
  if ((double)f > nms_thre) f = nextafterf(f, -INFINITY);
  return f;
}

static int smem_keys_cap(long long per_image) {
  const long long p = next_pow2_ll(per_image);
  return (int)(p > kMaxSmemKeys ? kMaxSmemKeys : p);
}
static int kept_cap_for(long long per_image) {
  const long long budget = kNmsSmemBudget - kNmsFixedBytes;
  long long cap = budget / kKeptEntryBytes;
  if (cap > per_image) cap = per_image;
  return (int)(cap < 1 ? 1 : cap);
}
static size_t nms_smem_bytes(long long per_image) {
  const size_t sort_bytes = (size_t)smem_keys_cap(per_image) * 8;
  const size_t nms_bytes = (size_t)kNmsFixedBytes + (size_t)kept_cap_for(per_image) * kKeptEntryBytes;
  return sort_bytes > nms_bytes ? sort_bytes : nms_bytes;
}

// Cluster size for the batch: the largest of 8 / 4 / 2 whose batch clusters are co-resident (one CTA per SM at this
// shared-memory size; asked from the occupancy API once per device), 1 otherwise. Small candidate capacities and key
// lists beyond shared memory stay on the single-CTA kernel. YX_NMS_CLUSTER=<1|2|4|8> caps it (tests compare the paths).
static int nms_cluster_size(int batch, long long per_image, size_t smem) {
  if (per_image <= 2 * kChunk || per_image > kMaxSmemKeys) return 1;
  int cap = kNmsMaxCluster;
  if (const char* e = getenv("YX_NMS_CLUSTER")) { cap = atoi(e); if (cap < 1) cap = 1; }
  static int max_clusters_dev[kMaxDevices][4] = {};          // [device][log2 R]: co-resident clusters, 0 = not asked yet
  static size_t asked_smem_dev[kMaxDevices] = {};
  const int slot = current_device_slot();
  if (asked_smem_dev[slot] != smem) { memset(max_clusters_dev[slot], 0, sizeof(max_clusters_dev[slot])); asked_smem_dev[slot] = smem; }
  for (int lg = 3; lg >= 1; --lg) {
    const int R = 1 << lg;
    if (R > cap) continue;
    int& mc = max_clusters_dev[slot][lg];
    if (mc == 0) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)R * 16u, 1, 1); cfg.blockDim = dim3(kNmsThreads, 1, 1); cfg.dynamicSmemBytes = smem;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)R; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      int got = 0;
      if (cudaOccupancyMaxActiveClusters(&got, sort_nms_kernel<true>, &cfg) != cudaSuccess) { cudaGetLastError(); got = 0; }
      mc = got > 0 ? got : -1;
    }
    if (mc >= batch) return R;
  }
  return 1;
}

static int launch_sort_nms(NmsArgs& g, int batch, cudaStream_t s) {
  g.smem_keys_cap = smem_keys_cap(g.src.per_image);
  g.kept_cap = kept_cap_for(g.src.per_image);
  g.gkeys_stride = next_pow2_ll(g.src.per_image);
  g.no_small = getenv("YX_NMS_NO_SMALL") ? 1 : 0;
  const size_t smem = nms_smem_bytes(g.src.per_image);
  g.smem_bytes = (int)smem;
  static size_t configured_dev[kMaxDevices] = {};
  size_t& configured = configured_dev[current_device_slot()];
  if (smem > configured) {
    YX_CUDA(cudaFuncSetAttribute(sort_nms_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    YX_CUDA(cudaFuncSetAttribute(sort_nms_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const int R = nms_cluster_size(batch, g.src.per_image, smem);
  if (R > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(batch * R), 1, 1); cfg.blockDim = dim3(kNmsThreads, 1, 1);
    cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)R; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    YX_CUDA(cudaLaunchKernelEx(&cfg, sort_nms_kernel<true>, (const NmsArgs)g));
  } else {
    sort_nms_kernel<false><<<batch, kNmsThreads, smem, s>>>(g);
  }
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int filter_launch(float* pred, int batch, int anchors, int nc, float conf_thre, int inplace_xyxy, const PostWs& w,
                  cudaStream_t s) {
  YX_CUDA(cudaMemsetAsync(w.counts, 0, (size_t)batch * 4, s));
  const int chunks = (anchors + kFilterAnchors - 1) / kFilterAnchors;
  const size_t smem = (size_t)kFilterAnchors * (5 + nc) * sizeof(float);
  YX_REQUIRE(smem <= 200 * 1024, YX_ERR_UNSUPPORTED, "postprocess: %d classes exceed the shared-memory row staging", nc);
  static size_t configured_dev[kMaxDevices] = {};
  size_t& configured = configured_dev[current_device_slot()];
  if (configured == 0) configured = 48 * 1024;
  if (smem > configured) {
    YX_CUDA(cudaFuncSetAttribute(filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  filter_kernel<<<batch * chunks, kFilterAnchors, smem, s>>>(pred, batch, anchors, nc, conf_thre, inplace_xyxy, w.cand,
                                                             w.keys, w.counts);
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int postprocess_launch(float* pred, int batch, int anchors, int nc, float conf_thre, double nms_thre, int nms_variant,
                       int inplace_xyxy, float* dets, long long* det_idx, int* det_count, int max_det, void* ws,
                       long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(pred && dets && det_count && ws, YX_ERR_INVALID_ARG, "postprocess: null pointer");
  YX_REQUIRE(batch > 0 && anchors > 0 && nc > 0 && max_det > 0, YX_ERR_INVALID_ARG, "postprocess: bad sizes");
  YX_REQUIRE(nms_variant >= 0 && nms_variant <= 5, YX_ERR_INVALID_ARG, "postprocess: nms_variant must be 0..5");
  YX_REQUIRE(((uintptr_t)ws & 255) == 0, YX_ERR_INVALID_ARG, "postprocess: workspace must be 256-byte aligned");
  PostWs w = carve_ws(ws, batch, anchors);
  YX_REQUIRE((long long)w.total <= ws_bytes, YX_ERR_CAPACITY, "postprocess: workspace %lld < %lld bytes", ws_bytes, (long long)w.total);
  int rc = filter_launch(pred, batch, anchors, nc, conf_thre, inplace_xyxy, w, s);
  if (rc) return rc;
  NmsArgs g;
  memset(&g, 0, sizeof(g));
  g.src.boxes = w.cand; g.src.box_stride = 8;
  g.src.scores = w.cand + 7; g.src.score_stride = 8;
  g.src.cls = w.cand + 6; g.src.cls_stride = 8; g.src.cls_is_float = 1; g.src.cand_rows = 1;
  g.src.per_image = anchors;
  g.keys = w.keys; g.counts = w.counts;
  g.thr = thr_for_strict_gt(nms_thre);
  g.variant = nms_variant;
  g.gkeys = w.gkeys; g.sorted_box = w.sbox; g.sorted_cls = w.scls; g.sorted_idx = w.sidx; g.kept_pos = w.kept;
  g.dets = dets; g.det_idx = det_idx; g.det_count = det_count; g.max_det = max_det;
  return launch_sort_nms(g, batch, s);
}

int postprocess_ws_ptrs(void* ws, int batch, int anchors, float** cand, unsigned long long** keys, int** counts) {
  YX_REQUIRE(ws && batch > 0 && anchors > 0, YX_ERR_INVALID_ARG, "postprocess_workspace_ptrs: bad arguments");
  YX_REQUIRE(((uintptr_t)ws & 255) == 0, YX_ERR_INVALID_ARG, "postprocess: workspace must be 256-byte aligned");
  PostWs w = carve_ws(ws, batch, anchors);
  if (cand) *cand = w.cand;
  if (keys) *keys = w.keys;
  if (counts) *counts = w.counts;
  return YX_OK;
}

int postprocess_begin_launch(void* ws, int batch, int anchors, cudaStream_t s) {
  YX_REQUIRE(ws && batch > 0 && anchors > 0, YX_ERR_INVALID_ARG, "postprocess_begin: bad arguments");
  PostWs w = carve_ws(ws, batch, anchors);
  YX_CUDA(cudaMemsetAsync(w.counts, 0, (size_t)batch * 4, s));
  return YX_OK;
}

// Stage 2 only: the head epilogues (YX_EPI_HEAD with head_cand) have filled cand / keys / counts.
int nms_prefiltered_launch(int batch, int anchors, double nms_thre, int nms_variant, float* dets, long long* det_idx,
                           int* det_count, int max_det, void* ws, long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(dets && det_count && ws, YX_ERR_INVALID_ARG, "nms_prefiltered: null pointer");
  YX_REQUIRE(batch > 0 && anchors > 0 && max_det > 0, YX_ERR_INVALID_ARG, "nms_prefiltered: bad sizes");
  YX_REQUIRE(nms_variant >= 0 && nms_variant <= 5, YX_ERR_INVALID_ARG, "nms_prefiltered: nms_variant must be 0..5");
  YX_REQUIRE(((uintptr_t)ws & 255) == 0, YX_ERR_INVALID_ARG, "nms_prefiltered: workspace must be 256-byte aligned");
  PostWs w = carve_ws(ws, batch, anchors);
  YX_REQUIRE((long long)w.total <= ws_bytes, YX_ERR_CAPACITY, "nms_prefiltered: workspace %lld < %lld bytes", ws_bytes, (long long)w.total);
  NmsArgs g;
  memset(&g, 0, sizeof(g));
  g.src.boxes = w.cand; g.src.box_stride = 8;
  g.src.scores = w.cand + 7; g.src.score_stride = 8;
  g.src.cls = w.cand + 6; g.src.cls_stride = 8; g.src.cls_is_float = 1; g.src.cand_rows = 1;
  g.src.per_image = anchors;
  g.keys = w.keys; g.counts = w.counts;
  g.thr = thr_for_strict_gt(nms_thre);
  g.variant = nms_variant;
  g.gkeys = w.gkeys; g.sorted_box = w.sbox; g.sorted_cls = w.scls; g.sorted_idx = w.sidx; g.kept_pos = w.kept;
  g.dets = dets; g.det_idx = det_idx; g.det_count = det_count; g.max_det = max_det;
  return launch_sort_nms(g, batch, s);
}

int filter_compact_launch(const float* pred, int batch, int anchors, int nc, float conf_thre, float* cand,
                          int* cand_idx, int* cand_count, void* ws, long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(pred && cand && cand_idx && cand_count && ws, YX_ERR_INVALID_ARG, "filter: null pointer");
  YX_REQUIRE(batch > 0 && anchors > 0 && nc > 0, YX_ERR_INVALID_ARG, "filter: bad sizes");
  PostWs w = carve_ws(ws, batch, anchors);
  YX_REQUIRE((long long)w.total <= ws_bytes, YX_ERR_CAPACITY, "filter: workspace %lld < %lld bytes", ws_bytes, (long long)w.total);
  int rc = filter_launch(const_cast<float*>(pred), batch, anchors, nc, conf_thre, 0, w, s);
  if (rc) return rc;
  compact_kernel<<<batch, 1024, 0, s>>>(w.cand, anchors, conf_thre, cand, cand_idx, cand_count);
  YX_CUDA(cudaGetLastError());
  return YX_OK;
}

int batched_nms_launch(const float* boxes, const float* scores, const int* cls, const int* counts, int batch,
                       int n_max, double nms_thre, int nms_variant, int* keep, int* keep_count, void* ws,
                       long long ws_bytes, cudaStream_t s) {
  YX_REQUIRE(boxes && scores && cls && counts && keep && keep_count && ws, YX_ERR_INVALID_ARG, "nms: null pointer");
  YX_REQUIRE(batch > 0 && n_max > 0, YX_ERR_INVALID_ARG, "nms: bad sizes");
  YX_REQUIRE(nms_variant >= 0 && nms_variant <= 5, YX_ERR_INVALID_ARG, "nms: nms_variant must be 0..5");
  PostWs w = carve_ws(ws, batch, n_max);
  YX_REQUIRE((long long)w.total <= ws_bytes, YX_ERR_CAPACITY, "nms: workspace %lld < %lld bytes", ws_bytes, (long long)w.total);
  NmsArgs g;
  memset(&g, 0, sizeof(g));
  g.src.boxes = boxes; g.src.box_stride = 4;
  g.src.scores = scores; g.src.score_stride = 1;
  g.src.cls = cls; g.src.cls_stride = 1; g.src.cls_is_float = 0;
  g.src.per_image = n_max;
  g.keys = nullptr; g.counts = counts;
  g.thr = thr_for_strict_gt(nms_thre);
  g.variant = nms_variant;
  g.gkeys = w.gkeys; g.sorted_box = w.sbox; g.sorted_cls = w.scls; g.sorted_idx = w.sidx; g.kept_pos = w.kept;
  g.keep = keep; g.keep_count = keep_count;
  return launch_sort_nms(g, batch, s);
}

}  // namespace yx
