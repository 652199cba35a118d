// Gradient all-reduce + SGD (momentum, nesterov, weight decay) + EMA as ONE kernel over NVLink peer memory.
//
// Replaces, for the data-parallel training step on the GPUs of one node, the sequence
//   ncclAllReduce(gradients)                       torch DDP, yolox/core/trainer.py:169 (model = DDP(model, ...))
//   optimizer.step()                               yolox/core/trainer.py:119-121, SGD built by yolox/config.py:307-333
//   ema_model.update(model)                        yolox/core/trainer.py:123-124, yolox/utils/ema.py:46-58
// Every rank keeps its gradients in one flat fp32 buffer allocated as SYMMETRIC memory (torch.distributed._symmetric_memory:
// the same allocation on every rank, each mapped into every peer's address space over NVLink / NVSwitch); the kernel reads and
// writes the peers' buffers directly with ordinary loads / stores.
//
//   barrier A   every rank has finished its backward (its gradient buffer is complete)
//   phase 1     reduce-scatter: rank r sums slice r of the flat buffer over all ranks in rank order (fixed order: the result
//               does not depend on timing), scales by 1 / world and writes it back into slice r of ITS OWN buffer
//   barrier B   every slice is reduced
//   phase 2     all-gather fused with the update: every rank walks all parameter chunks and reads the reduced gradient of
//               each element from the rank that owns its slice (7/8 of the reads cross NVLink), then applies the SGD + EMA
//               arithmetic of sgd_ema_kernel
//   barrier C   every rank has finished reading: the buffers may be zeroed for the next step
// A barrier = grid-wide arrival on the local GPU (counter + sense in device memory; the launch is sized to be co-resident),
// then the last CTA exchanges an epoch number with every peer through a small symmetric flag array (st.release.sys /
// ld.acquire.sys), then releases the local CTAs. All spins are bounded and trap.
#include <stdlib.h>
#include <string.h>

#include "yx_common.cuh"

namespace yx {

static constexpr int kArThreads = 256;
static constexpr int kArMaxWorld = 16;

struct ArSgdParams {
  const long long* table; const int* chunks; int n_chunks; int chunk_elems;
  float momentum; int nesterov; int first_step; const float* hyper;
  long long peer_grad[kArMaxWorld];     // flat gradient buffer of every rank (peer-mapped addresses; [rank] is the local one)
  long long peer_flag[kArMaxWorld];     // flag array (uint32 [world]) of every rank: flag[r] on rank q = last epoch r announced to q
  long long flat_elems;
  int rank, world;
  unsigned* state;                      // local: [0] arrival count, [1] sense, [2] epoch
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// grid-wide + cross-GPU barrier; `sense` is the value the local sense word takes, `epoch` the number exchanged with the peers.
// wait_local == false (last barrier): the CTAs that are not last leave at once, only the last one waits for the peers.
__device__ __forceinline__ void ar_barrier(const ArSgdParams& p, unsigned sense, unsigned epoch, bool wait_local) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned old = atomicAdd(&p.state[0], 1u);
    if (old == gridDim.x - 1) {
      p.state[0] = 0;
      for (int q = 0; q < p.world; ++q)
        if (q != p.rank) st_release_sys(reinterpret_cast<unsigned*>(p.peer_flag[q]) + p.rank, epoch);
      const unsigned* mine = reinterpret_cast<const unsigned*>(p.peer_flag[p.rank]);
      for (int q = 0; q < p.world; ++q) {
        if (q == p.rank) continue;
        unsigned spins = 0;
        while ((int)(ld_acquire_sys(mine + q) - epoch) < 0) {
          __nanosleep(100);
          if (++spins > (1u << 24)) { printf("yx_b200: all-reduce barrier timed out (rank %d waits for rank %d, epoch %u)\n", p.rank, q, epoch); __trap(); }
        }
      }
      __threadfence_system();
      atomicExch(&p.state[1], sense);
    } else if (wait_local) {
      unsigned spins = 0;
      while (*reinterpret_cast<volatile unsigned*>(&p.state[1]) != sense) {
        __nanosleep(100);
        if (++spins > (1u << 24)) { printf("yx_b200: all-reduce grid barrier timed out (block %d)\n", (int)blockIdx.x); __trap(); }
      }
      __threadfence_system();
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kArThreads)
allreduce_sgd_ema_kernel(const ArSgdParams p) {
  const unsigned sense0 = *reinterpret_cast<volatile unsigned*>(&p.state[1]);
  const unsigned epoch0 = *reinterpret_cast<volatile unsigned*>(&p.state[2]);
  const float lr = p.hyper[0], ema_decay = p.hyper[1], ema_rest = p.hyper[2];
  const long long SL = ((p.flat_elems + p.world - 1) / p.world + 3) / 4 * 4;       // slice length, a multiple of 4 elements
  float* mine = reinterpret_cast<float*>(p.peer_grad[p.rank]);

  ar_barrier(p, sense0 + 1, epoch0 + 1, true);                                        // A: every backward is done

  // ---- phase 1: reduce slice `rank` over all ranks, in rank order
  {
    const long long lo = (long long)p.rank * SL, hi = min(p.flat_elems, lo + SL);
    const float inv = 1.0f / (float)p.world;
    const long long n4 = hi > lo ? (hi - lo) / 4 : 0;
    for (long long i = (long long)blockIdx.x * kArThreads + threadIdx.x; i < n4; i += (long long)gridDim.x * kArThreads) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 v[kArMaxWorld];
#pragma unroll
      for (int q = 0; q < kArMaxWorld; ++q)
        if (q < p.world) v[q] = __ldcg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.peer_grad[q]) + lo) + i);
#pragma unroll
      for (int q = 0; q < kArMaxWorld; ++q)
        if (q < p.world) { acc.x += v[q].x; acc.y += v[q].y; acc.z += v[q].z; acc.w += v[q].w; }
      reinterpret_cast<float4*>(mine + lo)[i] = make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
    }
    if (blockIdx.x == 0) {                                                             // tail of the last slice (< 4 elements)
      for (long long i = lo + n4 * 4 + threadIdx.x; i < hi; i += kArThreads) {
        float acc = 0.f;
        for (int q = 0; q < p.world; ++q) acc += __ldcg(reinterpret_cast<const float*>(p.peer_grad[q]) + i);
        mine[i] = acc * inv;
      }
    }
  }

  ar_barrier(p, sense0 + 2, epoch0 + 2, true);                                        // B: every slice is reduced

  // ---- phase 2: SGD + EMA over every chunk, the reduced gradient read from the rank that owns its slice
  for (int c = blockIdx.x; c < p.n_chunks; c += gridDim.x) {
    const int t = p.chunks[2 * c], e0 = p.chunks[2 * c + 1];
    const long long* row = p.table + (long long)t * 6;
    float* w = reinterpret_cast<float*>(row[0]);
    const float* g = reinterpret_cast<const float*>(row[1]);
    float* buf = reinterpret_cast<float*>(row[2]);
    float* ema = reinterpret_cast<float*>(row[3]);
    const long long n = row[4];
    const float wd = __int_as_float((int)(row[5] & 0xffffffffll));
    const long long e1 = min(n, (long long)e0 + p.chunk_elems);
    const long long goff = g ? (g - mine) : 0;                                       // offset of this tensor in the flat buffer
    // U items per thread in flight: the remote gradient loads take microseconds over NVLink (a one-element-at-a-time loop, the
    // first version, spent 540 us on 36 MB at two ranks). Tensors whose element count and flat offset are multiples of four
    // (all but the 1-element objectness biases: FusedSgdEma pads every slot of the flat buffer to 16 bytes) move as float4.
    constexpr int U = 4;
    const bool vec = (n & 3) == 0 && (e0 & 3) == 0 && (goff & 3) == 0 && ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(buf) |
                      reinterpret_cast<uintptr_t>(ema)) & 15) == 0;
    const bool mom = p.momentum != 0.0f;
    if (vec) {
      const long long q0 = e0 >> 2, q1 = e1 >> 2;
      for (long long base = q0; base < q1; base += (long long)kArThreads * U) {
        float4 gv[U], wv[U], bv[U], ev[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = base + (long long)u * kArThreads + threadIdx.x;
          if (i < q1) {
            wv[u] = reinterpret_cast<const float4*>(w)[i];
            if (g) {
              const long long off = goff + 4 * i;
              const int owner = (int)(off / SL);                    // SL and off are multiples of 4: a vector never straddles slices
              gv[u] = __ldcg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.peer_grad[owner]) + off));
              if (mom && !p.first_step) bv[u] = reinterpret_cast<const float4*>(buf)[i];
            }
            if (ema) ev[u] = reinterpret_cast<const float4*>(ema)[i];
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = base + (long long)u * kArThreads + threadIdx.x;
          if (i < q1) {
            float v[4] = {wv[u].x, wv[u].y, wv[u].z, wv[u].w};
            if (g) {
              const float d4[4] = {gv[u].x, gv[u].y, gv[u].z, gv[u].w};
              const float b4[4] = {bv[u].x, bv[u].y, bv[u].z, bv[u].w};
              float nb[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float d = d4[k];
                if (wd != 0.0f) d = fmaf(wd, v[k], d);
                if (mom) {
                  nb[k] = p.first_step ? d : __fadd_rn(__fmul_rn(p.momentum, b4[k]), d);
                  d = p.nesterov ? fmaf(p.momentum, nb[k], d) : nb[k];
                }
                v[k] = fmaf(-lr, d, v[k]);
              }
              if (mom) reinterpret_cast<float4*>(buf)[i] = make_float4(nb[0], nb[1], nb[2], nb[3]);
              reinterpret_cast<float4*>(w)[i] = make_float4(v[0], v[1], v[2], v[3]);
            }
            if (ema) {
              const float e4[4] = {ev[u].x, ev[u].y, ev[u].z, ev[u].w};
              float r[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) r[k] = __fadd_rn(__fmul_rn(e4[k], ema_decay), __fmul_rn(ema_rest, v[k]));
              reinterpret_cast<float4*>(ema)[i] = make_float4(r[0], r[1], r[2], r[3]);
            }
          }
        }
      }
    } else {
      for (long long base = e0; base < e1; base += (long long)kArThreads * U) {
        float gv[U], wv[U], bv[U], ev[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = base + (long long)u * kArThreads + threadIdx.x;
          if (i < e1) {
            wv[u] = w[i];
            if (g) {
              const long long off = goff + i;
              const int owner = (int)(off / SL);
              gv[u] = __ldcg(reinterpret_cast<const float*>(p.peer_grad[owner]) + off);   // L2 / NVLink, never a stale L1 line of phase 1
              if (mom && !p.first_step) bv[u] = buf[i];
            }
            if (ema) ev[u] = ema[i];
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = base + (long long)u * kArThreads + threadIdx.x;
          if (i < e1) {
            float v = wv[u];
            if (g) {
              float d = gv[u];
              if (wd != 0.0f) d = fmaf(wd, v, d);
              if (mom) {
                const float nb = p.first_step ? d : __fadd_rn(__fmul_rn(p.momentum, bv[u]), d);
                buf[i] = nb;
                d = p.nesterov ? fmaf(p.momentum, nb, d) : nb;
              }
              v = fmaf(-lr, d, v);
              w[i] = v;
            }
            if (ema) ema[i] = __fadd_rn(__fmul_rn(ev[u], ema_decay), __fmul_rn(ema_rest, v));
          }
        }
      }
    }
  }

  if (blockIdx.x == 0 && threadIdx.x == 0) p.state[2] = epoch0 + 3;                    // (read again only by the next launch)
  ar_barrier(p, sense0 + 3, epoch0 + 3, false);                                       // C: every rank is done reading
}

int allreduce_sgd_ema_launch(const long long* table, const int* chunks, int n_chunks, int chunk_elems, float momentum, int nesterov,
                             int first_step, const float* hyper, const long long* peer_grad, const long long* peer_flag,
                             long long flat_elems, int rank, int world, unsigned* state, cudaStream_t s) {
  YX_REQUIRE(table && chunks && hyper && peer_grad && peer_flag && state, YX_ERR_INVALID_ARG, "allreduce_sgd_ema: null pointer");
  YX_REQUIRE(world >= 1 && world <= kArMaxWorld && rank >= 0 && rank < world, YX_ERR_INVALID_ARG, "allreduce_sgd_ema: rank %d of %d", rank, world);
  YX_REQUIRE(n_chunks > 0 && chunk_elems > 0 && flat_elems > 0, YX_ERR_INVALID_ARG, "allreduce_sgd_ema: sizes");
  ArSgdParams p;
  memset(&p, 0, sizeof(p));
  p.table = table; p.chunks = chunks; p.n_chunks = n_chunks; p.chunk_elems = chunk_elems;
  p.momentum = momentum; p.nesterov = nesterov; p.first_step = first_step; p.hyper = hyper;
  for (int q = 0; q < world; ++q) {
    YX_REQUIRE(peer_grad[q] != 0 && peer_flag[q] != 0 && (peer_grad[q] & 15) == 0, YX_ERR_INVALID_ARG, "allreduce_sgd_ema: peer pointer %d", q);
    p.peer_grad[q] = peer_grad[q]; p.peer_flag[q] = peer_flag[q];
  }
  p.flat_elems = flat_elems; p.rank = rank; p.world = world; p.state = state;
  static int cap_dev[kMaxDevices] = {};
  int& cap = cap_dev[current_device_slot()];
  if (cap == 0) {
    int per_sm = 0;
    YX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, allreduce_sgd_ema_kernel, kArThreads, 0));
    YX_REQUIRE(per_sm >= 1, YX_ERR_CUDA, "allreduce_sgd_ema: the kernel does not fit an SM");
    if (per_sm > 4) per_sm = 4;
    cap = per_sm * num_sms();
  }
  // co-resident grid (the barriers need every CTA running): cooperative launch makes the driver check it
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)cap); cfg.blockDim = dim3(kArThreads); cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  YX_CUDA(cudaLaunchKernelEx(&cfg, allreduce_sgd_ema_kernel, p));
  return YX_OK;
}

}  // namespace yx
