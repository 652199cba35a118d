// Shared device/host helpers for the sm_100a YOLOX kernels: error plumbing, TMA maps, tcgen05 descriptor
// formats and launches, PTX wrappers for mbarrier / TMA / tcgen05 / TMEM, and small numeric helpers.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

#include "../../include/yx_b200.h"

namespace yx {

// Function attributes (opt-in shared memory) belong to a device: launch helpers cache "already configured" per device,
// so one process may drive several GPUs (each with its own module / engine).
static constexpr int kMaxDevices = 64;
inline int current_device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}

// ------------------------------------------------------------------------------------------
// host-side error plumbing (thread-local message, never throws)
// ------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define YX_CUDA(call)                                                         \
  do {                                                                        \
    cudaError_t _e = (call);                                                  \
    if (_e != cudaSuccess) return ::yx::cuda_fail(_e, #call, __FILE__, __LINE__); \
  } while (0)

#define YX_REQUIRE(cond, code, ...)  \
  do {                               \
    if (!(cond)) {                   \
      ::yx::set_error(__VA_ARGS__);  \
      return (code);                 \
    }                                \
  } while (0)

int num_sms();  // SM count of the current device (cached)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int dtype_size(int dt) { return dt == YX_FP32 ? 4 : (dt == YX_U8 ? 1 : 2); }

// ------------------------------------------------------------------------------------------
// host side: tcgen05 operand formats and TMA tensor maps
// ------------------------------------------------------------------------------------------
int max_smem_optin();  // opt-in shared memory per block of the current device (cached; 0 if it cannot be queried)

// Encodes a tiled TMA map (no interleave, zero fill out of bounds); elem_strides == nullptr means all 1. Returns YX_OK,
// YX_ERR_NO_DEVICE without a driver entry point, or YX_ERR_CUDA with an error message naming `what` and the shape.
int encode_tma(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
               const cuuint64_t* byte_strides, const cuuint32_t* box, const cuuint32_t* elem_strides,
               CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what);

inline CUtensorMapDataType tma_dtype(int dt) {
  switch (dt) {
    case YX_BF16: return CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    case YX_FP16: return CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    case YX_FP32: return CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    default: return CU_TENSOR_MAP_DATA_TYPE_UINT8;
  }
}

// Operand rows of 32, 64 or 128 bytes (16, 32 or 64 16-bit channels) are stored with the swizzle of the same span: TMA writes
// that layout with tma_swizzle(row_bytes) and the UMMA descriptor names it by layout type 6, 4 or 2.
inline CUtensorMapSwizzle tma_swizzle(unsigned row_bytes) {
  return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}
// Upper word of the UMMA shared-memory descriptor: stride byte offset = one 8-row atom (>> 4), version 1, layout type
inline unsigned umma_desc_hi(unsigned row_bytes) {
  const unsigned layout = row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
  return (((8u * row_bytes) >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29);
}
// UMMA instruction descriptor of a kind::f16 MMA, M = 128, N = n: fp32 accumulate, A and B in `dtype` (bf16 or fp16),
// both K-major, or both MN-major (bits 15, 16)
inline unsigned umma_idesc(int dtype, int n, bool mn_major = false) {
  const unsigned fmt = dtype == YX_BF16 ? 1u : 0u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (mn_major ? (1u << 15) | (1u << 16) : 0u) | ((unsigned)(n >> 3) << 17) |
         ((128u >> 4) << 24);
}

#ifdef __CUDACC__
// Plain launch that returns the launch error. The training step's chains of small kernels (BatchNorm, wgrad, packing) do
// not use programmatic dependent launch: it measured slower than plain launches there (9.32 vs 8.70 ms per step, 8 images).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// launch_kernel with programmatic dependent launch: the kernel's prologue may overlap the tail of its predecessor in the
// stream; the kernel waits for the predecessor's writes with pdl_wait().
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchAttribute pdl = {};
  pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  pdl.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cfg.attrs = &pdl; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// Raises the dynamic shared-memory limit of every kernel in `kernels` (one kernel pointer or an array of them of any rank)
// to smem_bytes(i) for the i-th in row-major order. Kernel attributes belong to a device: this happens on the first call on
// each device, `done` holding the table's per-device flags. Later calls make no CUDA runtime call besides the device lookup,
// so launches inside a CUDA-graph capture may make them; smem_bytes is evaluated on the first call only.
template <typename Table, typename Bytes>
inline cudaError_t opt_in_smem(bool (&done)[kMaxDevices], const Table& kernels, Bytes smem_bytes) {
  bool& d = done[current_device_slot()];
  if (d) return cudaSuccess;
  using Kernel = typename std::remove_all_extents<Table>::type;
  const Kernel* k = reinterpret_cast<const Kernel*>(&kernels);
  for (int i = 0; i < (int)(sizeof(Table) / sizeof(Kernel)); ++i) {
    const cudaError_t e = cudaFuncSetAttribute(k[i], cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(i));
    if (e != cudaSuccess) return e;
  }
  d = true;
  return cudaSuccess;
}

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      // suspend-time hint (ns): the thread sleeps in hardware until the phase completes instead of
      // re-issuing the poll every ~100 cycles (8+ waiting warps per SM otherwise eat a third of the issue slots)
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
      : "memory");
  return ok != 0;
}
// float -> uint32 whose unsigned order is the float order (sort keys of the score filter)
__device__ __forceinline__ uint32_t orderable_f32(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// Bounded spin: a pipeline bug must surface as a trapped launch, never as a hung GPU.
// cold path, kept out of line so the waiting loops stay a handful of instructions
static __device__ __noinline__ void mbar_timed_out(uint32_t bar_smem, uint32_t parity) {
  printf("yx_b200: mbarrier wait timed out (block %d thread %d barrier smem 0x%x parity %u)\n", (int)blockIdx.x,
         (int)threadIdx.x, bar_smem, parity);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 18)) mbar_timed_out(smem_u32(bar), parity);
  }
}

// ---- TMA (cp.async.bulk.tensor) ----
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const void* desc, uint64_t* bar, void* dst, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(const void* desc, uint64_t* bar, void* dst, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      :
      : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---- tcgen05 / TMEM ----
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; 128xNx16 (kind::f16: bf16/fp16 in, fp32 accumulate)
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp gets row (lane base + i)
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}

// ---- programmatic dependent launch (PDL) ----
// launch_dependents: the next kernel in the stream may start being scheduled (its prologue overlaps our
// tail); wait: block until the previous kernel has completed and its writes are visible.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- numerics ----
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }
__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case YX_ACT_SILU: return silu_f(x);
    case YX_ACT_RELU: return fmaxf(x, 0.0f);
    case YX_ACT_LRELU: return x > 0.0f ? x : 0.1f * x;
    default: return x;
  }
}

template <typename T> struct Cvt;
template <> struct Cvt<__nv_bfloat16> {
  static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Cvt<__half> {
  static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};
template <> struct Cvt<float> {
  static __device__ __forceinline__ float to_f(float v) { return v; }
  static __device__ __forceinline__ float from_f(float v) { return v; }
};

// pack two fp32 into one 32-bit word of 16-bit floats (lo = a, hi = b)
__device__ __forceinline__ uint32_t pack16(float a, float b, bool fp16) {
  if (fp16) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void unpack16(uint32_t w, bool fp16, float& a, float& b) {
  if (fp16) {
    float2 f = __half22float2(*reinterpret_cast<__half2*>(&w));
    a = f.x; b = f.y;
  } else {
    float2 f = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&w));
    a = f.x; b = f.y;
  }
}
#endif  // __CUDACC__

}  // namespace yx
