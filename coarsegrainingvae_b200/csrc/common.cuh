// Shared helpers for libcgvae_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>
#include <atomic>
#include <algorithm>

#include "../../include/cgvae_b200.h"

namespace cgvae {

constexpr int kNumSM = 148;  // B200: 2 dies x 74 SMs

extern thread_local char g_err[512];
extern std::atomic<unsigned long long> g_launches;

// Device-side index validation.  The raw-pointer kernels cannot raise, so an out-of-range index (atoms of a bead >= F
// at the lifting gather, an embedding id >= table rows, a bead / node index outside its range) is SKIPPED (never read
// or written out of bounds) and recorded as a bit in a caller-owned int32 word registered per device with
// cgvae_set_error_flags(); the host turns it into the IndexError the reference raises (cgvae.py:473, nn.Embedding).
enum { CGVAE_ERR_LIFT_RANK = 1, CGVAE_ERR_EMBED_INDEX = 2, CGVAE_ERR_BEAD_INDEX = 4, CGVAE_ERR_NODE_INDEX = 8 };
constexpr int kMaxDevices = 64;
extern std::atomic<int32_t*> g_err_flags[kMaxDevices];
inline int32_t* err_flags() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) return nullptr;
  return g_err_flags[d].load(std::memory_order_relaxed);
}
__device__ __forceinline__ void raise_flag(int32_t* flags, int bit) {
  if (flags != nullptr) atomicOr(flags, bit);
}

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// call after every kernel launch: counts the launch and converts launch errors to a return code
inline int launched(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

#define CGVAE_REQUIRE(cond, ...)                      \
  do {                                                \
    if (!(cond)) return ::cgvae::fail(-1, __VA_ARGS__); \
  } while (0)

#define CGVAE_CUDA(expr)                                                               \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) return ::cgvae::fail((int)_e, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------
// A training step is ~450 dependent kernels of a few microseconds each: the launch latency between dependent nodes,
// not the work, dominates.  Every kernel of this library starts with pdl_wait() (griddepcontrol.wait: blocks until the
// preceding grid has completed and flushed its writes -- all global-memory accesses come after it, so ordering is exactly
// that of a plain stream) and pdl_trigger() (griddepcontrol.launch_dependents: lets the NEXT kernel's launch and prologue
// overlap with this kernel's execution).  Launches carry cudaLaunchAttributeProgrammaticStreamSerialization while
// pdl_enabled() (on by default; CGVAE_PDL=0 or cgvae_set_pdl(0) turn it off, see graph.cu).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#define CGVAE_KERNEL_PROLOGUE() \
  do {                          \
    ::cgvae::pdl_wait();        \
    ::cgvae::pdl_trigger();     \
  } while (0)

bool pdl_enabled();
// 0: the tensor-core GEMMs and the message filter run 3xTF32 (fp32 parity); 1: 1xTF32 (graph.cu, cgvae_set_matmul_precision)
int matmul_precision();
// inside a parameter range registered with cgvae_register_const_range, and PDL on (gemm_stream.cu)
bool weights_are_constant(const void* p, size_t bytes);

// cluster == nullptr: no cluster attribute.  The PDL attribute is attached while pdl_enabled().
template <typename... KArgs, typename... Args>
inline void launch_with_attrs(void (*kernel)(KArgs...), dim3 grid, dim3 block, const dim3* cluster, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster != nullptr) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster->x;
    attr[n].val.clusterDim.y = cluster->y;
    attr[n].val.clusterDim.z = cluster->z;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface through launched()
}

template <typename... KArgs, typename... Args>
inline void launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  launch_with_attrs(kernel, grid, block, nullptr, smem, st, args...);
}

// thread-block cluster of shape `cluster` (every grid extent a multiple of it); a cluster of one CTA is still a cluster
// launch: the kernels that call cooperative_groups::this_cluster() need the attribute whatever its size
template <typename... KArgs, typename... Args>
inline void launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, dim3 cluster, size_t smem, cudaStream_t st,
                           Args... args) {
  launch_with_attrs(kernel, grid, block, &cluster, smem, st, args...);
}

// Zero fill as a KERNEL.  Inside a captured CUDA graph a memset node costs 3..11 us of idle time before the next kernel
// node starts (CUPTI timeline of the chignolin step: every Memset -> kernel edge), a kernel -> kernel edge 0.06 us.
static __global__ void __launch_bounds__(256) zero_words_kernel(uint32_t* __restrict__ p, size_t n_words) {
  CGVAE_KERNEL_PROLOGUE();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x) p[i] = 0u;
}
// bytes must be a multiple of 4 and p 4-byte aligned (every caller zeroes int32 / float arrays)
inline int zero_fill(void* p, size_t bytes, cudaStream_t st) {
  const size_t n_words = bytes / 4;
  if (n_words == 0) return 0;
  const unsigned blocks = (unsigned)std::min<size_t>((n_words + 255) / 256, (size_t)kNumSM * 8);
  launch_kernel(zero_words_kernel, dim3(blocks), dim3(256), 0, st, reinterpret_cast<uint32_t*>(p), n_words);
  return launched("zero_fill");
}
#define CGVAE_ZERO(ptr, bytes, st)                               \
  do {                                                           \
    if (int _rc = ::cgvae::zero_fill((ptr), (bytes), (st))) return _rc; \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// receiver of CSR slot `slot`: the largest row with rowptr[row] <= slot
__device__ __forceinline__ int row_of_slot(const int32_t* __restrict__ rowptr, int64_t n_rows, int slot) {
  int64_t lo = 0, hi = n_rows;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (rowptr[mid] <= slot) lo = mid; else hi = mid;
  }
  return (int)lo;
}

// message filter column for (split k, channel f): rows r < R from Wf[(k*F+f)][r], row R = bias, rest zero
__device__ __forceinline__ float filter_entry(const float* __restrict__ Wf, const float* __restrict__ bf, int F, int R,
                                              int k, int f, int r) {
  if (r < R) return Wf[((int64_t)k * F + f) * R + r];
  if (r == R) return bf[(int64_t)k * F + f];
  return 0.f;
}

__device__ __forceinline__ float swish_f(float z) { return z / (1.0f + expf(-z)); }
// d/dz [z * sigmoid(z)] = sig * (1 + z * (1 - sig))
__device__ __forceinline__ float dswish_f(float z) {
  float sig = 1.0f / (1.0f + expf(-z));
  return sig * (1.0f + z * (1.0f - sig));
}

__device__ __forceinline__ float sigmoid_f(float z) { return 1.0f / (1.0f + expf(-z)); }

__device__ __forceinline__ float act_fwd(int act, float z) {
  switch (act) {
    case CGVAE_ACT_SWISH: return swish_f(z);
    case CGVAE_ACT_RELU: return z > 0.f ? z : 0.f;
    case CGVAE_ACT_TANH: return tanhf(z);
    case CGVAE_ACT_SIGMOID: return sigmoid_f(z);
    // F.softplus(z) - ln 2 (modules.py:8-14); torch switches to the identity above its threshold of 20
    case CGVAE_ACT_SHIFTED_SOFTPLUS: return (z > 20.f ? z : log1pf(expf(z))) - 0.6931471805599453f;
    case CGVAE_ACT_LEAKY_RELU: return z > 0.f ? z : 0.01f * z;            // nn.LeakyReLU default slope
    case CGVAE_ACT_ELU: return z > 0.f ? z : expm1f(z);                   // nn.ELU default alpha = 1
    default: return z;
  }
}
__device__ __forceinline__ float act_bwd(int act, float z) {
  switch (act) {
    case CGVAE_ACT_SWISH: return dswish_f(z);
    case CGVAE_ACT_RELU: return z > 0.f ? 1.f : 0.f;
    case CGVAE_ACT_TANH: { float t = tanhf(z); return 1.f - t * t; }
    case CGVAE_ACT_SIGMOID: { float sg = sigmoid_f(z); return sg * (1.f - sg); }
    case CGVAE_ACT_SHIFTED_SOFTPLUS: return z > 20.f ? 1.f : sigmoid_f(z);
    case CGVAE_ACT_LEAKY_RELU: return z > 0.f ? 1.f : 0.01f;
    case CGVAE_ACT_ELU: return z > 0.f ? 1.f : expf(z);
    default: return 1.f;
  }
}

}  // namespace cgvae
