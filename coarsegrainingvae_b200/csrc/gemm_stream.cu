// Weight-streaming contractions for small node sets (decoder graphs of the molecule configs: 12 beads, 36 vector rows).
//
// With M <= 48 rows a Dense layer is M simultaneous matrix-vector products: the cost is reading the weight matrix
// ONCE from HBM (1.4 .. 13 MB at F = 600), the flops are noise.  The tiled kernels of gemm.cu spend their time in
// register -> shared staging and short dependent chains (9 .. 18 us per launch = 0.15 .. 0.7 TB/s; a first version of
// this file that kept the weights in registers was no better: too few bytes in flight per SM, two waves of CTAs).
// Here the TMA engine moves each CTA's whole share of the weight matrix into shared memory with a handful of bulk
// copies issued by ONE thread at kernel start: every byte of the matrix is in flight at once, one wave of CTAs, one
// mbarrier wait, then the math runs out of shared memory:
//
//  NT  Y[M,N] = X[M,K] W[N,K]^T   each CTA owns a contiguous slab of ~N/148 weight rows (cp.async.bulk, 1-D); a warp
//      takes RW rows, lanes run along K; the M x RW accumulators per lane are reduced with a transposing butterfly
//      (n/2 shuffles per halving step instead of 5 per value).
//  NN  C[M,N] = G[M,K] W[K,N]     each CTA owns a [rows x 64|128 columns] panel (cp.async.bulk.tensor 2-D boxes through a
//      tensor map encoded per launch), the contraction (weight rows) is split over the warps and over a thread-block
//      cluster (1,1,S<=8); G^T staged in smem (broadcast LDS.128); warp partials reduced in smem, CTA partials through
//      distributed shared memory in rank order.
//
// Both are deterministic (fixed reduction trees) and carry the epilogue of cgvae_gemm.
#include "common.cuh"
#include <cooperative_groups.h>
#include <cuda.h>
#include <algorithm>
#include <vector>

namespace cgvae {

struct StreamEpilogue {
  const float* bias;
  int act;
  float* z_out;
  const float* z_in;
  int dact;
  const float* add;
  // NT only: output columns n >= n_split go to a second matrix C2[m][n - n_split] (row stride ldc2): two Dense layers
  // that share their input and whose weights are adjacent in memory run as ONE launch (u_mat / v_mat of UpdateBlock)
  float* C2;
  int n_split;
  int64_t ldc2;
};

__device__ __forceinline__ float stream_epilogue(const StreamEpilogue& ep, float v, int64_t m, int64_t n, int64_t ldc) {
  if (ep.bias) v += ep.bias[n];
  if (ep.z_out) ep.z_out[m * ldc + n] = v;
  v = act_fwd(ep.act, v);
  if (ep.z_in) v *= act_bwd(ep.dact, ep.z_in[m * ldc + n]);
  if (ep.add) v += ep.add[m * ldc + n];
  return v;
}

// ---- transposing warp reduction ---------------------------------------------------------------------------------
// Every lane holds N partial values; afterwards the warp-wide sums are spread over the lanes: lane l holds
// wtr_count(N) sums whose original indices are base .. base + count - 1; lanes with (l & wtr_dupmask(N)) != 0 hold
// duplicates.  While the count is even a step sends one half and keeps the other (N/2 shuffles); an odd remainder is
// finished with plain xor-shuffles.
__host__ __device__ constexpr int wtr_count(int n, int off) { return (off >= 1 && n % 2 == 0) ? wtr_count(n / 2, off / 2) : n; }
__host__ __device__ constexpr int wtr_dupmask(int n, int off) { return (off >= 1 && n % 2 == 0) ? wtr_dupmask(n / 2, off / 2) : (off >= 1 ? 2 * off - 1 : 0); }

template <int N, int OFF>
__device__ __forceinline__ void wtr_step(float* v, int lane, int& base) {
  if constexpr (OFF >= 1 && (N % 2 == 0)) {
    constexpr int H = N / 2;
    const bool up = (lane & OFF) != 0;
#pragma unroll
    for (int i = 0; i < H; ++i) {
      const float send = up ? v[i] : v[i + H];
      const float keep = up ? v[i + H] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
    }
    if (up) base += H;
    wtr_step<H, OFF / 2>(v, lane, base);
  } else if constexpr (OFF >= 1) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
      for (int o = OFF; o >= 1; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
    }
  }
}

// ---- mbarrier / TMA primitives -----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sm_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sm_u32(bar)), "r"(count));
}
__device__ __forceinline__ void bar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sm_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t* bar, uint32_t parity) {
  // bounded: a copy that never lands (bad descriptor) traps instead of hanging the GPU
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(sm_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
  }
  asm volatile("trap;");
}
// one elected lane of a converged warp: bulk copies issued under a divergent `if (tid == 0)` are each wrapped by ptxas in an
// ELECT / R2UR / BRA.U.ANY serialisation loop (~200 cycles per copy, measured for tcgen05.mma with tools/tc_latency.cu)
__device__ __forceinline__ bool elect_lane() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// 1-D bulk copy global -> shared (UBLKCP): 16-byte aligned addresses, size a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sm_u32(dst)),
               "l"(src), "r"(bytes), "r"(sm_u32(bar))
               : "memory");
}
// 2-D tiled copy through a tensor map (UTMALDG): coordinates (c0 = innermost element index, c1 = row)
__device__ __forceinline__ void tma_2d_g2s(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   sm_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(sm_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------------------------------
// NT: Y[m][n] = sum_k X[m][k] W[n][k]
// ------------------------------------------------------------------------------------------------------------------
constexpr uint32_t kBulkPiece = 32768;   // bytes per bulk copy of a contiguous range

template <int MR, int RW>
__global__ void __launch_bounds__(MR > 16 ? 256 : 512) gemm_nt_stream_kernel(
    const float* __restrict__ X, int64_t ldx, const float* __restrict__ W, int64_t ldw, float* __restrict__ C, int64_t ldc,
    int M, int N, int K, int rows_per_cta, StreamEpilogue ep, int w_const) {
  // w_const: the weight matrix is not written by any kernel still in flight (a registered parameter range): its bulk copies
  // are issued BEFORE griddepcontrol.wait, i.e. while the preceding kernel is still running (programmatic dependent launch)
  if (!w_const) CGVAE_KERNEL_PROLOGUE();
  extern __shared__ __align__(128) float smem[];
  constexpr int NV = RW * MR;
  float* Xs = smem;                                   // [MR][K]
  float* Ws = smem + (size_t)MR * K;                  // [rows_per_cta][K]
  uint64_t* bar = reinterpret_cast<uint64_t*>(Ws + (size_t)rows_per_cta * K);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int row0 = blockIdx.x * rows_per_cta;
  const int rows = min(rows_per_cta, N - row0);       // >= 1 by construction of the grid

  if (tid == 0) {
    bar_init(bar, 1);
    bar_fence_init();
  }
  // rows of X beyond M read as zero (plain stores: a region the bulk copies never touch)
  for (int idx = tid; idx < (MR - M) * (K / 4); idx += blockDim.x)
    reinterpret_cast<float4*>(Xs + (size_t)M * K)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  if (warp == 0 && elect_lane()) {
    const uint32_t row_bytes = (uint32_t)K * 4u;
    bar_expect_tx(bar, (uint32_t)(M + rows) * row_bytes);
    if (ldw == K) {
      const char* src = reinterpret_cast<const char*>(W + (int64_t)row0 * ldw);
      char* dst = reinterpret_cast<char*>(Ws);
      for (uint32_t off = 0, total = (uint32_t)rows * row_bytes; off < total; off += kBulkPiece)
        bulk_g2s(dst + off, src + off, min(kBulkPiece, total - off), bar);
    } else {
      for (int r = 0; r < rows; ++r) bulk_g2s(Ws + (size_t)r * K, W + (int64_t)(row0 + r) * ldw, row_bytes, bar);
    }
    if (w_const) pdl_wait();              // the activations ARE produced by the preceding kernel
    if (ldx == K) {
      const char* src = reinterpret_cast<const char*>(X);
      char* dst = reinterpret_cast<char*>(Xs);
      for (uint32_t off = 0, total = (uint32_t)M * row_bytes; off < total; off += kBulkPiece)
        bulk_g2s(dst + off, src + off, min(kBulkPiece, total - off), bar);
    } else {
      for (int m = 0; m < M; ++m) bulk_g2s(Xs + (size_t)m * K, X + (int64_t)m * ldx, row_bytes, bar);
    }
  }
  if (w_const) CGVAE_KERNEL_PROLOGUE();     // every thread: the epilogue operands / the output belong to the dependency chain
  bar_wait(bar, 0);

  const int nchunks = (K + 127) / 128;
  for (int t0 = warp * RW; t0 < rows; t0 += nwarps * RW) {
    float acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.f;
    for (int c = 0; c < nchunks; ++c) {
      const int k = c * 128 + lane * 4;
      if (k < K) {                                     // K % 4 == 0: the float4 is inside the row
        float4 w[RW];
#pragma unroll
        for (int r = 0; r < RW; ++r)
          w[r] = (t0 + r < rows) ? *reinterpret_cast<const float4*>(Ws + (size_t)(t0 + r) * K + k) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int m = 0; m < MR; ++m) {
          const float4 xv = *reinterpret_cast<const float4*>(Xs + (size_t)m * K + k);
#pragma unroll
          for (int r = 0; r < RW; ++r) {
            float a = acc[r * MR + m];
            a = fmaf(w[r].x, xv.x, a);
            a = fmaf(w[r].y, xv.y, a);
            a = fmaf(w[r].z, xv.z, a);
            a = fmaf(w[r].w, xv.w, a);
            acc[r * MR + m] = a;
          }
        }
      }
    }
    int base = 0;
    wtr_step<NV, 16>(acc, lane, base);
    constexpr int CNT = wtr_count(NV, 16);
    constexpr int DUP = wtr_dupmask(NV, 16);
    if ((lane & DUP) == 0) {
#pragma unroll
      for (int i = 0; i < CNT; ++i) {
        const int idx = base + i;
        const int r = idx / MR, m = idx % MR;
        const int n = row0 + t0 + r;
        if (m < M && t0 + r < rows) {
          if (ep.C2 != nullptr && n >= ep.n_split) ep.C2[(int64_t)m * ep.ldc2 + (n - ep.n_split)] = acc[i];
          else C[(int64_t)m * ldc + n] = stream_epilogue(ep, acc[i], m, n, ldc);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// NN: C[m][n] = sum_k G[m][k] W[k][n]      (k = weight rows: the contraction; n = weight columns: the outputs)
// ------------------------------------------------------------------------------------------------------------------
constexpr int NN_MAXBOX = 8;

template <int VEC> struct VecT;
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int MR, int VEC, int NW>
__global__ void __launch_bounds__(NW * 32) gemm_nn_stream_kernel(
    const __grid_constant__ CUtensorMap wmap, const float* __restrict__ G, int64_t ldg, float* __restrict__ C, int64_t ldc,
    int M, int N, int K, int k_per_cta, int box_rows, StreamEpilogue ep, int w_const) {
  if (!w_const) CGVAE_KERNEL_PROLOGUE();     // w_const: see gemm_nt_stream_kernel
  namespace cg = cooperative_groups;
  using vec_t = typename VecT<VEC>::type;
  constexpr int COLS = 32 * VEC;         // output columns per CTA = inner box extent
  extern __shared__ __align__(128) float smem[];
  const int nbox = (k_per_cta + box_rows - 1) / box_rows;
  float* Wt = smem;                                          // [nbox * box_rows][COLS]   TMA destination
  float* red = smem;                                         // [NW][MR][COLS]            (after the main loop; aliases Wt)
  const size_t wt_floats = (size_t)max(nbox * box_rows, NW * MR) * COLS;
  float* part = smem + wt_floats;                            // [MR][COLS] CTA partial (read by the cluster)
  float* Gt = part + MR * COLS;                              // [k_per_cta][MR]
  uint64_t* bars = reinterpret_cast<uint64_t*>(Gt + (size_t)k_per_cta * MR);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int col0 = blockIdx.x * COLS;
  const int kbeg = blockIdx.z * k_per_cta;
  const int cnt = max(0, min(K, kbeg + k_per_cta) - kbeg);

  if (tid == 0) {
    for (int b = 0; b < nbox; ++b) bar_init(bars + b, 1);
    bar_fence_init();
  }
  __syncwarp();
  if (warp == 0 && elect_lane()) {
    // rows beyond K (and columns beyond N) are zero-filled by the TMA unit; the byte count is that of the full box
    for (int b = 0; b < nbox; ++b) {
      if (b * box_rows < cnt) {
        bar_expect_tx(bars + b, (uint32_t)box_rows * COLS * 4u);
        tma_2d_g2s(Wt + (size_t)b * box_rows * COLS, &wmap, col0, kbeg + b * box_rows, bars + b);
      }
    }
  }
  if (w_const) CGVAE_KERNEL_PROLOGUE();
  // G^T for this CTA's slice of the contraction (plain loads; overlaps with the weight panel in flight)
  for (int idx = tid; idx < MR * cnt; idx += NW * 32) {
    const int m = idx / cnt, j = idx - m * cnt;
    Gt[j * MR + m] = (m < M) ? __ldg(G + (int64_t)m * ldg + kbeg + j) : 0.f;
  }
  __syncthreads();          // Gt complete, barrier initialisation visible to every waiter

  float acc[MR][VEC];
#pragma unroll
  for (int m = 0; m < MR; ++m)
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[m][v] = 0.f;

  for (int b = 0; b * box_rows < cnt; ++b) {
    bar_wait(bars + b, 0);
    const int jend = min(cnt, (b + 1) * box_rows);
#pragma unroll 2
    for (int j = b * box_rows + warp; j < jend; j += NW) {
      const vec_t t = *reinterpret_cast<const vec_t*>(Wt + (size_t)j * COLS + lane * VEC);
      float w[VEC];
      if constexpr (VEC == 2) { w[0] = t.x; w[1] = t.y; }
      if constexpr (VEC == 4) { w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w; }
      const float* g = Gt + j * MR;
#pragma unroll
      for (int m4 = 0; m4 < MR / 4; ++m4) {
        const float4 g4 = *reinterpret_cast<const float4*>(g + 4 * m4);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          acc[4 * m4 + 0][v] = fmaf(g4.x, w[v], acc[4 * m4 + 0][v]);
          acc[4 * m4 + 1][v] = fmaf(g4.y, w[v], acc[4 * m4 + 1][v]);
          acc[4 * m4 + 2][v] = fmaf(g4.z, w[v], acc[4 * m4 + 2][v]);
          acc[4 * m4 + 3][v] = fmaf(g4.w, w[v], acc[4 * m4 + 3][v]);
        }
      }
    }
  }
  __syncthreads();                         // the weight panel is dead: its storage becomes the warp-partial buffer
#pragma unroll
  for (int m = 0; m < MR; ++m)
#pragma unroll
    for (int v = 0; v < VEC; ++v) red[(warp * MR + m) * COLS + lane * VEC + v] = acc[m][v];
  __syncthreads();
  for (int o = tid; o < MR * COLS; o += NW * 32) {
    float s = 0.f;
#pragma unroll
    for (int wv = 0; wv < NW; ++wv) s += red[wv * MR * COLS + o];   // warp order: deterministic
    part[o] = s;
  }
  cg::cluster_group cluster = cg::this_cluster();
  cluster.sync();
  const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  // rank r finishes rows r, r + S, ...: sum of the S CTA partials in rank order, epilogue, store
  for (int o = tid; o < MR * COLS; o += NW * 32) {
    const int m = o / COLS, c = o - m * COLS;
    if (m % S != rank) continue;
    const int n = col0 + c;
    if (m < M && n < N) {
      float s = 0.f;
      for (int z = 0; z < S; ++z) s += *cluster.map_shared_rank(part + o, z);
      C[(int64_t)m * ldc + n] = stream_epilogue(ep, s, m, n, ldc);
    }
  }
  cluster.sync();
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      (void)cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

constexpr size_t kMaxStreamSmem = 220 * 1024;

// Parameter ranges registered by the host (cgvae_register_const_range: the flat parameter buffer of a training step): memory
// that no kernel writes between two optimiser steps.  A weight matrix inside such a range may be fetched before the
// dependency wait of a programmatic dependent launch -- its bulk copies then overlap with the tail of the preceding kernel
// instead of starting after it.  The optimiser is the only writer; every kernel between it and the first weight-streaming
// launch of the next step runs its own griddepcontrol.wait before triggering its dependents, so the chain of completed
// grids always includes the optimiser.
struct ConstRange {
  uintptr_t begin, end;
};
static std::vector<ConstRange> g_const_ranges;     // sorted by begin, disjoint (host-side, launch thread only)

bool weights_are_constant(const void* p, size_t bytes) {
  if (!pdl_enabled() || g_const_ranges.empty()) return false;
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  auto it = std::upper_bound(g_const_ranges.begin(), g_const_ranges.end(), a,
                             [](uintptr_t v, const ConstRange& r) { return v < r.begin; });
  if (it == g_const_ranges.begin()) return false;
  --it;
  return a >= it->begin && a + bytes <= it->end;
}

template <int MR, int RW>
static bool launch_nt(const float* X, int64_t ldx, const float* W, int64_t ldw, float* C, int64_t ldc, int M, int N, int K,
                      const StreamEpilogue& ep, cudaStream_t st) {
  const int w_const = weights_are_constant(W, sizeof(float) * ((size_t)(N - 1) * (size_t)ldw + (size_t)K)) ? 1 : 0;
  int rpc = (int)ceil_div(ceil_div(N, kNumSM), RW) * RW;       // one CTA per SM, whole tasks
  const size_t smem = sizeof(float) * ((size_t)MR * K + (size_t)rpc * K) + 16;
  if (smem > kMaxStreamSmem) return false;
  static size_t attr_bytes = 0;
  if (smem > attr_bytes) {
    if (cudaFuncSetAttribute(gemm_nt_stream_kernel<MR, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxStreamSmem) != cudaSuccess) {
      (void)cudaGetLastError();
      return false;
    }
    attr_bytes = kMaxStreamSmem;
  }
  const int tasks = rpc / RW;
  const int nwarps = tasks <= 2 ? 2 : (tasks <= 4 ? 4 : ((tasks <= 8 || MR > 16) ? 8 : 16));
  launch_kernel(gemm_nt_stream_kernel<MR, RW>, dim3((unsigned)ceil_div(N, rpc)), dim3(nwarps * 32), smem, st, X, ldx, W, ldw, C, ldc, M,
                N, K, rpc, ep, w_const);
  return true;
}

template <int MR, int VEC, int NW>
static bool launch_nn(const float* G, int64_t ldg, const float* W, int64_t ldw, float* C, int64_t ldc, int M, int N, int K,
                      const StreamEpilogue& ep, cudaStream_t st) {
  const int w_const = weights_are_constant(W, sizeof(float) * ((size_t)(K - 1) * (size_t)ldw + (size_t)N)) ? 1 : 0;
  constexpr int COLS = 32 * VEC;
  EncodeTiledFn encode = encode_tiled_fn();
  if (encode == nullptr) return false;
  const int blocks = (int)ceil_div(N, COLS);
  int S = (int)std::min<int64_t>(8, std::max<int64_t>(1, kNumSM / blocks));          // one wave of CTAs
  S = (int)std::min<int64_t>(S, std::max<int64_t>(1, K / NW));
  while (S & (S - 1)) S &= S - 1;                                                    // cluster sizes 1, 2, 4, 8
  int k_per_cta = (int)ceil_div(K, S);
  S = (int)ceil_div(K, k_per_cta);
  const int nbox = (int)ceil_div(k_per_cta, 256);
  if (nbox > NN_MAXBOX) return false;
  const int box_rows = (int)ceil_div(k_per_cta, nbox);
  const size_t wt_floats = (size_t)std::max(nbox * box_rows, NW * MR) * COLS;
  const size_t smem = sizeof(float) * (wt_floats + (size_t)MR * COLS + (size_t)k_per_cta * MR) + 8 * NN_MAXBOX;
  if (smem > kMaxStreamSmem) return false;
  CUtensorMap map;
  const cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)K};
  const cuuint64_t gstride[1] = {(cuuint64_t)ldw * 4};
  const cuuint32_t box[2] = {(cuuint32_t)COLS, (cuuint32_t)box_rows};
  const cuuint32_t estride[2] = {1, 1};
  if (encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(W), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  static size_t attr_bytes = 0;
  if (smem > attr_bytes) {
    if (cudaFuncSetAttribute(gemm_nn_stream_kernel<MR, VEC, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxStreamSmem) != cudaSuccess) {
      (void)cudaGetLastError();
      return false;
    }
    attr_bytes = kMaxStreamSmem;
  }
  launch_cluster(gemm_nn_stream_kernel<MR, VEC, NW>, dim3((unsigned)blocks, 1, (unsigned)S), dim3(NW * 32), dim3(1, 1, (unsigned)S), smem,
                 st, map, G, ldg, C, ldc, M, N, K, k_per_cta, box_rows, ep, w_const);
  return true;
}

// returns 1 when the problem was launched here, 0 when the caller should use the tiled kernels
int launch_gemm_stream(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                       int64_t N, int64_t K, const float* bias, int act, float* z_out, const float* z_in, int dact,
                       const float* add, cudaStream_t st) {
  if (M > 48 || M < 1 || form == CGVAE_GEMM_TN) return 0;
  if (N * K < 64 * 64 || N >= (1 << 24) || K >= (1 << 24)) return 0;
  const StreamEpilogue ep{bias, act, z_out, z_in, dact, add, nullptr, 0, 0};
  const int m = (int)M, n = (int)N, k = (int)K;
  if (form == CGVAE_GEMM_NT) {
    // rows of X and W travel as bulk copies: 16-byte aligned rows of a multiple of 16 bytes
    if (K % 4 != 0 || K < 128 || lda % 4 != 0 || ldb % 4 != 0 || !aligned16(A) || !aligned16(B)) return 0;
    if (M <= 12) return launch_nt<12, 4>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
    if (M <= 16) return launch_nt<16, 4>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
    if (M <= 36) return launch_nt<36, 2>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
    return launch_nt<48, 2>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
  }
  // NN: C[M,N] = A[M,K] B[K,N]; lanes run along N; the weight panel travels through a tensor map (16-byte row pitch)
  if (K < 64 || N < 64 || ldb % 4 != 0 || !aligned16(B)) return 0;
  const bool wide = ceil_div(N, 64) * 2 > kNumSM;       // many columns: 128-column panels keep the grid within one wave
  if (M <= 12) return wide ? launch_nn<12, 4, 16>(A, lda, B, ldb, C, ldc, m, n, k, ep, st) : launch_nn<12, 2, 16>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
  if (M <= 16) return wide ? launch_nn<16, 4, 16>(A, lda, B, ldb, C, ldc, m, n, k, ep, st) : launch_nn<16, 2, 16>(A, lda, B, ldb, C, ldc, m, n, k, ep, st);
  // 17..48 rows: measured on B200 (tools/bench_skinny.py, M = 36), 36- and 48-row panels were slower than the cluster
  // split-K tiles of gemm.cu (9.0 vs 8.0 us at 600x600, 12.4 vs 10.6 us at 600x1200): the G^T broadcasts dominate the math
  return 0;
}

// two Dense layers on the same input, weights adjacent in memory: W = [W1 (N1 rows); W2 (N2 rows)], no bias / activation
int launch_dense_pair_stream(const float* X, int64_t ldx, const float* W, int64_t ldw, float* C1, int64_t ldc1, float* C2,
                             int64_t ldc2, int64_t M, int64_t N1, int64_t N2, int64_t K, cudaStream_t st) {
  if (M > 48 || M < 1 || N1 + N2 >= (1 << 24) || K >= (1 << 24)) return 0;
  if (K % 4 != 0 || K < 128 || ldx % 4 != 0 || ldw % 4 != 0 || !aligned16(X) || !aligned16(W)) return 0;
  const StreamEpilogue ep{nullptr, 0, nullptr, nullptr, 0, nullptr, C2, (int)N1, ldc2};
  const int m = (int)M, n = (int)(N1 + N2), k = (int)K;
  if (M <= 12) return launch_nt<12, 4>(X, ldx, W, ldw, C1, ldc1, m, n, k, ep, st);
  if (M <= 16) return launch_nt<16, 4>(X, ldx, W, ldw, C1, ldc1, m, n, k, ep, st);
  if (M <= 36) return launch_nt<36, 2>(X, ldx, W, ldw, C1, ldc1, m, n, k, ep, st);
  return launch_nt<48, 2>(X, ldx, W, ldw, C1, ldc1, m, n, k, ep, st);
}

}  // namespace cgvae

extern "C" {

int cgvae_register_const_range(const void* p, size_t bytes) {
  using namespace cgvae;
  if (p == nullptr || bytes == 0) {        // clear
    g_const_ranges.clear();
    return 0;
  }
  ConstRange r{reinterpret_cast<uintptr_t>(p), reinterpret_cast<uintptr_t>(p) + bytes};
  // insert, merging every range that overlaps or touches the new one
  std::vector<ConstRange> out;
  out.reserve(g_const_ranges.size() + 1);
  for (const ConstRange& q : g_const_ranges) {
    if (q.end < r.begin || q.begin > r.end) out.push_back(q);
    else {
      r.begin = std::min(r.begin, q.begin);
      r.end = std::max(r.end, q.end);
    }
  }
  out.push_back(r);
  std::sort(out.begin(), out.end(), [](const ConstRange& x, const ConstRange& y) { return x.begin < y.begin; });
  g_const_ranges.swap(out);
  return 0;
}

}  // extern "C"
