// Dense fp32 contractions (node phi-MLPs, UpdateBlock mixes, weight / input gradients).
// Round-1 implementation: register-tiled SIMT FMA kernel, three operand forms, fused epilogue
// (bias, pre-activation copy, activation, activation-backward, residual add), deterministic
// split-K for skinny problems (decoder graphs have 12..96 rows: weight streaming bound).
#include "common.cuh"
#include <cooperative_groups.h>

namespace cgvae {


struct Epilogue {
  const float* bias;   // [N] or null
  int act;             // forward activation applied to the value
  float* z_out;        // pre-activation copy or null
  const float* z_in;   // saved pre-activation for activation backward, or null
  int dact;            // activation code for z_in
  const float* add;    // residual [M][N] (ld = ldc) or null
};

__device__ __forceinline__ float apply_epilogue(const Epilogue& ep, float v, int64_t m, int64_t n, int64_t ldc) {
  if (ep.bias) v += ep.bias[n];
  if (ep.z_out) ep.z_out[m * ldc + n] = v;
  v = act_fwd(ep.act, v);
  if (ep.z_in) v *= act_bwd(ep.dact, ep.z_in[m * ldc + n]);
  if (ep.add) v += ep.add[m * ldc + n];
  return v;
}

// Loads a [ROWS x BK] operand tile into smem laid out as tile[k][row] (row stride ROWS+PAD).
// KCONTIG: global element (row, k) at ptr[row*ld + k] ; else at ptr[k*ld + row].
template <int ROWS, int BK, bool KCONTIG, int NTHREADS, int PAD = 4>
struct TileLoader {
  static constexpr int NVEC = ROWS * BK / 4;
  static constexpr int PER_THREAD = (NVEC + NTHREADS - 1) / NTHREADS;
  float4 reg[PER_THREAD];

  __device__ __forceinline__ void fetch(const float* __restrict__ ptr, int64_t ld, int64_t row0, int64_t nrows, int64_t k0,
                                        int64_t kend, bool vec_ok, int tid) {
#pragma unroll
    for (int p = 0; p < PER_THREAD; ++p) {
      const int v = tid + p * NTHREADS;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (v < NVEC) {
        if (KCONTIG) {
          const int r = v / (BK / 4), kq = v % (BK / 4);
          const int64_t row = row0 + r, k = k0 + kq * 4;
          if (row < nrows) {
            const float* src = ptr + row * ld + k;
            if (vec_ok && k + 3 < kend) {
              val = *reinterpret_cast<const float4*>(src);
            } else {
              if (k + 0 < kend) val.x = src[0];
              if (k + 1 < kend) val.y = src[1];
              if (k + 2 < kend) val.z = src[2];
              if (k + 3 < kend) val.w = src[3];
            }
          }
        } else {
          const int kk = v / (ROWS / 4), rq = v % (ROWS / 4);
          const int64_t k = k0 + kk, row = row0 + rq * 4;
          if (k < kend) {
            const float* src = ptr + k * ld + row;
            if (vec_ok && row + 3 < nrows) {
              val = *reinterpret_cast<const float4*>(src);
            } else {
              if (row + 0 < nrows) val.x = src[0];
              if (row + 1 < nrows) val.y = src[1];
              if (row + 2 < nrows) val.z = src[2];
              if (row + 3 < nrows) val.w = src[3];
            }
          }
        }
      }
      reg[p] = val;
    }
  }

  // smem layouts.  k-major tile[k][row] (row stride ROWS+4): vector reads in the inner loop, used by the large tile.
  // row-major tile[row][k] (row stride BK+1) for K-contiguous operands of the deep-k skinny tiles: the transposing
  // scatter of the k-major layout would be an 8-way bank conflict at BK = 64.
  static constexpr bool ROWMAJOR = KCONTIG && (BK > 16);
  static constexpr int SMEM_FLOATS = ROWMAJOR ? ROWS * (BK + 1) : BK * (ROWS + PAD);
  __device__ __forceinline__ static float at(const float* tile, int row, int k) {
    return ROWMAJOR ? tile[row * (BK + 1) + k] : tile[k * (ROWS + PAD) + row];
  }

  __device__ __forceinline__ void store(float* tile, int tid) {
#pragma unroll
    for (int p = 0; p < PER_THREAD; ++p) {
      const int v = tid + p * NTHREADS;
      if (v < NVEC) {
        if (KCONTIG) {
          const int r = v / (BK / 4), kq = v % (BK / 4);
          if (ROWMAJOR) {
            float* d = tile + r * (BK + 1) + kq * 4;
            d[0] = reg[p].x; d[1] = reg[p].y; d[2] = reg[p].z; d[3] = reg[p].w;
          } else {
            tile[(kq * 4 + 0) * (ROWS + PAD) + r] = reg[p].x;
            tile[(kq * 4 + 1) * (ROWS + PAD) + r] = reg[p].y;
            tile[(kq * 4 + 2) * (ROWS + PAD) + r] = reg[p].z;
            tile[(kq * 4 + 3) * (ROWS + PAD) + r] = reg[p].w;
          }
        } else {
          const int kk = v / (ROWS / 4), rq = v % (ROWS / 4);
          *reinterpret_cast<float4*>(&tile[kk * (ROWS + PAD) + rq * 4]) = reg[p];
        }
      }
    }
  }
};

// C tile BM x BN per CTA, TM x TN per thread, (BM/TM)*(BN/TN) threads.  gridDim.z = split-K factor:
// splits > 1 write raw partial sums to `partial[z][M][N]` and the epilogue runs in splitk_reduce_kernel.
// CLUSTER: the gridDim.z K-slices of one output tile form a thread-block cluster (1,1,S); partial tiles are exchanged
// through distributed shared memory and summed in slice order (deterministic) -- no global round trip, no second launch.
template <int BM, int BN, int BK, int TM, int TN, bool A_KC, bool B_KC, bool CLUSTER>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) gemm_kernel(
    const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
    int64_t M, int64_t N, int64_t K, int64_t k_per_split, Epilogue ep, float* __restrict__ partial, bool a_vec, bool b_vec) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int NT = (BM / TM) * (BN / TN);
  using LoaderA = TileLoader<BM, BK, A_KC, NT>;
  using LoaderB = TileLoader<BN, BK, B_KC, NT>;
  // one buffer: the double-buffered operand tiles during the k-loop, the CTA's partial output tile for the cluster
  // reduction afterwards (the tiles are dead by then)
  constexpr int SA = LoaderA::SMEM_FLOATS, SB = LoaderB::SMEM_FLOATS;
  constexpr int TILE_FLOATS = 2 * (SA + SB);
  constexpr int SMEM_FLOATS = (CLUSTER && BM * BN > TILE_FLOATS) ? BM * BN : TILE_FLOATS;
  __shared__ __align__(16) float smem_all[SMEM_FLOATS];
  float (*As)[SA] = reinterpret_cast<float (*)[SA]>(smem_all);
  float (*Bs)[SB] = reinterpret_cast<float (*)[SB]>(smem_all + 2 * SA);
  const int tid = threadIdx.x;
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const int64_t kbeg = (int64_t)blockIdx.z * k_per_split;
  const int64_t kend = min(K, kbeg + k_per_split);

  // two-level accumulation: `acc` is folded into `tot` every kFold k-tiles so the rounding error grows with
  // sqrt(kFold*BK) + sqrt(K/(kFold*BK)) instead of sqrt(K) (weight gradients reduce over up to 1e5 rows)
  constexpr int kFold = 256 / BK;
  float acc[TM][TN], tot[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) { acc[i][j] = 0.f; tot[i][j] = 0.f; }

  // PD k-tiles are kept in flight in registers (static slots, loop unrolled by PD): a CTA that streams a weight slab is a
  // chain of dependent DRAM round trips otherwise (one per k-tile: 10-25 us for the 13 MB decoder matrices).
  // (deeper prefetch for the 64x64x16 tile -- 6 tiles, 48 KB per CTA in flight -- measured SLOWER on B200: 57 vs 43 us for
  // the 350 x 600 <- 1800 input-gradient contraction: the tile is bound by shared-memory loads, not by load latency)
  constexpr int PD = (BK >= 32) ? 3 : 2;
  LoaderA las[PD];
  LoaderB lbs[PD];
#pragma unroll
  for (int p = 0; p < PD; ++p) {
    if (kbeg + (int64_t)p * BK < kend) {
      las[p].fetch(A, lda, m0, M, kbeg + (int64_t)p * BK, kend, a_vec, tid);
      lbs[p].fetch(B, ldb, n0, N, kbeg + (int64_t)p * BK, kend, b_vec, tid);
    }
  }
  int buf = 0;
  int fold = 0;
  for (int64_t base = kbeg; base < kend; base += (int64_t)PD * BK) {
#pragma unroll
    for (int p = 0; p < PD; ++p) {
      const int64_t k0 = base + (int64_t)p * BK;
      if (k0 < kend) {
        // tile k0 sits in register slot p; smem is double buffered, one barrier per tile
        las[p].store(As[buf], tid);
        lbs[p].store(Bs[buf], tid);
        __syncthreads();
        if (k0 + (int64_t)PD * BK < kend) {
          las[p].fetch(A, lda, m0, M, k0 + (int64_t)PD * BK, kend, a_vec, tid);
          lbs[p].fetch(B, ldb, n0, N, k0 + (int64_t)PD * BK, kend, b_vec, tid);
        }
#pragma unroll
        for (int k = 0; k < BK; ++k) {
          float a[TM], b[TN];
#pragma unroll
          for (int i = 0; i < TM; ++i) a[i] = LoaderA::at(As[buf], ty * TM + i, k);
#pragma unroll
          for (int j = 0; j < TN; ++j) b[j] = LoaderB::at(Bs[buf], tx * TN + j, k);
#pragma unroll
          for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (++fold == kFold) {
          fold = 0;
#pragma unroll
          for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) { tot[i][j] += acc[i][j]; acc[i][j] = 0.f; }
        }
        buf ^= 1;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] += tot[i][j];

  if constexpr (CLUSTER) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __syncthreads();                 // every warp is done reading the operand tiles
    float* red = smem_all;
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) red[(ty * TM + i) * BN + tx * TN + j] = acc[i][j];
    cluster.sync();
    const int S = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    // every CTA of the cluster finishes a strided share of the tile; slices are added in order 0..S-1
    for (int idx = rank * NT + tid; idx < BM * BN; idx += S * NT) {
      const int64_t m = m0 + idx / BN, n = n0 + idx % BN;
      float v = 0.f;
      for (int z = 0; z < S; ++z) v += *cluster.map_shared_rank(&red[idx], z);
      if (m < M && n < N) C[m * ldc + n] = apply_epilogue(ep, v, m, n, ldc);
    }
    cluster.sync();   // remote shared memory must stay alive until every CTA has read it
    return;
  }
  const bool split = gridDim.z > 1;
  float* dst = split ? partial + (int64_t)blockIdx.z * M * N : C;
  const int64_t ldd = split ? N : ldc;
  const int64_t nb = n0 + tx * TN;
  // a thread owns TN consecutive columns: store them as one vector when the row pointer allows it
  const bool vec_store = (TN == 2 || TN == 4) && (ldd % TN == 0) && (nb + TN <= N) &&
                         ((reinterpret_cast<uintptr_t>(dst) & (4 * TN - 1)) == 0);
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int64_t m = m0 + ty * TM + i;
    if (m >= M) continue;
    float o[TN];
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      o[j] = acc[i][j];
      if (!split && nb + j < N) o[j] = apply_epilogue(ep, acc[i][j], m, nb + j, ldc);
    }
    if (vec_store) {
      if (TN == 4) *reinterpret_cast<float4*>(dst + m * ldd + nb) = make_float4(o[0], o[1], o[2], o[3]);
      else *reinterpret_cast<float2*>(dst + m * ldd + nb) = make_float2(o[0], o[1]);
    } else {
#pragma unroll
      for (int j = 0; j < TN; ++j)
        if (nb + j < N) dst[m * ldd + nb + j] = o[j];
    }
  }
}

__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ partial, int splits, int64_t M, int64_t N,
                                                            float* __restrict__ C, int64_t ldc, Epilogue ep) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * N) return;
  const int64_t m = idx / N, n = idx % N;
  float v = 0.f;
  for (int s = 0; s < splits; ++s) v += partial[(int64_t)s * M * N + idx];  // fixed order: deterministic
  C[m * ldc + n] = apply_epilogue(ep, v, m, n, ldc);
}

// ------------------------------------------------------------------------------------------------------------
// Skinny kernel: M <= 16 rows (decoder graphs of the molecule configs: 12 beads).  The generic tile above is bound by
// shared-memory LOADS for such shapes (1x2 micro-tile: 3 LDS per 2 FMA, measured 15-25 us for the 13 MB matrices).
// Here a thread owns ONE output column and ALL 16 rows: per k it reads the 16 activations as four broadcast LDS.128
// and one weight element, i.e. 5 LDS per 16 FMA.  K is split over a thread-block cluster (1,1,S) and reduced through
// distributed shared memory in slice order.  A [M,K] is K-contiguous (NT and NN forms); B_KC selects W[N,K] (NT)
// or W[K,N] (NN).
// ------------------------------------------------------------------------------------------------------------
constexpr int SK_BK = 32;

template <int BN, bool B_KC>
__global__ void __launch_bounds__(BN) gemm_skinny_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B,
                                                        int64_t ldb, float* __restrict__ C, int64_t ldc, int64_t M, int64_t N,
                                                        int64_t K, int64_t k_per_split, Epilogue ep, bool a_vec, bool b_vec) {
  CGVAE_KERNEL_PROLOGUE();
  namespace cg = cooperative_groups;
  constexpr int NV_B = SK_BK * BN / 4 / BN;       // float4 of the weight tile per thread (= 8)
  __shared__ __align__(16) float As[2][SK_BK][20];          // k-major: As[k][row], 16 rows + pad
  __shared__ __align__(16) float Bs[2][SK_BK][BN + 4];      // k-major: Bs[k][n]
  __shared__ __align__(16) float red[16][BN];
  const int tid = threadIdx.x;
  const int64_t n0 = (int64_t)blockIdx.x * BN;
  const int64_t kbeg = (int64_t)blockIdx.z * k_per_split;
  const int64_t kend = min(K, kbeg + k_per_split);

  constexpr int NV_A = 128 / BN;                  // the activation tile is 16 rows x 8 chunks = 128 float4
  float4 a_reg[NV_A];
  float4 b_reg[NV_B];
  auto fetch = [&](int64_t k0) {
#pragma unroll
    for (int ia = 0; ia < NV_A; ++ia) {
      const int v = tid + BN * ia;
      const int r = v >> 3, c = v & 7;
      const int64_t k = k0 + 4 * c;
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < M) {
        const float* src = A + (int64_t)r * lda + k;
        if (a_vec && k + 3 < kend) x = __ldg(reinterpret_cast<const float4*>(src));
        else {
          if (k + 0 < kend) x.x = src[0];
          if (k + 1 < kend) x.y = src[1];
          if (k + 2 < kend) x.z = src[2];
          if (k + 3 < kend) x.w = src[3];
        }
      }
      a_reg[ia] = x;
    }
#pragma unroll
    for (int it = 0; it < NV_B; ++it) {
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (B_KC) {
        // W[N,K]: thread = output column n, it = k-chunk: 16 bytes of row n (the next chunk hits the same sector / line)
        const int64_t n = n0 + tid, k = k0 + 4 * it;
        if (n < N) {
          const float* src = B + n * ldb + k;
          if (b_vec && k + 3 < kend) x = __ldg(reinterpret_cast<const float4*>(src));
          else {
            if (k + 0 < kend) x.x = src[0];
            if (k + 1 < kend) x.y = src[1];
            if (k + 2 < kend) x.z = src[2];
            if (k + 3 < kend) x.w = src[3];
          }
        }
      } else {
        // W[K,N]: v = tid + BN*it -> k row = v / (BN/4), column quad = v % (BN/4): coalesced along n
        const int v = tid + BN * it;
        const int kk = v / (BN / 4), q = v % (BN / 4);
        const int64_t k = k0 + kk, n = n0 + 4 * q;
        if (k < kend) {
          const float* src = B + k * ldb + n;
          if (b_vec && n + 3 < N) x = __ldg(reinterpret_cast<const float4*>(src));
          else {
            if (n + 0 < N) x.x = src[0];
            if (n + 1 < N) x.y = src[1];
            if (n + 2 < N) x.z = src[2];
            if (n + 3 < N) x.w = src[3];
          }
        }
      }
      b_reg[it] = x;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int ia = 0; ia < NV_A; ++ia) {
      const int v = tid + BN * ia;
      const int r = v >> 3, c = v & 7;
      As[buf][4 * c + 0][r] = a_reg[ia].x;
      As[buf][4 * c + 1][r] = a_reg[ia].y;
      As[buf][4 * c + 2][r] = a_reg[ia].z;
      As[buf][4 * c + 3][r] = a_reg[ia].w;
    }
#pragma unroll
    for (int it = 0; it < NV_B; ++it) {
      if (B_KC) {
        Bs[buf][4 * it + 0][tid] = b_reg[it].x;
        Bs[buf][4 * it + 1][tid] = b_reg[it].y;
        Bs[buf][4 * it + 2][tid] = b_reg[it].z;
        Bs[buf][4 * it + 3][tid] = b_reg[it].w;
      } else {
        const int v = tid + BN * it;
        const int kk = v / (BN / 4), q = v % (BN / 4);
        *reinterpret_cast<float4*>(&Bs[buf][kk][4 * q]) = b_reg[it];
      }
    }
  };

  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  int buf = 0;
  if (kbeg < kend) fetch(kbeg);
  for (int64_t k0 = kbeg; k0 < kend; k0 += SK_BK) {
    stash(buf);
    __syncthreads();
    if (k0 + SK_BK < kend) fetch(k0 + SK_BK);
#pragma unroll
    for (int k = 0; k < SK_BK; ++k) {
      const float b = Bs[buf][k][tid];
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][0]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][4]);
      const float4 a2 = *reinterpret_cast<const float4*>(&As[buf][k][8]);
      const float4 a3 = *reinterpret_cast<const float4*>(&As[buf][k][12]);
      acc[0] = fmaf(a0.x, b, acc[0]);   acc[1] = fmaf(a0.y, b, acc[1]);   acc[2] = fmaf(a0.z, b, acc[2]);   acc[3] = fmaf(a0.w, b, acc[3]);
      acc[4] = fmaf(a1.x, b, acc[4]);   acc[5] = fmaf(a1.y, b, acc[5]);   acc[6] = fmaf(a1.z, b, acc[6]);   acc[7] = fmaf(a1.w, b, acc[7]);
      acc[8] = fmaf(a2.x, b, acc[8]);   acc[9] = fmaf(a2.y, b, acc[9]);   acc[10] = fmaf(a2.z, b, acc[10]); acc[11] = fmaf(a2.w, b, acc[11]);
      acc[12] = fmaf(a3.x, b, acc[12]); acc[13] = fmaf(a3.y, b, acc[13]); acc[14] = fmaf(a3.z, b, acc[14]); acc[15] = fmaf(a3.w, b, acc[15]);
    }
    buf ^= 1;
  }
  // cluster reduction over the K-slices, slice order 0..S-1 (deterministic), every CTA finishes a share of the rows
  cg::cluster_group cluster = cg::this_cluster();
#pragma unroll
  for (int i = 0; i < 16; ++i) red[i][tid] = acc[i];
  cluster.sync();
  const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int64_t n = n0 + tid;
  for (int i = rank; i < 16; i += S) {
    if (i < M && n < N) {
      float v = 0.f;
      for (int z = 0; z < S; ++z) v += *cluster.map_shared_rank(&red[i][tid], z);
      C[(int64_t)i * ldc + n] = apply_epilogue(ep, v, i, n, ldc);
    }
  }
  cluster.sync();
}

// column sums: out[n] = sum_m X[m][n]; one thread per column per row-chunk, two-stage, fixed order.
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ X, int64_t ldx, int64_t M, int64_t N,
                                                     float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  // blockDim = (32, 8): 32 columns x 8 row-lanes
  __shared__ float red[8][33];
  const int64_t n = (int64_t)blockIdx.x * 32 + threadIdx.x;
  float s = 0.f;
  if (n < N)
    for (int64_t m = threadIdx.y; m < M; m += 8) s += X[m * ldx + n];
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) t += red[r][threadIdx.x];
    out[n] = t;
  }
}

// tall matrices (bias gradients over 1e4 .. 1e5 node rows): the rows are split over a cluster (1, S, 1) and 32 row-lanes per
// CTA with four loads in flight per thread; CTA partials are combined by rank 0 through DSMEM in rank order (deterministic)
__global__ void __launch_bounds__(1024) colsum_tall_kernel(const float* __restrict__ X, int64_t ldx, int64_t M, int64_t N,
                                                           float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  namespace cgx = cooperative_groups;
  cgx::cluster_group cluster = cgx::this_cluster();
  __shared__ float red[32][33];
  __shared__ float part[32];
  const int S = (int)gridDim.y, z = (int)blockIdx.y;
  const int64_t rows_per = (M + S - 1) / S, m_lo = z * rows_per, m_hi = min(M, m_lo + rows_per);
  const int64_t n = (int64_t)blockIdx.x * 32 + threadIdx.x;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (n < N) {
    int64_t m = m_lo + threadIdx.y;
    for (; m + 96 < m_hi; m += 128) {
      s0 += X[m * ldx + n];
      s1 += X[(m + 32) * ldx + n];
      s2 += X[(m + 64) * ldx + n];
      s3 += X[(m + 96) * ldx + n];
    }
    for (; m < m_hi; m += 32) s0 += X[m * ldx + n];
  }
  red[threadIdx.y][threadIdx.x] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (threadIdx.y == 0) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) t += red[r][threadIdx.x];
    part[threadIdx.x] = t;
  }
  cluster.sync();
  if (z == 0 && threadIdx.y == 0 && n < N) {
    float t = 0.f;
    for (int rk = 0; rk < S; ++rk) t += cluster.map_shared_rank(part, rk)[threadIdx.x];
    out[n] = t;
  }
  cluster.sync();
}

template <int BM, int BN, int BK, int TM, int TN>
static int launch_gemm(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                       int64_t N, int64_t K, const Epilogue& ep, float* ws, size_t ws_bytes, cudaStream_t st) {
  constexpr int NT = (BM / TM) * (BN / TN);
  const int64_t tiles = ceil_div(M, BM) * ceil_div(N, BN);
  // split-K only when the output grid leaves most of the 148 SMs idle and K is deep
  int splits = 1;
  if (ws != nullptr && tiles < kNumSM && K >= 8 * BK) {
    splits = (int)std::min<int64_t>(ceil_div(2 * kNumSM, tiles), ceil_div(K, 128));
    const int64_t cap = (int64_t)(ws_bytes / (sizeof(float) * (size_t)(M * N)));
    splits = (int)std::max<int64_t>(1, std::min<int64_t>(splits, cap));
  }
  int64_t k_per_split = ceil_div(ceil_div(K, splits), BK) * BK;
  splits = (int)ceil_div(K, k_per_split);
  if (splits < 1) splits = 1;
  const bool a_kc = (form != CGVAE_GEMM_TN), b_kc = (form == CGVAE_GEMM_NT);
  const bool a_vec = aligned16(A) && (lda % 4 == 0), b_vec = aligned16(B) && (ldb % 4 == 0);
  if (tiles < kNumSM && K >= 8 * BK && form != CGVAE_GEMM_TN) {
    // cluster split-K: up to 8 K-slices per output tile (portable cluster size), reduced through DSMEM
    int S = (int)std::min<int64_t>(std::min<int64_t>(8, ceil_div(2 * kNumSM, tiles)), ceil_div(K, 128));
    int64_t kps = ceil_div(ceil_div(K, S), BK) * BK;
    S = (int)ceil_div(K, kps);
    if (S > 1) {
      const dim3 grid((unsigned)ceil_div(N, BN), (unsigned)ceil_div(M, BM), (unsigned)S), cluster(1, 1, (unsigned)S);
      if (b_kc)
        launch_cluster(gemm_kernel<BM, BN, BK, TM, TN, true, true, true>, grid, dim3(NT), cluster, 0, st, A, lda, B, ldb, C, ldc, M,
                       N, K, kps, ep, nullptr, a_vec, b_vec);
      else
        launch_cluster(gemm_kernel<BM, BN, BK, TM, TN, true, false, true>, grid, dim3(NT), cluster, 0, st, A, lda, B, ldb, C, ldc, M,
                       N, K, kps, ep, nullptr, a_vec, b_vec);
      return launched("gemm_cluster");
    }
  }
  dim3 grid((unsigned)ceil_div(N, BN), (unsigned)ceil_div(M, BM), (unsigned)splits);
  // partial sums are added by a second launch: inside a CUDA graph that costs less than an in-kernel "last CTA" fix-up
  // (fence + ticket: 6.0 vs 5.4 ms per chignolin step on B200)
  float* partial = splits > 1 ? ws : nullptr;
  if (a_kc && b_kc)
    launch_kernel(gemm_kernel<BM, BN, BK, TM, TN, true, true, false>, dim3(grid), dim3(NT), 0, st, A, lda, B, ldb, C, ldc, M, N, K, k_per_split, ep, partial, a_vec, b_vec);
  else if (a_kc && !b_kc)
    launch_kernel(gemm_kernel<BM, BN, BK, TM, TN, true, false, false>, dim3(grid), dim3(NT), 0, st, A, lda, B, ldb, C, ldc, M, N, K, k_per_split, ep, partial, a_vec, b_vec);
  else
    launch_kernel(gemm_kernel<BM, BN, BK, TM, TN, false, false, false>, dim3(grid), dim3(NT), 0, st, A, lda, B, ldb, C, ldc, M, N, K, k_per_split, ep, partial, a_vec, b_vec);
  if (int rc = launched("gemm")) return rc;
  if (splits > 1) {
    launch_kernel(splitk_reduce_kernel, dim3((unsigned)ceil_div(M * N, 256)), dim3(256), 0, st, (const float*)partial, splits, M, N,
                  C, ldc, ep);
    return launched("gemm_splitk_reduce");
  }
  return 0;
}

}  // namespace cgvae

namespace cgvae {
int launch_gemm_tcgen05(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                        int64_t N, int64_t K, const float* bias, int act, float* z_out, const float* z_in, int dact,
                        const float* add, float* ws, size_t ws_bytes, cudaStream_t st);
int launch_gemm_stream(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                       int64_t N, int64_t K, const float* bias, int act, float* z_out, const float* z_in, int dact,
                       const float* add, cudaStream_t st);
}

namespace cgvae {
int launch_dense_pair_stream(const float* X, int64_t ldx, const float* W, int64_t ldw, float* C1, int64_t ldc1, float* C2,
                             int64_t ldc2, int64_t M, int64_t N1, int64_t N2, int64_t K, cudaStream_t st);
}

using namespace cgvae;

extern "C" {

int cgvae_dense_pair_fwd(const float* x, int64_t ldx, const float* W, int64_t ldw, int64_t M, int64_t N1, int64_t N2, int64_t K,
                         float* C1, float* C2, cgvae_stream_t stream) {
  CGVAE_REQUIRE(M >= 0 && N1 >= 1 && N2 >= 1 && K >= 1, "dense_pair_fwd: bad sizes");
  if (M == 0) return 0;
  CGVAE_REQUIRE(x && W && C1 && C2, "dense_pair_fwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (launch_dense_pair_stream(x, ldx, W, ldw, C1, N1, C2, N2, M, N1, N2, K, st)) return launched("dense_pair_stream");
  // not eligible for the weight-streaming kernel: two ordinary launches
  if (int rc = cgvae_gemm(CGVAE_GEMM_NT, x, ldx, W, ldw, C1, N1, M, N1, K, nullptr, 0, nullptr, nullptr, 0, nullptr, nullptr, 0,
                          nullptr, 0, stream))
    return rc;
  return cgvae_gemm(CGVAE_GEMM_NT, x, ldx, W + N1 * ldw, ldw, C2, N2, M, N2, K, nullptr, 0, nullptr, nullptr, 0, nullptr, nullptr, 0,
                    nullptr, 0, stream);
}

int cgvae_gemm(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M, int64_t N,
               int64_t K, const float* bias, int act, float* z_out, const float* z_in, int dact, const float* add,
               void* ws, size_t ws_bytes, int32_t* /*counters*/, int /*n_counters*/, cgvae_stream_t stream) {
  CGVAE_REQUIRE(form >= 0 && form <= 2, "gemm: bad form %d", form);
  CGVAE_REQUIRE(M >= 0 && N >= 0 && K >= 0, "gemm: negative size");
  if (M == 0 || N == 0) return 0;
  CGVAE_REQUIRE(A && B && C, "gemm: null operand");
  CGVAE_REQUIRE(ldc >= N, "gemm: ldc < N");
  Epilogue ep{bias, act, z_out, z_in, dact, add};
  cudaStream_t st = (cudaStream_t)stream;
  // large node GEMMs: 3xTF32 on the tcgen05 tensor cores (gemm_tc.cu); everything else: fp32 SIMT tiles below
  if (int tc_rc = launch_gemm_tcgen05(form, A, lda, B, ldb, C, ldc, M, N, K, bias, act, z_out, z_in, dact, add,
                                      reinterpret_cast<float*>(ws), ws_bytes, st)) {
    if (int rc = launched("gemm_tcgen05")) return rc;
    if (tc_rc > 1) {     // several cluster groups: add their partial matrices in group order, then the epilogue
      launch_kernel(splitk_reduce_kernel, dim3((unsigned)ceil_div(M * N, 256)), dim3(256), 0, st, (const float*)ws, tc_rc - 1, M, N, C,
                    ldc, ep);
      return launched("gemm_splitk_reduce");
    }
    return 0;
  }
  // M <= 48 rows (decoder graphs): weight-streaming kernels (gemm_stream.cu)
  if (launch_gemm_stream(form, A, lda, B, ldb, C, ldc, M, N, K, bias, act, z_out, z_in, dact, add, st))
    return launched("gemm_stream");
  float* wsf = reinterpret_cast<float*>(ws);
  // measured in isolation inside a CUDA graph (tools/bench_skinny.py, weights rotated through > L2): the column-per-thread
  // kernel wins for wide outputs (W2 forward, 5400 columns: 17.9 vs 23.2 us) and loses where 8 cluster slices of 64-wide
  // tiles leave too few threads in flight (N = 600 outputs: 80 CTAs x 64 threads), so it takes the NT form with N >= 1024
  if (M <= 16 && form == CGVAE_GEMM_NT && K >= 64 && N >= 1024) {
    // one output column per thread, K split over a cluster of up to 8 CTAs
    const bool b_kc = (form == CGVAE_GEMM_NT);
    const bool a_vec = aligned16(A) && (lda % 4 == 0), b_vec = aligned16(B) && (ldb % 4 == 0);
    const bool narrow = ceil_div(N, 128) * 8 < kNumSM;        // few columns: 64-wide tiles double the CTA count
    const int BNs = narrow ? 64 : 128;
    const int64_t tiles = ceil_div(N, BNs);
    int S = (int)std::min<int64_t>(std::min<int64_t>(8, std::max<int64_t>(1, ceil_div(2 * kNumSM, tiles))), ceil_div(K, 2 * SK_BK));
    int64_t kps = ceil_div(ceil_div(K, S), SK_BK) * SK_BK;
    S = (int)ceil_div(K, kps);
    const dim3 grid((unsigned)tiles, 1, (unsigned)S), cluster(1, 1, (unsigned)S);
    if (narrow) {
      if (b_kc) launch_cluster(gemm_skinny_kernel<64, true>, grid, dim3(BNs), cluster, 0, st, A, lda, B, ldb, C, ldc, M, N, K, kps, ep, a_vec, b_vec);
      else launch_cluster(gemm_skinny_kernel<64, false>, grid, dim3(BNs), cluster, 0, st, A, lda, B, ldb, C, ldc, M, N, K, kps, ep, a_vec, b_vec);
    } else {
      if (b_kc) launch_cluster(gemm_skinny_kernel<128, true>, grid, dim3(BNs), cluster, 0, st, A, lda, B, ldb, C, ldc, M, N, K, kps, ep, a_vec, b_vec);
      else launch_cluster(gemm_skinny_kernel<128, false>, grid, dim3(BNs), cluster, 0, st, A, lda, B, ldb, C, ldc, M, N, K, kps, ep, a_vec, b_vec);
    }
    return launched("gemm_skinny");
  }
  // skinny problems (decoder graphs: 12..96 rows) stream the weight matrix: deep k-tiles keep 8-16 KB per CTA in flight
  if (M <= 16) return launch_gemm<16, 32, 64, 1, 2>(form, A, lda, B, ldb, C, ldc, M, N, K, ep, wsf, ws_bytes, st);
  if (M <= 32) return launch_gemm<32, 32, 64, 2, 2>(form, A, lda, B, ldb, C, ldc, M, N, K, ep, wsf, ws_bytes, st);
  if (M <= 48 && form != CGVAE_GEMM_TN)   // UpdateBlock mixes on 12-bead graphs: 36 rows
    return launch_gemm<48, 32, 32, 3, 2>(form, A, lda, B, ldb, C, ldc, M, N, K, ep, wsf, ws_bytes, st);
  // 64x64 tiles: a 128x64 tile with 8x4 per thread measured slower on B200 at the chignolin atom-level layers (350 rows,
  // 3.55 vs 3.49 ms per step): 3 row tiles of 128 waste 9 % and halve the CTA count
  return launch_gemm<64, 64, 16, 4, 4>(form, A, lda, B, ldb, C, ldc, M, N, K, ep, wsf, ws_bytes, st);
}

int cgvae_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, cgvae_stream_t stream) {
  if (N == 0) return 0;
  CGVAE_REQUIRE(X && out, "colsum: null pointer");
  if (M >= 4096) {
    const int blocks = (int)ceil_div(N, 32);
    int S = (int)std::min<int64_t>(8, std::max<int64_t>(1, (2 * kNumSM) / blocks));
    while (S & (S - 1)) S &= S - 1;
    launch_cluster(colsum_tall_kernel, dim3((unsigned)blocks, (unsigned)S, 1), dim3(32, 32, 1), dim3(1, (unsigned)S, 1), 0,
                   (cudaStream_t)stream, X, ldx, M, N, out);
    return launched("colsum_tall");
  }
  launch_kernel(colsum_kernel, dim3((unsigned)ceil_div(N, 32)), dim3(dim3(32, 8)), 0, (cudaStream_t)stream, X, ldx, M, N, out);
  return launched("colsum");
}

}  // extern "C"
