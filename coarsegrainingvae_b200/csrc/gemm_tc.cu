// 3xTF32 GEMM on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM) for every node-level contraction
// with >= 64 rows: the phi-MLPs / UpdateBlock mixes of the atom graphs (350 rows at chignolin, 1e4 .. 1e5 rows for the
// protein configurations), their input gradients (NN) and their weight gradients (TN).
//
// fp32 parity needs more than one TF32 pass.  The tensor core reads the upper 19 bits of a 32-bit operand, i.e. it sees
//   hi = trunc_tf32(x);      the remainder  x - hi  is exact in fp32 and   lo = rn_tf32(x - hi)
// so   A*B ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi   with the RAW fp32 tile standing in for `hi`: operands arrive by TMA
// (cp.async.bulk.tensor, SWIZZLE_128B) exactly as they lie in global memory, no register staging, and the only SIMT work
// per k-step is the element-wise, layout-agnostic lo pass: smem -> registers -> smem at the same (swizzled) offset.
//
// Operand tiles (BK = 32 fp32 = one 128-byte swizzle row):
//   K-contiguous operand (A of NT / NN, B of NT): one box [rows][32 k]  -> canonical K-major  SW128 (SBO = 1024)
//   MN-contiguous operand (B of NN, A and B of TN): rows/32 boxes [32 k][32 mn] of 4 KB each, TMA swizzle 128B_ATOM_32B
//                 -> canonical MN-major SWIZZLE_128B_BASE32B, the only MN-major layout of 32-bit operands (32-byte chunks
//                    XOR-ed with the k-row modulo 4; LBO = 4096 between 32-wide MN atoms, SBO = 512 between 4-row k groups)
// so all three forms share one pipeline and nothing is transposed by threads (instruction-descriptor bits 15 / 16).
//
// Warp roles: warps 0..7 lo pass + epilogue, warp 8 TMA producer, warp 9 MMA issuer (one elected lane of the converged
// warp).  Small problems (350-row layers: 15 .. 75 output tiles for 148 SMs) split K over a thread-block cluster (1,1,S<=8):
// every CTA parks its partial tile in its own shared memory and CTA r reduces rows [r*128/S, (r+1)*128/S) of all S
// partials through distributed shared memory in rank order (deterministic), applying the fused epilogue.
#include "tc_common.cuh"
#include <cooperative_groups.h>
#include <cuda.h>

namespace cgvae {

namespace tc {

using namespace tcx;
namespace cg = cooperative_groups;

constexpr int BM = 128, BN = 128, BK = 32, STAGES = 3;
constexpr int NUM_SPLIT_WARPS = 8;
constexpr int NUM_THREADS = (NUM_SPLIT_WARPS + 2) * 32;
constexpr uint32_t A_BYTES = BM * BK * 4, B_BYTES = BN * BK * 4;      // 16 KB each
constexpr uint32_t RAW_BYTES = A_BYTES + B_BYTES;                      // [A raw | B raw]
constexpr uint32_t STAGE_BYTES = 2 * RAW_BYTES;                        // [raw | lo]
constexpr uint32_t BAR_BYTES = 256;
constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;   // + slack for the 1024-byte alignment
// TMEM accumulation truncates: every accumulate step loses up to one ulp of the accumulator, one-sided, so the error of a
// single accumulator grows linearly with the number of MMAs chained on it (measured: 3.5e-6 of the result scale after 16
// k-steps x 12 MMAs, 8.6e-6 after 32).  Two remedies, both free on an otherwise idle TMEM:
//   * the two small products (A_lo*B_hi, A_hi*B_lo; 2^-11 of the result) go to their OWN accumulator: their truncation is
//     relative to that small sum -> the big accumulator sees one MMA per K = 8 instead of three;
//   * NBIG big accumulators take the k-steps round-robin: each carries 1/NBIG of the sum over 1/NBIG of the steps.
// The epilogue adds the four accumulators in fp32 (round to nearest).  512 columns = the whole TMEM (one CTA per SM anyway).
constexpr int NBIG = 3;
constexpr uint32_t TMEM_COLS = 512;
static_assert((1 + NBIG) * BN <= (int)TMEM_COLS, "accumulators must fit in TMEM");
constexpr int PS = BN + 4;                                             // row stride (floats) of a parked partial tile
constexpr int MAX_KT_PER_CTA = 96;   // longest accumulation chain per CTA (k-steps of 32): keeps the 1e-5 gate with margin
constexpr int MIN_M = 64;            // fewer rows: the SIMT tiles and the weight-streaming kernels (gemm.cu, gemm_stream.cu)

struct Ep {
  const float* bias;
  int act;
  float* z_out;
  const float* z_in;
  int dact;
  const float* add;
};

__device__ __forceinline__ float ep_apply(const Ep& ep, float v, int64_t m, int64_t n, int64_t ldc) {
  if (ep.bias) v += ep.bias[n];
  if (ep.z_out) ep.z_out[m * ldc + n] = v;
  v = act_fwd(ep.act, v);
  if (ep.z_in) v *= act_bwd(ep.dact, ep.z_in[m * ldc + n]);
  if (ep.add) v += ep.add[m * ldc + n];
  return v;
}

// One 32-row x 32-column block from a warp's transpose buffer (tr[row][33]) to C, lane = column.  The epilogue variant is
// chosen ONCE per kernel (the per-element `ep_apply` with its pointer tests, 64-bit index arithmetic and run-time activation
// switch was 60 % of the kernel's instructions at the 16 000 x 2048 x 512 layer): MODE 0 plain, 1 + bias, 2 + bias and swish
// (the phi-MLP hidden layer), 3 generic.
__device__ __forceinline__ int ep_mode(const Ep& ep) {
  // backward forms: input gradient through a swish layer (v * swish'(z_in)), residual / accumulating add
  if (!ep.bias && !ep.z_out && ep.act == 0) {
    if (ep.z_in && !ep.add && ep.dact == CGVAE_ACT_SWISH) return 4;
    if (ep.add && !ep.z_in) return 5;
  }
  // forward hidden layer of a phi-MLP in training: bias, pre-activation copy (saved for the backward), swish
  if (ep.z_out && ep.bias && !ep.z_in && !ep.add && ep.act == CGVAE_ACT_SWISH) return 6;
  if (ep.z_out || ep.z_in || ep.add) return 3;
  if (ep.act == 0) return ep.bias ? 1 : 0;
  return (ep.act == CGVAE_ACT_SWISH && ep.bias) ? 2 : 3;
}
template <int MODE>
__device__ __forceinline__ void store_block_mode(const Ep& ep, const float* __restrict__ tr, int lane, float* __restrict__ C, int64_t ldc,
                                                 int64_t m_base, int64_t n, int64_t M, int64_t N) {
  if (n >= N) return;
  const int rows = (int)min((int64_t)32, M - m_base);
  float* dst = C + m_base * ldc + n;
  const float b = (MODE == 1 || MODE == 2 || MODE == 6) ? __ldg(ep.bias + n) : 0.f;
  if constexpr (MODE == 4 || MODE == 5) {
    // the second operand of the epilogue (z_in / add) is as large as the output: all 32 row loads of this block are issued
    // before the first is used -- read one by one inside the store loop (4 in flight per warp) this epilogue ran at ~0.3 TB/s
    const float* aux = ((MODE == 4) ? ep.z_in : ep.add) + m_base * ldc + n;
    float a[32];
#pragma unroll
    for (int rr = 0; rr < 32; ++rr) a[rr] = (rr < rows) ? __ldg(aux + (int64_t)rr * ldc) : 0.f;
#pragma unroll
    for (int rr = 0; rr < 32; ++rr) {
      if (rr < rows) {
        const float v = tr[rr * 33 + lane];
        dst[(int64_t)rr * ldc] = (MODE == 4) ? v * dswish_f(a[rr]) : v + a[rr];
      }
    }
  } else {
#pragma unroll 4
    for (int rr = 0; rr < rows; ++rr, dst += ldc) {
      float v = tr[rr * 33 + lane];
      if (MODE == 3) {
        *dst = ep_apply(ep, v, m_base + rr, n, ldc);
      } else {
        v += b;
        if (MODE == 6) ep.z_out[(m_base + rr) * ldc + n] = v;
        if (MODE == 2 || MODE == 6) v = swish_f(v);
        *dst = v;
      }
    }
  }
}
// one element through the epilogue variant MODE (see ep_mode)
template <int MODE>
__device__ __forceinline__ float ep_apply_mode(const Ep& ep, float v, int64_t m, int64_t n, int64_t ldc) {
  if (MODE == 0) return v;
  if (MODE == 1) return v + __ldg(ep.bias + n);
  if (MODE == 2) return swish_f(v + __ldg(ep.bias + n));
  if (MODE == 4) return v * dswish_f(__ldg(ep.z_in + m * ldc + n));
  if (MODE == 5) return v + __ldg(ep.add + m * ldc + n);
  if (MODE == 6) {
    const float zz = v + __ldg(ep.bias + n);
    ep.z_out[m * ldc + n] = zz;
    return swish_f(zz);
  }
  return ep_apply(ep, v, m, n, ldc);
}
// rows [r_lo, r_hi) of the output tile = sum of the S parked partial tiles of the cluster in rank order, through the epilogue
template <int MODE>
__device__ __forceinline__ void cluster_reduce_rows(const Ep& ep, cg::cluster_group& cluster, float* P, int S, int r_lo, int r_hi, int tid,
                                                    float* __restrict__ C, int64_t ldc, int64_t m0, int64_t n0, int64_t M, int64_t N) {
  for (int idx = tid; idx < (r_hi - r_lo) * (BN / 4); idx += NUM_THREADS) {
    const int row = r_lo + idx / (BN / 4), c4 = (idx % (BN / 4)) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int rk = 0; rk < S; ++rk) {
      const float4 v = *reinterpret_cast<const float4*>(cluster.map_shared_rank(P, rk) + row * PS + c4);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
    const int64_t m = m0 + row, n = n0 + c4;
    if (m < M) {
      float* dst = C + m * ldc + n;
      if (n + 0 < N) dst[0] = ep_apply_mode<MODE>(ep, acc.x, m, n + 0, ldc);
      if (n + 1 < N) dst[1] = ep_apply_mode<MODE>(ep, acc.y, m, n + 1, ldc);
      if (n + 2 < N) dst[2] = ep_apply_mode<MODE>(ep, acc.z, m, n + 2, ldc);
      if (n + 3 < N) dst[3] = ep_apply_mode<MODE>(ep, acc.w, m, n + 3, ldc);
    }
  }
}

__device__ __forceinline__ void store_block(int mode, const Ep& ep, const float* __restrict__ tr, int lane, float* __restrict__ C,
                                            int64_t ldc, int64_t m_base, int64_t n, int64_t M, int64_t N) {
  switch (mode) {                       // warp-uniform
    case 0: store_block_mode<0>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    case 1: store_block_mode<1>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    case 2: store_block_mode<2>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    case 4: store_block_mode<4>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    case 5: store_block_mode<5>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    case 6: store_block_mode<6>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
    default: store_block_mode<3>(ep, tr, lane, C, ldc, m_base, n, M, N); break;
  }
}

// shared-memory matrix descriptor, descriptor version 1 (sm_100); layout type in bits 61..63:
//   K-major operand: SWIZZLE_128B (2), SBO = 1024 (8-row groups), LBO unused;  MN-major: SWIZZLE_128B_BASE32B (1)
template <bool KC>
__device__ __forceinline__ uint64_t make_desc_op(uint32_t smem_addr) {
  constexpr uint32_t lbo = KC ? 16u : 4096u, sbo = KC ? 1024u : 512u;
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(KC ? 2 : 1) << 61;
  return d;
}

__device__ __forceinline__ void tma_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}

// lo = rn_tf32(x - trunc_tf32(x)): the part of x the tensor core does not see, rounded (to nearest) to what it can see
__device__ __forceinline__ float lo_of(float x) {
  const float r = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  return __uint_as_float((__float_as_uint(r) + 0x1000u) & 0xFFFFE000u);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

// 32 columns of the result for this thread's row: small accumulator + the big accumulators that were written, in order
__device__ __forceinline__ void load_acc(uint32_t taddr, int nbig, float (&out)[32]) {
  if (nbig == 0) {                       // empty K-slice
#pragma unroll
    for (int j = 0; j < 32; ++j) out[j] = 0.f;
    return;
  }
  uint32_t r[32], t[32];
  tmem_ld32(taddr, r);
  tmem_ld32(taddr + BN, t);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < 32; ++j) out[j] = __uint_as_float(r[j]) + __uint_as_float(t[j]);
#pragma unroll 1
  for (int b = 1; b < nbig; ++b) {
    tmem_ld32(taddr + (uint32_t)(1 + b) * BN, t);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 32; ++j) out[j] += __uint_as_float(t[j]);
  }
}

// ONE = false: 3xTF32 (the default).  ONE = true: 1xTF32 (cgvae_set_matmul_precision(1)) -- the stage holds the raw tile
// only, rounded to nearest TF32 in place by the split warps, so twice as many stages fit in the same shared memory, and
// one MMA per K = 8 accumulates into a single accumulator (its truncation drift, <= chain length x 2^-23 relative, is
// negligible next to the 2^-11 of the operand rounding).
template <bool ONE>
struct Ring {
  static constexpr int STAGES = ONE ? 2 * tc::STAGES : tc::STAGES;
  static constexpr uint32_t STAGE_BYTES = ONE ? RAW_BYTES : tc::STAGE_BYTES;
  static_assert(STAGES * STAGE_BYTES == tc::STAGES * tc::STAGE_BYTES, "both forms use the same shared memory");
    static_assert(3 * STAGES * 8 + 4 * 8 + 4 <= (int)BAR_BYTES, "barriers must fit in BAR_BYTES");
};

// the split warps' pass over one landed stage: 3xTF32 writes the lo tile next to the raw one; 1xTF32 rounds the raw tile
// to nearest TF32 in place (the tensor core would truncate: a one-sided error that grows with K instead of averaging out)
template <bool ONE, int NT>
__device__ __forceinline__ void split_stage(char* stage, int t) {
  const float4* raw = reinterpret_cast<const float4*>(stage);
  constexpr int PER = (int)(RAW_BYTES / 16) / NT;   // 8 float4 per thread
  float4 x[PER];
#pragma unroll
  for (int it = 0; it < PER; ++it) x[it] = raw[t + it * NT];
  if constexpr (ONE) {
    float4* rawm = reinterpret_cast<float4*>(stage);
#pragma unroll
    for (int it = 0; it < PER; ++it)
      rawm[t + it * NT] = make_float4(to_tf32(x[it].x), to_tf32(x[it].y), to_tf32(x[it].z), to_tf32(x[it].w));
  } else {
    float4* lo = reinterpret_cast<float4*>(stage + RAW_BYTES);
#pragma unroll
    for (int it = 0; it < PER; ++it) {
      float4 l;
      l.x = lo_of(x[it].x);
      l.y = lo_of(x[it].y);
      l.z = lo_of(x[it].z);
      l.w = lo_of(x[it].w);
      lo[t + it * NT] = l;
    }
  }
}

// 32 columns of the single 1xTF32 accumulator for this thread's row
__device__ __forceinline__ void load_acc1(uint32_t taddr, bool any, float (&out)[32]) {
  if (!any) {                            // empty K-slice
#pragma unroll
    for (int j = 0; j < 32; ++j) out[j] = 0.f;
    return;
  }
  uint32_t r[32];
  tmem_ld32(taddr, r);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < 32; ++j) out[j] = __uint_as_float(r[j]);
}

template <bool A_KC, bool B_KC, bool ONE>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& map_a, const CUtensorMap& map_b, float* __restrict__ C, int64_t ldc,
                                             int64_t M, int64_t N, int64_t K, int kt_per_split, const Ep& ep, int cluster_size,
                                             float* __restrict__ partial, int b_const) {
  constexpr int STAGES = Ring<ONE>::STAGES;
  constexpr uint32_t STAGE_BYTES = Ring<ONE>::STAGE_BYTES;
  // b_const: B is a weight matrix inside a registered parameter range -- the producer issues its first tiles BEFORE the
  // dependency wait of the programmatic dependent launch (they overlap with the preceding kernel), A follows the wait
  if (!b_const) CGVAE_KERNEL_PROLOGUE();
  extern __shared__ __align__(1024) char smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte aligned bases: add the (runtime) pad to the extern array, not to an integer
  char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* raw_full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* lo_done = raw_full + STAGES;
  uint64_t* empty_bar = lo_done + STAGES;
  uint64_t* acc_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_sh = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const int num_kt = (int)((K + BK - 1) / BK);
  // gridDim.z = groups x cluster_size K-slices: a cluster reduces its slices through DSMEM; with more than one group
  // (reductions over > 8 x MAX_KT_PER_CTA k-steps) every group writes a raw partial matrix and splitk_reduce_kernel
  // (gemm.cu) adds the groups in order and applies the epilogue
  const int S = cluster_size, z = (int)blockIdx.z % cluster_size, group = (int)blockIdx.z / cluster_size;
  const int kt0 = (int)blockIdx.z * kt_per_split, kt1 = min(num_kt, kt0 + kt_per_split);
  const int nkt = max(0, kt1 - kt0);        // trailing slices of the last group may be empty: they park zeros
  if (partial != nullptr) {
    C = partial + (int64_t)group * M * N;
    ldc = N;
  }

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&raw_full[s], 1);
      mbar_init(&lo_done[s], NUM_SPLIT_WARPS);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(acc_bar, 1);
    mbar_fence_init();
  }
  if (warp == NUM_SPLIT_WARPS + 1) tmem_alloc<TMEM_COLS>(tmem_ptr_sh);   // the MMA warp owns the TMEM allocation
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_sh;
  const uint32_t smem_base = smem_u32(smem);
  const int npre = b_const ? min(nkt, STAGES) : 0;
  if (b_const) {
    if (warp == NUM_SPLIT_WARPS) {
      if (elect_one()) {
        for (int i = 0; i < npre; ++i) {
          const int k0 = (kt0 + i) * BK;
          const uint32_t b_dst = smem_base + (uint32_t)i * STAGE_BYTES + A_BYTES;
          mbar_expect_tx(&raw_full[i], RAW_BYTES);
          if (B_KC) {
            tma_2d(b_dst, &map_b, k0, (int)n0, &raw_full[i]);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 32; ++j) tma_2d(b_dst + (uint32_t)j * 4096u, &map_b, (int)n0 + 32 * j, k0, &raw_full[i]);
          }
        }
      }
      __syncwarp();
    }
    CGVAE_KERNEL_PROLOGUE();
  }

  if (warp < NUM_SPLIT_WARPS) {
    // ---------------- lo pass: raw tile -> lo tile, same physical offset (the swizzle is irrelevant element-wise) ----------
    for (int i = 0; i < nkt; ++i) {
      const int s = i % STAGES;
      mbar_wait(&raw_full[s], (uint32_t)(i / STAGES) & 1u);
      split_stage<ONE, NUM_SPLIT_WARPS * 32>(smem + (uint32_t)s * STAGE_BYTES, tid);
      fence_async_smem();            // generic-proxy writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&lo_done[s]);
    }
  } else if (warp == NUM_SPLIT_WARPS) {
    // ---------------- TMA producer ----------------
    for (int i = 0; i < nkt; ++i) {
      const int s = i % STAGES;
      mbar_wait(&empty_bar[s], ((uint32_t)(i / STAGES) & 1u) ^ 1u);
      if (elect_one()) {
        const int k0 = (kt0 + i) * BK;
        const uint32_t a_dst = smem_base + (uint32_t)s * STAGE_BYTES, b_dst = a_dst + A_BYTES;
        if (i >= npre) mbar_expect_tx(&raw_full[s], RAW_BYTES);
        if (A_KC) {
          tma_2d(a_dst, &map_a, k0, (int)m0, &raw_full[s]);
        } else {
#pragma unroll
          for (int j = 0; j < BM / 32; ++j) tma_2d(a_dst + (uint32_t)j * 4096u, &map_a, (int)m0 + 32 * j, k0, &raw_full[s]);
        }
        if (i >= npre) {
          if (B_KC) {
            tma_2d(b_dst, &map_b, k0, (int)n0, &raw_full[s]);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 32; ++j) tma_2d(b_dst + (uint32_t)j * 4096u, &map_b, (int)n0 + 32 * j, k0, &raw_full[s]);
          }
        }
      }
      __syncwarp();
    }
  } else {
    // ---------------- MMA issuer: the whole warp stays in the loop, one elected lane drives the tensor core ----------------
    constexpr uint32_t idesc = idesc_tf32(BM, BN, !A_KC, !B_KC);
    constexpr uint32_t a_step = A_KC ? 32u : 1024u, b_step = B_KC ? 32u : 1024u;     // one MMA consumes K = 8
    for (int i = 0; i < nkt; ++i) {
      const int s = i % STAGES;
      mbar_wait(&lo_done[s], (uint32_t)(i / STAGES) & 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_hi = smem_base + (uint32_t)s * STAGE_BYTES, b_hi = a_hi + A_BYTES;
        const uint32_t a_lo = a_hi + RAW_BYTES, b_lo = b_hi + RAW_BYTES;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
          const uint32_t ao = (uint32_t)ks * a_step, bo = (uint32_t)ks * b_step;
          if constexpr (ONE) {
            umma_tf32_ss(tmem_base, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_hi + bo), (i > 0 || ks > 0) ? 1u : 0u, idesc);
          } else {
            const uint32_t d_big = tmem_base + (uint32_t)(1 + i % NBIG) * BN;
            umma_tf32_ss(tmem_base, make_desc_op<A_KC>(a_lo + ao), make_desc_op<B_KC>(b_hi + bo), (i > 0 || ks > 0) ? 1u : 0u, idesc);
            umma_tf32_ss(tmem_base, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_lo + bo), 1u, idesc);
            umma_tf32_ss(d_big, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_hi + bo), (i >= NBIG || ks > 0) ? 1u : 0u, idesc);
          }
        }
        umma_commit(&empty_bar[s]);                  // stage reusable once these MMAs have read it
        if (i == nkt - 1) umma_commit(acc_bar);      // accumulator complete
      }
      __syncwarp();
    }
  }

  // ---------------- epilogue ----------------
  // warp w < 8 reads TMEM lanes 32*(w%4)..+31 (= output rows) and the column half (w/4)
  if (warp < NUM_SPLIT_WARPS && nkt > 0) {
    mbar_wait(acc_bar, 0);
    tc_fence_after();
  }
  if (S == 1) {
    if (warp < NUM_SPLIT_WARPS) {
      // 32x32 blocks through shared memory (the stages are free by now) so that a warp writes 128 contiguous bytes per row
      const int q = warp & 3, half = warp >> 2;
      const int mode = ep_mode(ep);
      float* tr = reinterpret_cast<float*>(smem) + warp * (32 * 33);
#pragma unroll 1
      for (int cb = 0; cb < BN / 64; ++cb) {
        const int c0 = half * (BN / 2) + cb * 32;
        float r[32];
        if constexpr (ONE) load_acc1(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, nkt > 0, r);
        else load_acc(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, min(nkt, NBIG), r);
#pragma unroll
        for (int j = 0; j < 32; ++j) tr[lane * 33 + j] = r[j];   // row = lane, column = j
        __syncwarp();
        if (m0 + 32 * q < M) store_block(mode, ep, tr, lane, C, ldc, m0 + 32 * q, n0 + c0 + lane, M, N);
        __syncwarp();
      }
      tc_fence_before();
    }
    __syncthreads();
  } else {
    // split-K over the cluster: park the partial tile, then reduce a row slice of all partials in rank order
    cg::cluster_group cluster = cg::this_cluster();
    float* P = reinterpret_cast<float*>(smem);
    if (warp < NUM_SPLIT_WARPS) {
      const int q = warp & 3, half = warp >> 2;
      const int row = 32 * q + lane;
#pragma unroll 1
      for (int cb = 0; cb < BN / 64; ++cb) {
        const int c0 = half * (BN / 2) + cb * 32;
        float r[32];
        if constexpr (ONE) load_acc1(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, nkt > 0, r);
        else load_acc(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, min(nkt, NBIG), r);
#pragma unroll
        for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(P + row * PS + c0 + j) = make_float4(r[j], r[j + 1], r[j + 2], r[j + 3]);
      }
      tc_fence_before();
    }
    cluster.sync();
    const int rows_per = (BM + S - 1) / S;
    const int r_lo = z * rows_per, r_hi = min(BM, r_lo + rows_per);
    switch (ep_mode(ep)) {           // CTA-uniform
      case 0: cluster_reduce_rows<0>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      case 1: cluster_reduce_rows<1>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      case 2: cluster_reduce_rows<2>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      case 4: cluster_reduce_rows<4>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      case 5: cluster_reduce_rows<5>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      case 6: cluster_reduce_rows<6>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
      default: cluster_reduce_rows<3>(ep, cluster, P, S, r_lo, r_hi, tid, C, ldc, m0, n0, M, N); break;
    }
    cluster.sync();                  // nobody leaves while a peer may still read its partial tile
  }
  if (warp == NUM_SPLIT_WARPS + 1) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

#define GEMM_TC_PARAMS                                                                                                          \
  const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, float* __restrict__ C, int64_t ldc,    \
      int64_t M, int64_t N, int64_t K, int kt_per_split, Ep ep, int cluster_size, float* __restrict__ partial, int b_const
template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(NUM_THREADS, 1) gemm_tc_kernel(GEMM_TC_PARAMS) {
  gemm_tc_body<A_KC, B_KC, false>(map_a, map_b, C, ldc, M, N, K, kt_per_split, ep, cluster_size, partial, b_const);
}
template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(NUM_THREADS, 1) gemm_tc1_kernel(GEMM_TC_PARAMS) {
  gemm_tc_body<A_KC, B_KC, true>(map_a, map_b, C, ldc, M, N, K, kt_per_split, ep, cluster_size, partial, b_const);
}
#undef GEMM_TC_PARAMS


// ---------------------------------------------------------------------------------------------------------------------------
// Persistent variant for problems with many output tiles and a short k-loop (the 16 000 .. 128 000-row layers of the protein
// configurations: K = 512 .. 1280).  With one tile per CTA the prologue (barriers, TMEM allocation, pipeline fill) and the
// epilogue (TMEM -> registers -> smem transpose -> global) cost more than the 16 k-steps of MMAs between them.  Here a CTA
// walks tiles b, b + G, ...; the operand ring runs across tile boundaries; the accumulators (small + big, 256 columns) are
// DOUBLE-BUFFERED in TMEM and four dedicated epilogue warps drain tile t while the tensor core works on tile t + 1.
// Warp roles: 0 TMA producer, 1 MMA issuer (owns TMEM), 2..5 epilogue (TMEM lane quarter = warp % 4), 6..13 lo pass.
// ---------------------------------------------------------------------------------------------------------------------------
constexpr int P_EPI_WARPS = 4, P_LO_WARPS = 8;
constexpr int P_THREADS = (2 + P_EPI_WARPS + P_LO_WARPS) * 32;
constexpr uint32_t P_SCRATCH_BYTES = P_EPI_WARPS * 32 * 33 * 4;
constexpr uint32_t P_SMEM_BYTES = STAGES * STAGE_BYTES + P_SCRATCH_BYTES + BAR_BYTES + 1024;
constexpr int P_MAX_KT = 40;          // one big accumulator per tile: chain length bounded like the round-1 kernel (K <= 1280)

template <bool A_KC, bool B_KC, bool ONE>
__device__ __forceinline__ void gemm_tc_persistent_body(const CUtensorMap& map_a, const CUtensorMap& map_b, float* __restrict__ C,
                                                        int64_t ldc, int64_t M, int64_t N, int64_t K, const Ep& ep, int tiles_n,
                                                        int n_tiles) {
  constexpr int STAGES = Ring<ONE>::STAGES;
  constexpr uint32_t STAGE_BYTES = Ring<ONE>::STAGE_BYTES;
  CGVAE_KERNEL_PROLOGUE();
  extern __shared__ __align__(1024) char smem_raw[];
  char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* scratch = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
  uint64_t* raw_full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + P_SCRATCH_BYTES);
  uint64_t* lo_done = raw_full + STAGES;
  uint64_t* empty_bar = lo_done + STAGES;
  uint64_t* acc_full = empty_bar + STAGES;     // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]
  uint32_t* tmem_ptr_sh = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int num_kt = (int)((K + BK - 1) / BK);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&raw_full[s], 1);
      mbar_init(&lo_done[s], P_LO_WARPS);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], P_EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<TMEM_COLS>(tmem_ptr_sh);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_sh;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BN;
      for (int kt = 0; kt < num_kt; ++kt, ++it) {
        const int s = it % STAGES;
        mbar_wait(&empty_bar[s], ((uint32_t)(it / STAGES) & 1u) ^ 1u);
        if (elect_one()) {
          const int k0 = kt * BK;
          const uint32_t a_dst = smem_base + (uint32_t)s * STAGE_BYTES, b_dst = a_dst + A_BYTES;
          mbar_expect_tx(&raw_full[s], RAW_BYTES);
          if (A_KC) {
            tma_2d(a_dst, &map_a, k0, m0, &raw_full[s]);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 32; ++j) tma_2d(a_dst + (uint32_t)j * 4096u, &map_a, m0 + 32 * j, k0, &raw_full[s]);
          }
          if (B_KC) {
            tma_2d(b_dst, &map_b, k0, n0, &raw_full[s]);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 32; ++j) tma_2d(b_dst + (uint32_t)j * 4096u, &map_b, n0 + 32 * j, k0, &raw_full[s]);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc = idesc_tf32(BM, BN, !A_KC, !B_KC);
    constexpr uint32_t a_step = A_KC ? 32u : 1024u, b_step = B_KC ? 32u : 1024u;
    int it = 0, tcount = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const int buf = tcount & 1;
      mbar_wait(&acc_empty[buf], ((uint32_t)(tcount >> 1) & 1u) ^ 1u);      // the epilogue has drained this accumulator set
      tc_fence_after();
      const uint32_t d_small = tmem_base + (uint32_t)buf * 2u * BN, d_big = d_small + BN;
      for (int kt = 0; kt < num_kt; ++kt, ++it) {
        const int s = it % STAGES;
        mbar_wait(&lo_done[s], (uint32_t)(it / STAGES) & 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_hi = smem_base + (uint32_t)s * STAGE_BYTES, b_hi = a_hi + A_BYTES;
          const uint32_t a_lo = a_hi + RAW_BYTES, b_lo = b_hi + RAW_BYTES;
#pragma unroll
          for (int ks = 0; ks < BK / 8; ++ks) {
            const uint32_t ao = (uint32_t)ks * a_step, bo = (uint32_t)ks * b_step;
            const uint32_t acc = (kt > 0 || ks > 0) ? 1u : 0u;
            if constexpr (ONE) {
              umma_tf32_ss(d_small, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_hi + bo), acc, idesc);   // one accumulator
            } else {
              umma_tf32_ss(d_small, make_desc_op<A_KC>(a_lo + ao), make_desc_op<B_KC>(b_hi + bo), acc, idesc);
              umma_tf32_ss(d_small, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_lo + bo), 1u, idesc);
              umma_tf32_ss(d_big, make_desc_op<A_KC>(a_hi + ao), make_desc_op<B_KC>(b_hi + bo), acc, idesc);
            }
          }
          umma_commit(&empty_bar[s]);
          if (kt == num_kt - 1) umma_commit(&acc_full[buf]);
        }
        __syncwarp();
      }
    }
  } else if (warp < 2 + P_EPI_WARPS) {
    // ---------------- epilogue: TMEM -> registers -> smem transpose -> coalesced global stores ----------------
    const int q = warp & 3;                                   // TMEM lane quarter this warp may access
    const int mode = ep_mode(ep);
    float* tr = scratch + (warp - 2) * (32 * 33);
    int tcount = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const int buf = tcount & 1;
      const int64_t m0 = (int64_t)(tile / tiles_n) * BM, n0 = (int64_t)(tile % tiles_n) * BN;
      mbar_wait(&acc_full[buf], (uint32_t)(tcount >> 1) & 1u);
      tc_fence_after();
      const uint32_t t_small = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)buf * 2u * BN;
#pragma unroll 1
      for (int cb = 0; cb < BN / 32; ++cb) {
        uint32_t r[32], t[32];
        tmem_ld32(t_small + (uint32_t)cb * 32u, r);
        if constexpr (!ONE) tmem_ld32(t_small + BN + (uint32_t)cb * 32u, t);
        tmem_wait_ld();
        if (cb == BN / 32 - 1) {                              // everything of this set is in registers: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) tr[lane * 33 + j] = ONE ? __uint_as_float(r[j]) : __uint_as_float(r[j]) + __uint_as_float(t[j]);
        __syncwarp();
        if (m0 + 32 * q < M) store_block(mode, ep, tr, lane, C, ldc, m0 + 32 * q, n0 + cb * 32 + lane, M, N);
        __syncwarp();
      }
    }
  } else {
    // ---------------- lo pass ----------------
    const int t0 = tid - (2 + P_EPI_WARPS) * 32;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int kt = 0; kt < num_kt; ++kt, ++it) {
        const int s = it % STAGES;
        mbar_wait(&raw_full[s], (uint32_t)(it / STAGES) & 1u);
        split_stage<ONE, P_LO_WARPS * 32>(smem + (uint32_t)s * STAGE_BYTES, t0);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&lo_done[s]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

#define GEMM_TC_P_PARAMS                                                                                                        \
  const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, float* __restrict__ C, int64_t ldc,    \
      int64_t M, int64_t N, int64_t K, Ep ep, int tiles_n, int n_tiles
template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(P_THREADS, 1) gemm_tc_persistent_kernel(GEMM_TC_P_PARAMS) {
  gemm_tc_persistent_body<A_KC, B_KC, false>(map_a, map_b, C, ldc, M, N, K, ep, tiles_n, n_tiles);
}
template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(P_THREADS, 1) gemm_tc1_persistent_kernel(GEMM_TC_P_PARAMS) {
  gemm_tc_persistent_body<A_KC, B_KC, true>(map_a, map_b, C, ldc, M, N, K, ep, tiles_n, n_tiles);
}
#undef GEMM_TC_P_PARAMS

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
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

// 2-D fp32 map: inner (contiguous) extent `inner`, outer extent `outer` with row pitch ld; box [box_outer][32]
static bool encode_map(CUtensorMap* map, const float* base, int64_t inner, int64_t outer, int64_t ld, int box_outer, bool kc) {
  EncodeTiledFn encode = encode_fn();
  if (encode == nullptr) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {32u, (cuuint32_t)box_outer};
  const cuuint32_t estride[2] = {1, 1};
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estride,
                CU_TENSOR_MAP_INTERLEAVE_NONE, kc ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tc

// returns 1 when the problem was launched on the tensor-core path, 0 when the caller should use the SIMT kernel
int launch_gemm_tcgen05(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                        int64_t N, int64_t K, const float* bias, int act, float* z_out, const float* z_in, int dact,
                        const float* add, float* ws, size_t ws_bytes, cudaStream_t st) {
  if (M < tc::MIN_M || N < 64 || K < 32) return 0;
  // TMA: 16-byte aligned bases and row pitches
  if (!aligned16(A) || !aligned16(B) || (lda % 4) != 0 || (ldb % 4) != 0) return 0;
  const bool a_kc = (form != CGVAE_GEMM_TN), b_kc = (form == CGVAE_GEMM_NT);
  const int64_t tiles = ceil_div(M, tc::BM) * ceil_div(N, tc::BN);
  const int num_kt = (int)ceil_div(K, tc::BK);
  // split K over a cluster when the tiles leave SMs idle (>= 2 k-steps per CTA), and always enough to keep one TMEM
  // accumulation chain <= MAX_KT_PER_CTA k-steps
  int S = (int)std::min<int64_t>(8, std::max<int64_t>(1, kNumSM / tiles));
  S = std::min(S, std::max(1, num_kt / 2));
  S = std::max(S, (int)ceil_div(num_kt, tc::MAX_KT_PER_CTA));
  int groups = 1;
  if (S > 8) {
    // longer reductions (weight gradients over 1e4 .. 1e5 node rows): several clusters, one raw partial matrix each
    groups = (int)ceil_div(S, 8);
    if (ws == nullptr || (size_t)groups * (size_t)(M * N) * sizeof(float) > ws_bytes) return 0;
    S = 8;
  }
  const int kps = (int)ceil_div(num_kt, S * groups);
  if (groups == 1) S = (int)ceil_div(num_kt, kps);
  CUtensorMap map_a, map_b;
  // K-contiguous operand: inner = K, outer = rows, box [128 rows][32 k]; MN-contiguous: inner = rows, outer = K, box [32 k][32 mn]
  if (!(a_kc ? tc::encode_map(&map_a, A, K, M, lda, tc::BM, true) : tc::encode_map(&map_a, A, M, K, lda, tc::BK, false))) return 0;
  if (!(b_kc ? tc::encode_map(&map_b, B, K, N, ldb, tc::BN, true) : tc::encode_map(&map_b, B, N, K, ldb, tc::BK, false))) return 0;
  const int b_const = (form != CGVAE_GEMM_TN &&
                       weights_are_constant(B, sizeof(float) * (size_t)(((b_kc ? N : K) - 1) * ldb + (b_kc ? K : N)))) ? 1 : 0;
  tc::Ep ep{bias, act, z_out, z_in, dact, add};
  // the precision mode picks the kernel only: S, groups, persistent eligibility and grid are those of the 3xTF32 kernels
  const bool one = matmul_precision() == 1;
  if (S == 1 && groups == 1 && tiles >= 2 * kNumSM && num_kt <= tc::P_MAX_KT) {
    const dim3 grid((unsigned)std::min<int64_t>(tiles, kNumSM));
    const int tiles_n = (int)ceil_div(N, tc::BN), n_tiles = (int)tiles;
    static bool p_attr_done[6] = {false, false, false, false, false, false};
    auto pgo = [&](auto kernel, int idx) {
      if (!p_attr_done[idx]) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::P_SMEM_BYTES);
        p_attr_done[idx] = true;
      }
      launch_kernel(kernel, grid, dim3(tc::P_THREADS), tc::P_SMEM_BYTES, st, map_a, map_b, C, ldc, M, N, K, ep, tiles_n, n_tiles);
    };
    if (one) {
      if (a_kc && b_kc) pgo(tc::gemm_tc1_persistent_kernel<true, true>, 3);
      else if (a_kc) pgo(tc::gemm_tc1_persistent_kernel<true, false>, 4);
      else pgo(tc::gemm_tc1_persistent_kernel<false, false>, 5);
    } else {
      if (a_kc && b_kc) pgo(tc::gemm_tc_persistent_kernel<true, true>, 0);
      else if (a_kc) pgo(tc::gemm_tc_persistent_kernel<true, false>, 1);
      else pgo(tc::gemm_tc_persistent_kernel<false, false>, 2);
    }
    return 1;
  }
  if (groups > 1) ep = tc::Ep{nullptr, 0, nullptr, nullptr, 0, nullptr};
  float* partial = groups > 1 ? ws : nullptr;
  const dim3 grid((unsigned)ceil_div(N, tc::BN), (unsigned)ceil_div(M, tc::BM), (unsigned)(S * groups)), cluster(1, 1, (unsigned)S);
  static bool attr_done[6] = {false, false, false, false, false, false};
  auto go = [&](auto kernel, int idx) {
    if (!attr_done[idx]) {
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES);
      attr_done[idx] = true;
    }
    launch_cluster(kernel, grid, dim3(tc::NUM_THREADS), cluster, tc::SMEM_BYTES, st, map_a, map_b, C, ldc, M, N, K, kps, ep, S, partial,
                   b_const);
  };
  if (one) {
    if (a_kc && b_kc) go(tc::gemm_tc1_kernel<true, true>, 3);
    else if (a_kc) go(tc::gemm_tc1_kernel<true, false>, 4);
    else go(tc::gemm_tc1_kernel<false, false>, 5);
  } else {
    if (a_kc && b_kc) go(tc::gemm_tc_kernel<true, true>, 0);
    else if (a_kc) go(tc::gemm_tc_kernel<true, false>, 1);
    else go(tc::gemm_tc_kernel<false, false>, 2);
  }
  return groups > 1 ? 1 + groups : 1;          // > 1: the caller reduces `groups` partial matrices in ws
}

}  // namespace cgvae
