// Fused message layers on the 5th-generation tensor cores (EquiMessageBlock conv.py:505-563, EquiMessageCross
// conv.py:358-402 and their autograd).
//
// The edge filter  w_k[e][f] = sum_r basis[e][r] * Wf'[k][f][r]   (DistanceEmbed, modules.py:192-197: rbf @ W_filter +
// bias, times the envelope -- the bias rides as the basis column that holds the envelope) is the dense contraction of
// the layer.  Here it is a 3xTF32 tcgen05.mma per batch of 32 edge columns:
//      D_k[128 channels x 32 columns] = Wf'_k[128 x 16] * basis^T[16 x 32]          (accumulators in TMEM)
// with channels on the TMEM lanes, so that the thread that owns channel f reads w_k[.][f] of 32 edges with tcgen05.ld
// and keeps its gathers coalesced (a warp = 32 consecutive channels of one sender row) and its receiver sums in registers.
//
// Column tiles.  Edges are re-ordered into COLUMN TILES: a chunk of RC consecutive receivers x the sorted union of their
// senders.  Column (g, rr) = edge (receiver chunk*RC + rr  <-  sender gcol[g]); pairs that are not edges keep an all-zero
// basis row, so their filter value is exactly 0.  The thread gathers the six sender values (phi_0..2, v_x..z) ONCE per
// group and re-uses them from registers for the RC receivers of the chunk -- on the molecule graphs (chignolin: degree
// 159 of 175) that is ~7x fewer gathers than one gather set per edge, which is what the SIMT kernel of message.cu is
// bound by (26 % address arithmetic, 62 % issue utilisation, profiles/r1b_message_kernels_hotspots.txt).
// A batch record (32 columns: both tf32 halves of the basis tile in the canonical K-major core-matrix layout, unit
// vectors, sender ids) is ONE 4.6 KB cp.async.bulk; records are produced once per graph (cgvae_msg_tiles_build) and
// shared by every layer that runs on that graph.
//
// Warp roles (192 threads): warps 0-3 = 128 channel threads (gather, tcgen05.ld, mix, reduce), warp 4 lane 0 = bulk-copy
// producer (4-stage mbarrier ring), warp 5 lane 0 = MMA issuer (+ TMEM allocation: 2 accumulator buffers).
// Two CTAs per SM (256 TMEM columns, <= 84 KB shared memory each).
//
// Backward: the same structure on the transposed tiles (chunk of RC SENDERS x union of their receivers); the filter
// gradient dWf'_k[f][r] = sum_cols G_k[f][col] * basis[col][r] is a second tcgen05.mma whose A operand G_k (produced by
// the channel threads) is written to TMEM with tcgen05.st and whose B operand is the SAME shared-memory basis tile read
// MN-major.
#include "tc_common.cuh"

namespace cgvae {
namespace mtc {

using namespace tcx;

constexpr int NB = 64;                 // columns per batch = MMA N
constexpr int KT = 16;                 // padded filter K (R + 1 <= 16)
constexpr uint32_t TILE_SBO = (KT / 4) * kLBO;   // 512
constexpr int REC_BHI = 0;             // [NB x 16] tf32 hi, canonical layout (4096 B)
constexpr int REC_BLO = NB * KT * 4;   // [NB x 16] tf32 lo
constexpr int REC_UNIT = 2 * NB * KT * 4;          // unit vectors, component-major: ux[NB] uy[NB] uz[NB]
constexpr int REC_GCOL = REC_UNIT + 3 * NB * 4;    // partner (sender) index of each group of the batch: NB / RC <= 16 ints
constexpr int REC_BYTES = ((REC_GCOL + (NB / 4) * 4 + 127) / 128) * 128;   // 9088

// ------------------------------------------------------------------------------------------------------------------
// tile builder (integer work, exact, deterministic)
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTileThreads = 256;

// shared: bitmap[W] | seg_pref[kTileThreads + 1]
__device__ __forceinline__ int build_bitmap(uint32_t* bm, int W, const int32_t* __restrict__ col, int e0, int e1) {
  for (int w = threadIdx.x; w < W; w += kTileThreads) bm[w] = 0u;
  __syncthreads();
  for (int e = e0 + threadIdx.x; e < e1; e += kTileThreads) {
    const int j = col[e];
    atomicOr(&bm[j >> 5], 1u << (j & 31));
  }
  __syncthreads();
  const int SEG = (W + kTileThreads - 1) / kTileThreads;
  int cnt = 0;
  const int w0 = threadIdx.x * SEG, w1 = min(W, w0 + SEG);
  for (int w = w0; w < w1; ++w) cnt += __popc(bm[w]);
  return cnt;
}

// exclusive scan of one int per thread over the block into pref[0 .. kTileThreads] (pref[kTileThreads] = total)
__device__ __forceinline__ void block_scan(int v, int* pref) {
  __shared__ int warp_tot[kTileThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_tot[warp] = x;
  __syncthreads();
  int base = 0;
  for (int w = 0; w < warp; ++w) base += warp_tot[w];
  pref[threadIdx.x] = base + x - v;
  if (threadIdx.x == kTileThreads - 1) pref[kTileThreads] = base + x;
  __syncthreads();
}

__global__ void __launch_bounds__(kTileThreads) tile_count_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                                 int64_t n_rows, int64_t n_partners, int RC,
                                                                 int32_t* __restrict__ nbatch, int32_t* __restrict__ ngroups) {
  CGVAE_KERNEL_PROLOGUE();
  extern __shared__ uint32_t tile_sm[];
  const int W = (int)((n_partners + 31) / 32);
  uint32_t* bm = tile_sm;
  int* pref = reinterpret_cast<int*>(tile_sm + W);
  const int64_t r0 = (int64_t)blockIdx.x * RC, r1 = min(n_rows, r0 + RC);
  const int cnt = build_bitmap(bm, W, col, rowptr[r0], rowptr[r1]);
  block_scan(cnt, pref);
  if (threadIdx.x == 0) {
    const int ng = pref[kTileThreads], GB = NB / RC;
    ngroups[blockIdx.x] = ng;
    nbatch[blockIdx.x] = (ng + GB - 1) / GB;
  }
}

__global__ void __launch_bounds__(kTileThreads) tile_fill_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                                const int32_t* __restrict__ slot_map, int64_t n_rows,
                                                                int64_t n_partners, int RC, const int32_t* __restrict__ bptr,
                                                                const float* __restrict__ basis, const float* __restrict__ unit,
                                                                int RB, char* __restrict__ rec, int64_t n_batches_cap) {
  CGVAE_KERNEL_PROLOGUE();
  extern __shared__ uint32_t tile_sm[];
  const int W = (int)((n_partners + 31) / 32);
  uint32_t* bm = tile_sm;
  int* pref = reinterpret_cast<int*>(tile_sm + W);
  const int64_t r0 = (int64_t)blockIdx.x * RC, r1 = min(n_rows, r0 + RC);
  const int cnt = build_bitmap(bm, W, col, rowptr[r0], rowptr[r1]);
  block_scan(cnt, pref);
  const int SEG = (W + kTileThreads - 1) / kTileThreads;
  const int GB = NB / RC;
  const int64_t b0 = bptr[blockIdx.x];
  // sender id of every group (sorted ascending: bit order)
  {
    int g = pref[threadIdx.x];
    const int w0 = threadIdx.x * SEG, w1 = min(W, w0 + SEG);
    for (int w = w0; w < w1; ++w) {
      uint32_t bits = bm[w];
      while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const int64_t batch = b0 + g / GB;
        if (batch < n_batches_cap)
          reinterpret_cast<int32_t*>(rec + batch * REC_BYTES + REC_GCOL)[g % GB] = w * 32 + b;
        ++g;
      }
    }
  }
  // every edge of the chunk -> its column
  const int RBQ = RB / 4;
  for (int64_t i = r0; i < r1; ++i) {
    const int rr = (int)(i - r0);
    for (int e = rowptr[i] + threadIdx.x; e < rowptr[i + 1]; e += kTileThreads) {
      const int j = col[e];
      const int w = j >> 5, seg = w / SEG;
      int g = pref[seg];
      for (int ww = seg * SEG; ww < w; ++ww) g += __popc(bm[ww]);
      g += __popc(bm[w] & ((1u << (j & 31)) - 1u));
      const int64_t batch = b0 + g / GB;
      if (batch >= n_batches_cap) continue;
      const int c = (g % GB) * RC + rr;                  // column inside the batch
      char* r = rec + batch * REC_BYTES;
      const int64_t src = slot_map ? slot_map[e] : e;
      const float4* brow = reinterpret_cast<const float4*>(basis) + src * RBQ;
      for (int q = 0; q < RBQ; ++q) {
        const float4 x = __ldg(brow + q);
        float4 h, l;
        split_tf32(x.x, h.x, l.x);
        split_tf32(x.y, h.y, l.y);
        split_tf32(x.z, h.z, l.z);
        split_tf32(x.w, h.w, l.w);
        const uint32_t off = tile_off(c, 4 * q, TILE_SBO);
        *reinterpret_cast<float4*>(r + REC_BHI + off) = h;
        *reinterpret_cast<float4*>(r + REC_BLO + off) = l;
      }
      const float4 u = __ldg(reinterpret_cast<const float4*>(unit) + src);
      float* un = reinterpret_cast<float*>(r + REC_UNIT);
      un[c] = u.x;
      un[NB + c] = u.y;
      un[2 * NB + c] = u.z;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------------
// One persistent CTA per SM.  Work items = (128-channel slice, receiver chunk), slice-major; CTA b owns the contiguous
// item range [b * n_items / G, (b + 1) * n_items / G).  Warps: 4 lane quarters x NSUB consumer warps (thread = channel,
// the NSUB warps of a quarter take the groups of a batch round-robin and merge their partial receiver sums through shared
// memory in a fixed order), + 1 bulk-copy producer warp, + 1 MMA / TMEM-allocator warp.
// TMEM (512 columns): filter operand A = Wf' of the slice, both tf32 halves [KS][2][16 columns] (written by the channel
// threads with tcgen05.st: the MMA reads it from TMEM, so the only shared-memory operand traffic is the basis tile);
// accumulators D[buf][k][NB columns], double buffered for 3 splits.
// Measured on B200 while shaping this kernel (tools/tc_latency.cu, profiles/r2_*): a tcgen05.mma costs ~60 + N/2 cycles
// to issue whatever it computes, so the batch is as wide as TMEM allows (18 MMAs per 64 columns), and every
// instruction the channel threads execute per batch besides the ~9 FMAs per column (barrier addressing, gather
// addressing) is amortised over 16 columns per warp.
constexpr int NSTAGE = 6;
constexpr int TMEM_COLS = 512;

template <int KS>
struct Cols {
  static constexpr int NDBUF = (KS == 3) ? 2 : 1;        // accumulator buffers (4 splits: one buffer fits)
  static constexpr uint32_t A = 0;                       // [KS][hi | lo][KT]
  static constexpr uint32_t D = KS * 2 * KT;             // [NDBUF][KS][NB]
  static_assert(D + NDBUF * KS * NB <= TMEM_COLS, "TMEM budget");
};

// shared-memory map (byte offsets from the dynamic shared base; barriers addressed as u32 shared addresses)
template <int NSUB, int NACC>
struct Map {
  static constexpr uint32_t STAGES = 0;
  static constexpr uint32_t BARS = NSTAGE * REC_BYTES;
  static constexpr uint32_t STAGE_FULL = BARS;                    // [NSTAGE]  bulk copy landed
  static constexpr uint32_t STAGE_EMPTY = BARS + 8 * NSTAGE;      // [NSTAGE]  every consumer warp is done with the record
  static constexpr uint32_t D_FULL = BARS + 16 * NSTAGE;          // [2]       filter MMAs of the batch complete
  static constexpr uint32_t D_EMPTY = D_FULL + 16;                // [2]       every consumer warp has read its columns
  static constexpr uint32_t A_FULL = D_EMPTY + 16;                // filter operand of the current slice staged in TMEM
  static constexpr uint32_t TMEM_PTR = A_FULL + 8;
  static constexpr uint32_t XCHG = ((TMEM_PTR + 8 + 127) / 128) * 128;     // [NSUB - 1][NACC][128] floats
  static constexpr uint32_t BYTES = XCHG + (NSUB > 1 ? (NSUB - 1) * NACC * 128 * 4 : 0) + 64;
};

__device__ __forceinline__ void bar_wait(uint32_t bar_addr, uint32_t parity) {
  uint32_t done = 0;
#pragma unroll 1
  for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar_addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  asm volatile("trap;");
}
__device__ __forceinline__ void bar_arrive(uint32_t bar_addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}
__device__ __forceinline__ void bar_expect_tx(uint32_t bar_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_init(uint32_t bar_addr, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_addr), "r"(count));
}
__device__ __forceinline__ void bulk_g2s_a(uint32_t dst_addr, const void* src, uint32_t bytes, uint32_t bar_addr) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_addr), "l"(src),
               "r"(bytes), "r"(bar_addr)
               : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar_addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
}

// filter MMAs of one batch: D_k = A_k[tmem] * B^T[smem] for every split, 3xTF32 (small terms first), K = 16 in two steps.
// ONE (1xTF32, cgvae_set_matmul_precision(1)): the hi * hi product only -- both hi halves are already rounded to nearest
template <int KS, bool ONE>
__device__ __forceinline__ void issue_filter_mmas(uint32_t stage_addr, uint32_t tmem_base, uint32_t d_col) {
  constexpr uint32_t idesc = idesc_tf32(128, NB);
  const uint64_t b_hi = make_desc(stage_addr + REC_BHI, kLBO, TILE_SBO);
  [[maybe_unused]] const uint64_t b_lo = b_hi + (uint64_t)((REC_BLO - REC_BHI) >> 4);
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    const uint32_t a_hi = tmem_base + Cols<KS>::A + (uint32_t)(k * 2 * KT);
    [[maybe_unused]] const uint32_t a_lo = a_hi + KT;
    const uint32_t d = tmem_base + d_col + (uint32_t)(k * NB);
#pragma unroll
    for (int ks = 0; ks < KT / 8; ++ks) {
      const uint32_t ao = (uint32_t)ks * 8;
      const uint64_t bo = (uint64_t)((ks * 2 * kLBO) >> 4);
      if constexpr (ONE) {
        umma_tf32_ts(d, a_hi + ao, b_hi + bo, ks > 0 ? 1u : 0u, idesc);
      } else {
        umma_tf32_ts(d, a_lo + ao, b_hi + bo, ks > 0 ? 1u : 0u, idesc);
        umma_tf32_ts(d, a_hi + ao, b_lo + bo, 1u, idesc);
        umma_tf32_ts(d, a_hi + ao, b_hi + bo, 1u, idesc);
      }
    }
  }
}

// the thread that owns channel f0 + row writes its rows of Wf'_k = [Wf[(k*F + f)*R + r] (r < R) | bf[k*F + f] | 0 ...] into
// the TMEM operand region, both tf32 halves
template <int KS>
__device__ __forceinline__ void stage_filter_tmem(uint32_t t_lane, const float* __restrict__ Wf, const float* __restrict__ bf, int F,
                                                  int R, int ch) {
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    uint32_t hi[KT], lo[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) {
      float val = 0.f;
      if (ch < F) {
        if (r < R) val = __ldg(Wf + ((int64_t)k * F + ch) * R + r);
        else if (r == R) val = __ldg(bf + (int64_t)k * F + ch);
      }
      float h, l;
      split_tf32(val, h, l);
      hi[r] = __float_as_uint(h);
      lo[r] = __float_as_uint(l);
    }
    tmem_st16(t_lane + Cols<KS>::A + (uint32_t)(k * 2 * KT), hi);
    tmem_st16(t_lane + Cols<KS>::A + (uint32_t)(k * 2 * KT + KT), lo);
  }
  tmem_wait_st();
}

// Work partition.  The batches of all work items (slice-major, then chunk) form one sequence of n_slices * TB batches
// (TB = bptr[n_chunks]); CTA b owns the contiguous range [b * T / G, (b + 1) * T / G) -- equal work per SM whatever the item
// sizes (with whole items per CTA the chignolin layer ran 220 equal items on 148 SMs: 2 rounds, 46 % idle).  An item cut by
// a range boundary is finished by the LAST of its CTAs to arrive (ticket), which adds the partial sums of the others in CTA
// order: deterministic.  Every role of the CTA walks the same segments with this helper.
struct Segment {
  int item, slice, chunk;
  int b0, nb;          // first batch of the segment inside its item, number of batches
  int item_nb;         // batches of the whole item
};
__device__ __forceinline__ int chunk_of_batch(const int32_t* __restrict__ bptr, int n_chunks, int r) {
  int lo = 0, hi = n_chunks;           // largest c with bptr[c] <= r  (empty chunks are skipped: bptr[c] == bptr[c+1])
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (bptr[mid] <= r) lo = mid; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ bool next_segment(const int32_t* __restrict__ bptr, int n_chunks, int TB, int64_t& x, int64_t x1, Segment& sg) {
  if (x >= x1) return false;
  sg.slice = (int)(x / TB);
  const int r = (int)(x - (int64_t)sg.slice * TB);
  sg.chunk = chunk_of_batch(bptr, n_chunks, r);
  const int c0 = bptr[sg.chunk], c1 = bptr[sg.chunk + 1];
  sg.item = sg.slice * n_chunks + sg.chunk;
  sg.item_nb = c1 - c0;
  sg.b0 = r - c0;
  const int64_t item_end = (int64_t)sg.slice * TB + c1;
  sg.nb = (int)(min(x1, item_end) - x);
  x += sg.nb;
  return true;
}
// CTA that owns global batch x under the partition lo_b = b * T / G
__device__ __forceinline__ int cta_of_batch(int64_t x, int64_t T, int G) { return (int)(((x + 1) * G - 1) / T); }

#define MESSAGE_TC_FWD_PARAMS                                                                                              \
  const float* __restrict__ phi, const float* __restrict__ v_send, const float* __restrict__ v_recv,                        \
      const int32_t* __restrict__ bptr, const int32_t* __restrict__ ngroups, const char* __restrict__ rec,                  \
      const float* __restrict__ Wf, const float* __restrict__ bf, int64_t n_recv, int F, int R,                             \
      const float* __restrict__ res_s, const float* __restrict__ res_v, int v_is_zero, float* __restrict__ out_s,           \
      float* __restrict__ out_v, float* __restrict__ q_out, int n_chunks, int n_items, int32_t* __restrict__ tickets,       \
      float* __restrict__ part_ws
#define MESSAGE_TC_FWD_ARGS                                                                                                \
  phi, v_send, v_recv, bptr, ngroups, rec, Wf, bf, n_recv, F, R, res_s, res_v, v_is_zero, out_s, out_v, q_out, n_chunks,    \
      n_items, tickets, part_ws

template <int KS, int RC, int NSUB, bool ONE>
__device__ __forceinline__ void message_tc_fwd_body(MESSAGE_TC_FWD_PARAMS) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int GB = NB / RC;                  // groups per batch
  constexpr int GPW = GB / NSUB;               // groups per consumer warp and batch
  static_assert(GB % NSUB == 0 && GPW >= 1, "groups of a batch must divide over the sub-warps");
  constexpr int NQ = (KS == 4) ? 3 : 0;
  constexpr int NACC = RC * (4 + NQ);          // per-thread accumulators: s, v[3] (, q[3]) per receiver of the chunk
  constexpr int NCONS = 4 * NSUB;              // consumer warps
  constexpr int NDBUF = Cols<KS>::NDBUF;
  using M = Map<NSUB, NACC>;
  extern __shared__ __align__(1024) char smem_raw[];
  const uint32_t sbase = smem_u32(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int TB = bptr[n_chunks];                              // batches per slice
  const int64_t T = (int64_t)TB * (n_items / n_chunks);       // all batches
  // the grid is sized from the static record capacity; with fewer live batches than CTAs the surplus CTAs leave at once, so
  // that every remaining CTA owns at least one batch and an item's CTAs are consecutive
  const int G = (int)max((int64_t)1, min((int64_t)gridDim.x, T));
  if ((int)blockIdx.x >= G) return;
  const int64_t x_lo = ((int64_t)blockIdx.x * T) / G, x_hi = ((int64_t)(blockIdx.x + 1) * T) / G;

  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      bar_init(sbase + M::STAGE_FULL + 8 * s, 1);
      bar_init(sbase + M::STAGE_EMPTY + 8 * s, NCONS);
    }
    for (int b = 0; b < 2; ++b) {
      bar_init(sbase + M::D_FULL + 8 * b, 1);
      bar_init(sbase + M::D_EMPTY + 8 * b, NCONS);
    }
    bar_init(sbase + M::A_FULL, 4);
    mbar_fence_init();
  }
  if (warp == NCONS + 1) tmem_alloc<TMEM_COLS>(reinterpret_cast<uint32_t*>(smem_raw + M::TMEM_PTR));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<const uint32_t*>(smem_raw + M::TMEM_PTR);

  if (warp == NCONS) {
    // ---------------- bulk-copy producer (whole warp in the loop, one elected lane issues: see elect_one) ----------------
    uint32_t bc = 0;
    Segment sg;
    for (int64_t x = x_lo; next_segment(bptr, n_chunks, TB, x, x_hi, sg);) {
      const int nb = sg.nb;
      const char* src = rec + (int64_t)(bptr[sg.chunk] + sg.b0) * REC_BYTES;
      for (int b = 0; b < nb; ++b, ++bc) {
        const uint32_t s = bc % NSTAGE;
        bar_wait(sbase + M::STAGE_EMPTY + 8 * s, ((bc / NSTAGE) & 1u) ^ 1u);
        if (elect_one()) {
          bar_expect_tx(sbase + M::STAGE_FULL + 8 * s, REC_BYTES);
          bulk_g2s_a(sbase + M::STAGES + s * REC_BYTES, src + (int64_t)b * REC_BYTES, REC_BYTES, sbase + M::STAGE_FULL + 8 * s);
        }
        __syncwarp();
      }
    }
  } else if (warp == NCONS + 1) {
    // ---------------- MMA issuer (whole warp in the loop, one elected lane issues) ----------------
    uint32_t bc = 0, ac = 0;
    int staged_slice = -1;
    Segment sg;
    for (int64_t x = x_lo; next_segment(bptr, n_chunks, TB, x, x_hi, sg);) {
      const int nb = sg.nb, slice = sg.slice;
      if (slice != staged_slice) {
        bar_wait(sbase + M::A_FULL, ac & 1u);          // the channel threads have re-staged Wf' of the new slice
        ++ac;
        staged_slice = slice;
      }
      for (int b = 0; b < nb; ++b, ++bc) {
        const uint32_t s = bc % NSTAGE, buf = bc % NDBUF;
        bar_wait(sbase + M::STAGE_FULL + 8 * s, (bc / NSTAGE) & 1u);
        bar_wait(sbase + M::D_EMPTY + 8 * buf, ((bc / NDBUF) & 1u) ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          issue_filter_mmas<KS, ONE>(sbase + M::STAGES + s * REC_BYTES, tmem_base, Cols<KS>::D + buf * (KS * NB));
          umma_commit_a(sbase + M::D_FULL + 8 * buf);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- channel threads ----------------
    const int quarter = warp & 3, sub = warp >> 2;
    const int row = quarter * 32 + lane;                     // TMEM lane = channel inside the slice
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float* xchg = reinterpret_cast<float*>(smem_raw + M::XCHG);
    const uint32_t rowp = (uint32_t)(KS * F), rowv = (uint32_t)(3 * F);
    uint32_t bc = 0;
    int staged_slice = -1;
    // items without a single edge (isolated receivers): output = residual; spread over the CTAs
    if (sub == 0) {
      for (int item = blockIdx.x; item < n_items; item += G) {
        const int chunk = item % n_chunks, f = (item / n_chunks) * 128 + row;
        if (bptr[chunk + 1] != bptr[chunk] || f >= F) continue;
        for (int rr = 0; rr < RC; ++rr) {
          const int64_t i = (int64_t)chunk * RC + rr;
          if (i >= n_recv) break;
          const int64_t so = i * F + f, vo = i * 3 * F + f;
          out_s[so] = res_s ? res_s[so] : 0.f;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            out_v[vo + (int64_t)c * F] = res_v ? res_v[vo + (int64_t)c * F] : 0.f;
            if (KS == 4 && q_out) q_out[vo + (int64_t)c * F] = 0.f;
          }
        }
      }
    }
    Segment sg;
    bool first_seg = true;
    for (int64_t x = x_lo; next_segment(bptr, n_chunks, TB, x, x_hi, sg); first_seg = false) {
      const int chunk = sg.chunk, slice = sg.slice;
      const int nb = sg.nb, bo = sg.b0;             // batches of this segment, first batch inside the item
      const int ng = ngroups[chunk];
      const int f = slice * 128 + row;
      const bool active = f < F;
      const int fc = active ? f : F - 1;           // inactive lanes compute on a valid channel, never store
      const float* __restrict__ phi_f = phi + fc;
      const float* __restrict__ v_f = v_is_zero ? nullptr : v_send + fc;
      if (slice != staged_slice) {
        // all MMAs that read the previous operand are complete: this thread has consumed every batch of the last item
        if (sub == 0) {
          stage_filter_tmem<KS>(t_lane, Wf, bf, F, R, f);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) bar_arrive(sbase + M::A_FULL);
        }
        staged_slice = slice;
      }
      float acc_s[RC], acc_v[3][RC], acc_q[KS == 4 ? 3 : 1][RC];
#pragma unroll
      for (int rr = 0; rr < RC; ++rr) {
        acc_s[rr] = 0.f;
        acc_v[0][rr] = acc_v[1][rr] = acc_v[2][rr] = 0.f;
#pragma unroll
        for (int c = 0; c < (KS == 4 ? 3 : 1); ++c) acc_q[c][rr] = 0.f;
      }
      // gathers of this warp's groups of a batch: issued one batch ahead of their use
      float ph[GPW][KS], vv[GPW][3];
      auto gather = [&](uint32_t bcx, int b) {
        const uint32_t s = bcx % NSTAGE;
        bar_wait(sbase + M::STAGE_FULL + 8 * s, (bcx / NSTAGE) & 1u);
        const int32_t* gcol = reinterpret_cast<const int32_t*>(smem_raw + M::STAGES + s * REC_BYTES + REC_GCOL);
#pragma unroll
        for (int t = 0; t < GPW; ++t) {
          const int g = sub + t * NSUB;
          const bool live = (bo + b) * GB + g < ng;
          const uint32_t j = live ? (uint32_t)gcol[g] : 0u;
          const float* pj = phi_f + j * rowp;
#pragma unroll
          for (int k = 0; k < KS; ++k) ph[t][k] = live ? __ldg(pj + (uint32_t)k * (uint32_t)F) : 0.f;
          if (v_f != nullptr && live) {
            const float* vj = v_f + j * rowv;
            vv[t][0] = __ldg(vj); vv[t][1] = __ldg(vj + (uint32_t)F); vv[t][2] = __ldg(vj + 2u * (uint32_t)F);
          } else {
            vv[t][0] = vv[t][1] = vv[t][2] = 0.f;
          }
        }
      };
      if (nb > 0) gather(bc, 0);
      for (int b = 0; b < nb; ++b, ++bc) {
        const uint32_t s = bc % NSTAGE, buf = bc % NDBUF;
        float cph[GPW][KS], cvv[GPW][3];
#pragma unroll
        for (int t = 0; t < GPW; ++t) {
#pragma unroll
          for (int k = 0; k < KS; ++k) cph[t][k] = ph[t][k];
          cvv[t][0] = vv[t][0]; cvv[t][1] = vv[t][1]; cvv[t][2] = vv[t][2];
        }
        if (b + 1 < nb) gather(bc + 1, b + 1);       // next batch's sender rows: in flight during this batch's math
        const float* un = reinterpret_cast<const float*>(smem_raw + M::STAGES + s * REC_BYTES + REC_UNIT);
        bar_wait(sbase + M::D_FULL + 8 * buf, (bc / NDBUF) & 1u);
        tc_fence_after();
        const uint32_t t_buf = t_lane + Cols<KS>::D + buf * (KS * NB);
        // four columns (= four receivers of the chunk) at a time: filter values from TMEM, unit vectors from the record
#pragma unroll
        for (int t = 0; t < GPW; ++t) {
          const int g = sub + t * NSUB;
          const bool live = (bo + b) * GB + g < ng;
          const float p0 = cph[t][0] * cvv[t][0], p1 = cph[t][0] * cvv[t][1], p2 = cph[t][0] * cvv[t][2];
          float x0 = 0.f, x1 = 0.f, x2 = 0.f;
          if constexpr (KS == 4) {
            x0 = cph[t][3] * cvv[t][0]; x1 = cph[t][3] * cvv[t][1]; x2 = cph[t][3] * cvv[t][2];
          }
#pragma unroll
          for (int q4 = 0; q4 < RC / 4; ++q4) {
            const int c0 = g * RC + 4 * q4;
            uint32_t w[KS][4];
#pragma unroll
            for (int k = 0; k < KS; ++k) tmem_ld4(t_buf + (uint32_t)(k * NB + c0), w[k]);
            const float4 ux = *reinterpret_cast<const float4*>(un + c0);
            const float4 uy = *reinterpret_cast<const float4*>(un + NB + c0);
            const float4 uz = *reinterpret_cast<const float4*>(un + 2 * NB + c0);
            tmem_wait_ld();
            if (t == GPW - 1 && q4 == RC / 4 - 1) {
              // this warp's columns of the accumulator buffer and its part of the record are in registers: release both
              tc_fence_before();
              __syncwarp();
              if (lane == 0) {
                bar_arrive(sbase + M::D_EMPTY + 8 * buf);
                bar_arrive(sbase + M::STAGE_EMPTY + 8 * s);
              }
            }
            if (live) {
              const float uxa[4] = {ux.x, ux.y, ux.z, ux.w}, uya[4] = {uy.x, uy.y, uy.z, uy.w}, uza[4] = {uz.x, uz.y, uz.z, uz.w};
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const int rr = 4 * q4 + c;
                const float w0 = __uint_as_float(w[0][c]), w1 = __uint_as_float(w[1][c]), w2 = __uint_as_float(w[2][c]);
                acc_s[rr] = fmaf(cph[t][1], w1, acc_s[rr]);                    // dS_i += m1            (conv.py:526,558)
                const float m2 = cph[t][2] * w2;
                acc_v[0][rr] = fmaf(m2, uxa[c], acc_v[0][rr]);                 // dV_i += m2 * u_ij     (conv.py:524)
                acc_v[1][rr] = fmaf(m2, uya[c], acc_v[1][rr]);
                acc_v[2][rr] = fmaf(m2, uza[c], acc_v[2][rr]);
                acc_v[0][rr] = fmaf(w0, p0, acc_v[0][rr]);                     //        + m0 * v_j     (conv.py:525)
                acc_v[1][rr] = fmaf(w0, p1, acc_v[1][rr]);
                acc_v[2][rr] = fmaf(w0, p2, acc_v[2][rr]);
                if constexpr (KS == 4) {
                  const float w3 = __uint_as_float(w[3][c]);                   // q_i = sum m3 * v_j    (conv.py:379)
                  acc_q[0][rr] = fmaf(w3, x0, acc_q[0][rr]);
                  acc_q[1][rr] = fmaf(w3, x1, acc_q[1][rr]);
                  acc_q[2][rr] = fmaf(w3, x2, acc_q[2][rr]);
                }
              }
            }
          }
        }
      }
      // ---------------- merge the sub-warps (fixed order) and store: single store per output element ----------------
      if constexpr (NSUB > 1) {
        if (sub > 0) {
          float* dst = xchg + (size_t)(sub - 1) * NACC * 128 + row;
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) {
            dst[(rr * (4 + NQ) + 0) * 128] = acc_s[rr];
            dst[(rr * (4 + NQ) + 1) * 128] = acc_v[0][rr];
            dst[(rr * (4 + NQ) + 2) * 128] = acc_v[1][rr];
            dst[(rr * (4 + NQ) + 3) * 128] = acc_v[2][rr];
            if constexpr (KS == 4) {
              dst[(rr * 7 + 4) * 128] = acc_q[0][rr];
              dst[(rr * 7 + 5) * 128] = acc_q[1][rr];
              dst[(rr * 7 + 6) * 128] = acc_q[2][rr];
            }
          }
        }
        named_bar_sync(1, NCONS * 32);
      }
      if (sub == 0) {
        // merged sums of this CTA's segment, in registers: tot[rr][0..3(+3)]
        float tot[RC][4 + NQ];
#pragma unroll
        for (int rr = 0; rr < RC; ++rr) {
          tot[rr][0] = acc_s[rr]; tot[rr][1] = acc_v[0][rr]; tot[rr][2] = acc_v[1][rr]; tot[rr][3] = acc_v[2][rr];
          if constexpr (KS == 4) { tot[rr][4] = acc_q[0][rr]; tot[rr][5] = acc_q[1][rr]; tot[rr][6] = acc_q[2][rr]; }
#pragma unroll
          for (int o = 0; o < NSUB - 1; ++o) {
            const float* src = xchg + (size_t)o * NACC * 128 + row;
#pragma unroll
            for (int a = 0; a < 4 + NQ; ++a) tot[rr][a] += src[(rr * (4 + NQ) + a) * 128];
          }
        }
        bool finish = true;                          // this CTA writes the outputs of the item
        const bool whole = (bo == 0 && nb == sg.item_nb);
        if (!whole) {
          // the item is shared with neighbouring CTAs: park the partial sums, the last CTA to arrive adds them in CTA order
          const int64_t item_x0 = (int64_t)slice * TB + bptr[chunk];
          const int cta_first = cta_of_batch(item_x0, T, G), cta_last = cta_of_batch(item_x0 + sg.item_nb - 1, T, G);
          float* mine = part_ws + ((size_t)blockIdx.x * 2 + (first_seg ? 0 : 1)) * NACC * 128 + row;
#pragma unroll
          for (int rr = 0; rr < RC; ++rr)
#pragma unroll
            for (int a = 0; a < 4 + NQ; ++a) __stcg(mine + (rr * (4 + NQ) + a) * 128, tot[rr][a]);
          __threadfence();
          named_bar_sync(2, 128);
          int* flag = reinterpret_cast<int*>(smem_raw + M::TMEM_PTR + 4);
          if (tid == 0) *flag = (atomicAdd(&tickets[sg.item], 1) == cta_last - cta_first) ? 1 : 0;
          named_bar_sync(2, 128);
          finish = *flag != 0;
          if (finish) {
            __threadfence();
#pragma unroll
            for (int rr = 0; rr < RC; ++rr)
#pragma unroll
              for (int a = 0; a < 4 + NQ; ++a) tot[rr][a] = 0.f;
            for (int cb = cta_first; cb <= cta_last; ++cb) {
              // slot 0: the item is the first one of CTA cb's range; slot 1: a later one
              const int64_t cb_lo = ((int64_t)cb * T) / G;
              const int slot = (cb_lo >= item_x0) ? 0 : 1;
              const float* src = part_ws + ((size_t)cb * 2 + slot) * NACC * 128 + row;
#pragma unroll
              for (int rr = 0; rr < RC; ++rr)
#pragma unroll
                for (int a = 0; a < 4 + NQ; ++a) tot[rr][a] += __ldcg(src + (rr * (4 + NQ) + a) * 128);
            }
            if (tid == 0) tickets[sg.item] = 0;      // left zero for the next launch
          }
        }
        if (finish && active) {
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) {
            const int64_t i = (int64_t)chunk * RC + rr;
            if (i < n_recv) {
              float a_s = tot[rr][0], a0 = tot[rr][1], a1 = tot[rr][2], a2 = tot[rr][3];
              const int64_t so = i * F + f, vo = i * 3 * F + f;
              if constexpr (KS == 4) {
                // sum_e m3 (v_i x v_j) = v_i x q_i
                const float q0 = tot[rr][4], q1 = tot[rr][5], q2 = tot[rr][6];
                float vi0 = 0.f, vi1 = 0.f, vi2 = 0.f;
                if (!v_is_zero) {
                  vi0 = v_recv[vo]; vi1 = v_recv[vo + F]; vi2 = v_recv[vo + 2 * (int64_t)F];
                }
                a0 += vi1 * q2 - vi2 * q1;
                a1 += vi2 * q0 - vi0 * q2;
                a2 += vi0 * q1 - vi1 * q0;
                if (q_out) {
                  q_out[vo] = q0; q_out[vo + F] = q1; q_out[vo + 2 * (int64_t)F] = q2;
                }
              }
              out_s[so] = (res_s ? res_s[so] : 0.f) + a_s;
              out_v[vo] = (res_v ? res_v[vo] : 0.f) + a0;
              out_v[vo + F] = (res_v ? res_v[vo + F] : 0.f) + a1;
              out_v[vo + 2 * (int64_t)F] = (res_v ? res_v[vo + 2 * (int64_t)F] : 0.f) + a2;
            }
          }
        }
      }
      if constexpr (NSUB > 1) named_bar_sync(1, NCONS * 32);      // the exchange buffer is free again
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NCONS + 1) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// 3xTF32 filter (default) and 1xTF32 filter (cgvae_set_matmul_precision(1)): same records, same work partition
template <int KS, int RC, int NSUB>
__global__ void __launch_bounds__((4 * NSUB + 2) * 32, 1) message_tc_fwd_kernel(MESSAGE_TC_FWD_PARAMS) {
  message_tc_fwd_body<KS, RC, NSUB, false>(MESSAGE_TC_FWD_ARGS);
}
template <int KS, int RC, int NSUB>
__global__ void __launch_bounds__((4 * NSUB + 2) * 32, 1) message_tc1_fwd_kernel(MESSAGE_TC_FWD_PARAMS) {
  message_tc_fwd_body<KS, RC, NSUB, true>(MESSAGE_TC_FWD_ARGS);
}
#undef MESSAGE_TC_FWD_PARAMS
#undef MESSAGE_TC_FWD_ARGS

}  // namespace mtc
}  // namespace cgvae

using namespace cgvae;

extern "C" {

int64_t cgvae_msg_tiles_batches_cap(int64_t n_rows, int64_t n_partners, int64_t n_edge_slots, int RC) {
  if (RC != 4 && RC != 8 && RC != 16) return -1;
  const int64_t n_chunks = ceil_div(n_rows, RC), GB = mtc::NB / RC;
  int64_t groups = std::min(n_edge_slots, n_chunks * n_partners);   // every group holds at least one edge
  return ceil_div(groups, GB) + n_chunks + 1;
}
size_t cgvae_msg_tiles_rec_bytes(void) { return mtc::REC_BYTES; }

int cgvae_msg_tiles_build(const int32_t* rowptr, const int32_t* col, const int32_t* slot_map, int64_t n_rows, int64_t n_partners,
                          int64_t n_edge_slots, const float* basis, const float* unit, int RB, int RC, int32_t* nbatch,
                          int32_t* bptr, int32_t* ngroups, void* rec, int64_t n_batches_cap, cgvae_stream_t stream) {
  CGVAE_REQUIRE(RC == 4 || RC == 8 || RC == 16, "msg_tiles_build: RC must be 4, 8 or 16 (got %d)", RC);
  CGVAE_REQUIRE(RB == 8 || RB == 12 || RB == 16, "msg_tiles_build: RB must be 8, 12 or 16 (got %d)", RB);
  CGVAE_REQUIRE(n_partners <= 262144, "msg_tiles_build: at most 262144 partner nodes (got %lld)", (long long)n_partners);
  CGVAE_REQUIRE(rowptr && col && basis && unit && nbatch && bptr && ngroups && rec, "msg_tiles_build: null pointer");
  CGVAE_REQUIRE(n_batches_cap >= cgvae_msg_tiles_batches_cap(n_rows, n_partners, n_edge_slots, RC),
                "msg_tiles_build: record capacity too small");
  CGVAE_REQUIRE(aligned16(basis) && aligned16(unit) && aligned16(rec), "msg_tiles_build: buffers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_chunks = ceil_div(n_rows, RC);
  if (n_chunks == 0) return 0;
  const size_t W = (size_t)((n_partners + 31) / 32);
  const size_t sm_bytes = sizeof(uint32_t) * W + sizeof(int) * (mtc::kTileThreads + 1) + 16;
  static std::atomic<size_t> attr_bytes{0};
  if (sm_bytes > 48 * 1024 && attr_bytes.load() < sm_bytes) {
    CGVAE_CUDA(cudaFuncSetAttribute(mtc::tile_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_bytes));
    CGVAE_CUDA(cudaFuncSetAttribute(mtc::tile_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_bytes));
    attr_bytes.store(sm_bytes);
  }
  launch_kernel(mtc::tile_count_kernel, dim3((unsigned)n_chunks), dim3(mtc::kTileThreads), sm_bytes, st, rowptr, col, n_rows, n_partners, RC,
                nbatch, ngroups);
  if (int rc = launched("msg_tile_count")) return rc;
  if (int rc = cgvae_scan_i32(nbatch, n_chunks, bptr, stream)) return rc;
  CGVAE_ZERO(rec, (size_t)n_batches_cap * mtc::REC_BYTES, st);
  launch_kernel(mtc::tile_fill_kernel, dim3((unsigned)n_chunks), dim3(mtc::kTileThreads), sm_bytes, st, rowptr, col, slot_map, n_rows,
                n_partners, RC, (const int32_t*)bptr, basis, unit, RB, reinterpret_cast<char*>(rec), n_batches_cap);
  return launched("msg_tile_fill");
}

size_t cgvae_message_tc_ws_bytes(int n_split, int RC, int64_t n_rows, int F) {
  const int64_t n_items = ceil_div(n_rows, RC) * ceil_div(F, 128);
  const size_t nacc = (size_t)RC * (n_split == 4 ? 7 : 4);
  // [tickets: n_items int32 | pad] [partial sums: kNumSM x 2 x nacc x 128 floats]
  return ((size_t)n_items * 4 + 255) / 256 * 256 + (size_t)kNumSM * 2 * nacc * 128 * 4 + 256;
}

int cgvae_message_tc_fwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const int32_t* bptr,
                         const int32_t* ngroups, const void* rec, int64_t n_batches_cap, int RC, const float* Wf, const float* bf,
                         int64_t n_recv, int F, int R, const float* res_s, const float* res_v, int v_is_zero, float* out_s,
                         float* out_v, float* q, void* ws, size_t ws_bytes, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n_split == 3 || n_split == 4, "message_tc_fwd: n_split must be 3 or 4 (got %d)", n_split);
  CGVAE_REQUIRE(RC == 4 || RC == 8 || RC == 16, "message_tc_fwd: RC must be 4, 8 or 16 (got %d)", RC);
  CGVAE_REQUIRE(n_split == 3 || RC <= 8, "message_tc_fwd: the cross block runs with RC = 4 or 8 (register budget)");
  CGVAE_REQUIRE(R >= 1 && R + 1 <= mtc::KT && F >= 1, "message_tc_fwd: need 1 <= R <= 15");
  if (n_recv == 0) return 0;
  CGVAE_REQUIRE(phi && bptr && ngroups && rec && Wf && bf && out_s && out_v, "message_tc_fwd: null pointer");
  CGVAE_REQUIRE(v_is_zero || v_send, "message_tc_fwd: v_send missing");
  CGVAE_REQUIRE(n_split != 4 || v_is_zero || v_recv, "message_tc_fwd: v_recv missing for the cross block");
  CGVAE_REQUIRE(aligned16(rec), "message_tc_fwd: records must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_chunks = ceil_div(n_recv, RC), n_items = n_chunks * ceil_div(F, 128);
  CGVAE_REQUIRE(n_items < INT_MAX, "message_tc_fwd: too many work items");
  CGVAE_REQUIRE((int64_t)n_recv * n_split * F < (int64_t)1 << 31, "message_tc_fwd: feature arrays beyond 2^31 elements");
  CGVAE_REQUIRE(ws && ws_bytes >= cgvae_message_tc_ws_bytes(n_split, RC, n_recv, F), "message_tc_fwd: workspace too small");
  // one persistent CTA per SM (fewer only when there are fewer batches than SMs: the upper bound is the record capacity)
  dim3 grid((unsigned)std::max<int64_t>(1, std::min<int64_t>(n_batches_cap * ceil_div(F, 128), kNumSM)));
  const char* recp = reinterpret_cast<const char*>(rec);
  int32_t* tickets = reinterpret_cast<int32_t*>(ws);
  const size_t tick_bytes = ((size_t)n_items * 4 + 255) / 256 * 256;
  float* part_ws = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + tick_bytes);
  CGVAE_ZERO(tickets, tick_bytes, st);
  // the precision mode picks the kernel only (cgvae_set_matmul_precision): records, grid and partition are the same
  const int one = matmul_precision() == 1 ? 1 : 0;
#define LAUNCH_TC_FWD(KS, RCV, NSUB)                                                                                             \
  do {                                                                                                                           \
    static bool attr_done[2] = {false, false};                                                                                   \
    constexpr size_t smb = mtc::Map<NSUB, RCV*(KS == 4 ? 7 : 4)>::BYTES;                                                   \
    auto kernel = one ? mtc::message_tc1_fwd_kernel<KS, RCV, NSUB> : mtc::message_tc_fwd_kernel<KS, RCV, NSUB>;               \
    if (!attr_done[one]) {                                                                                                       \
      CGVAE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smb));                            \
      attr_done[one] = true;                                                                                                     \
    }                                                                                                                            \
    launch_kernel(kernel, grid, dim3((4 * NSUB + 2) * 32), smb, st, phi, v_send, v_recv, bptr, ngroups,                          \
                  recp, Wf, bf, n_recv, F, R, res_s, res_v, v_is_zero, out_s, out_v, q, (int)n_chunks, (int)n_items, tickets,    \
                  part_ws);                                                                                                      \
  } while (0)
  if (n_split == 3) {
    // RC = 8 with 8 consumer warps (NSUB = 2: 320 threads, no spills) beats 16 consumer warps at 96 registers (48-byte spill in
    // the column loop): 76.8 vs 80.7 us at the chignolin atom graph, 15.7 vs 16.2 ms at c5 / 12 A
    if (RC == 4) LAUNCH_TC_FWD(3, 4, 4);
    else if (RC == 8) LAUNCH_TC_FWD(3, 8, 2);
    else LAUNCH_TC_FWD(3, 16, 2);
  } else {
    // RC = 8: 56 accumulators per thread only fit with 8 consumer warps (NSUB = 2: 320 threads, 204 registers each)
    if (RC == 4) LAUNCH_TC_FWD(4, 4, 4); else LAUNCH_TC_FWD(4, 8, 2);
  }
#undef LAUNCH_TC_FWD
  return launched("message_tc_fwd");
}

}  // extern "C"
