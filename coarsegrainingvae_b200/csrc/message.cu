// Fused message layers (EquiMessageBlock / EquiMessageCross / ContractiveMessageBlock / EquiMessagePsuedo).
//
// Mapping (round 1, fp32 SIMT): one warp per receiver (forward) or per sender (backward), lane = channel,
// a CTA = 4 warps working on neighbouring rows of the same 32-channel slice so that the gathered
// sender rows (phi[j][k][f0..f0+31], v[j][c][f0..f0+31], 128 B each) are re-used out of L1.
// The filter slice [K][RB][32] lives in registers (K = 3, 4) or shared memory (K = 9); the per-edge
// metadata (sender index, basis row, unit vector) is staged 32 edges at a time per warp in shared memory
// (coalesced loads, next batch prefetched in registers) and read back as broadcasts.  Receivers accumulate in registers and store
// once: no atomics, fixed summation order (CSR order == reference edge-list order).
#include "common.cuh"

namespace cgvae {

constexpr int kMsgWarps = 4;
constexpr int kFwdWarps = 4;   // warps (= receivers in flight) per CTA of the forward kernel

template <int RBQ>
__device__ __forceinline__ void load_basis(const float* __restrict__ basis, int e, float (&b)[4 * RBQ]) {
  const float4* p = reinterpret_cast<const float4*>(basis) + (int64_t)e * RBQ;
#pragma unroll
  for (int q = 0; q < RBQ; ++q) {
    const float4 t = __ldg(p + q);
    b[4 * q + 0] = t.x; b[4 * q + 1] = t.y; b[4 * q + 2] = t.z; b[4 * q + 3] = t.w;
  }
}

// filter column for (split k, channel f): rows r < R from Wf[(k*F+f)][r], row R = bias, rest zero
__device__ __forceinline__ float filter_entry(const float* __restrict__ Wf, const float* __restrict__ bf, int F, int R,
                                              int k, int f, int r) {
  if (r < R) return Wf[((int64_t)k * F + f) * R + r];
  if (r == R) return bf[(int64_t)k * F + f];
  return 0.f;
}

// ------------------------------------------------------------------------------------------
// forward, 3 or 4 splits
// ------------------------------------------------------------------------------------------
template <int KS, int RBQ>
__global__ void __launch_bounds__(kFwdWarps * 32, 5) message_fwd_kernel(
    const float* __restrict__ phi, const float* __restrict__ v_send, const float* __restrict__ v_recv,
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ basis,
    const float* __restrict__ unit, const float* __restrict__ Wf, const float* __restrict__ bf, int64_t n_recv, int F, int R,
    const float* __restrict__ res_s, const float* __restrict__ res_v, int v_is_zero, float* __restrict__ out_s,
    float* __restrict__ out_v, float* __restrict__ q_out, int recv_per_cta) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int RB = 4 * RBQ;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int f = blockIdx.y * 32 + lane;
  const bool active = f < F;
  const int fc = active ? f : F - 1;  // clamp: inactive lanes compute on a valid channel, never store

  float W[KS][RB];
#pragma unroll
  for (int k = 0; k < KS; ++k)
#pragma unroll
    for (int r = 0; r < RB; ++r) W[k][r] = filter_entry(Wf, bf, F, R, k, fc, r);

  // A CTA handles recv_per_cta consecutive receivers, kFwdWarps at a time (neighbouring receivers share most of their
  // senders: the gathered 128-byte rows hit L1).  Measured on B200 (c5, 20 000 atoms): one pass of 4 receivers per CTA
  // (dynamic block scheduling, 231 M edges/s) beats 8-warp CTAs (214) and persistent chunks of 64..870 receivers
  // (193..126): co-resident CTAs of different chunks thrash L1, so the host passes recv_per_cta = kFwdWarps.
  const int64_t i_beg = (int64_t)blockIdx.x * recv_per_cta;
  const int64_t i_end = min(n_recv, i_beg + recv_per_cta);
  // Per-edge metadata (sender index, basis row, unit vector: 68 bytes at RB = 12) is warp-uniform.  Read per edge it was
  // five dependent L2 round trips in front of every gather (the slices of a receiver sit in different CTAs, so these
  // lines miss L1); now each warp stages 32 edges at a time through shared memory with coalesced loads, and the next
  // 32 are already in flight in registers while the current ones are processed.
  __shared__ float4 sbasis[kFwdWarps][32 * RBQ];
  __shared__ float4 sunit[kFwdWarps][32];
  __shared__ int scol[kFwdWarps][32];
  const float4* __restrict__ basis4 = reinterpret_cast<const float4*>(basis);
  const float4* __restrict__ unit4 = reinterpret_cast<const float4*>(unit);
  for (int64_t i = i_beg + warp; i < i_end; i += kFwdWarps) {
  float acc_s = 0.f, acc_v[3] = {0.f, 0.f, 0.f}, acc_q[3] = {0.f, 0.f, 0.f};
  const int beg = rowptr[i], end = rowptr[i + 1];
  int pc = 0;
  float4 pu = make_float4(0.f, 0.f, 0.f, 0.f), pb[RBQ];
  auto prefetch = [&](int e0, int n) {
    if (lane < n) {
      pc = __ldg(col + e0 + lane);
      pu = __ldg(unit4 + e0 + lane);
    }
#pragma unroll
    for (int q = 0; q < RBQ; ++q)
      if (q * 32 + lane < n * RBQ) pb[q] = __ldg(basis4 + (int64_t)e0 * RBQ + q * 32 + lane);
  };
  int e0 = beg, n = min(32, end - beg);
  if (n > 0) prefetch(e0, n);
  while (n > 0) {
    __syncwarp();                                   // everybody is done with the previous 32 edges
    if (lane < n) {
      scol[warp][lane] = pc;
      sunit[warp][lane] = pu;
    }
#pragma unroll
    for (int q = 0; q < RBQ; ++q)
      if (q * 32 + lane < n * RBQ) sbasis[warp][q * 32 + lane] = pb[q];
    __syncwarp();
    const int e1 = e0 + n, n1 = min(32, end - e1);
    if (n1 > 0) prefetch(e1, n1);      // measured on B200 (c5, 11 M edges): 490 M edges/s with this prefetch, 452 without
#pragma unroll 4
    for (int t = 0; t < n; ++t) {
      const int j = scol[warp][t];
      float b[RB];
#pragma unroll
      for (int q = 0; q < RBQ; ++q) {
        const float4 x = sbasis[warp][t * RBQ + q];
        b[4 * q + 0] = x.x; b[4 * q + 1] = x.y; b[4 * q + 2] = x.z; b[4 * q + 3] = x.w;
      }
      const float4 u = sunit[warp][t];
      const float* pj = phi + (int64_t)j * KS * F + fc;
      float m[KS];
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        float w = 0.f;
#pragma unroll
        for (int r = 0; r < RB; ++r) w = fmaf(b[r], W[k][r], w);
        m[k] = __ldg(pj + (int64_t)k * F) * w;
      }
      acc_s += m[1];
      acc_v[0] = fmaf(m[2], u.x, acc_v[0]);
      acc_v[1] = fmaf(m[2], u.y, acc_v[1]);
      acc_v[2] = fmaf(m[2], u.z, acc_v[2]);
      if (!v_is_zero) {
        const float* vj = v_send + (int64_t)j * 3 * F + fc;
        const float v0 = __ldg(vj), v1 = __ldg(vj + F), v2 = __ldg(vj + 2 * F);
        acc_v[0] = fmaf(m[0], v0, acc_v[0]);
        acc_v[1] = fmaf(m[0], v1, acc_v[1]);
        acc_v[2] = fmaf(m[0], v2, acc_v[2]);
        if (KS == 4) {
          acc_q[0] = fmaf(m[3], v0, acc_q[0]);
          acc_q[1] = fmaf(m[3], v1, acc_q[1]);
          acc_q[2] = fmaf(m[3], v2, acc_q[2]);
        }
      }
    }
    e0 = e1;
    n = n1;
  }
  if (!active) continue;
  if (KS == 4) {
    // sum_e m3 (v_i x v_j) = v_i x q_i  (conv.py:379)
    float vi[3] = {0.f, 0.f, 0.f};
    if (!v_is_zero) {
      const float* p = v_recv + (int64_t)i * 3 * F + f;
      vi[0] = p[0]; vi[1] = p[F]; vi[2] = p[2 * F];
    }
    acc_v[0] += vi[1] * acc_q[2] - vi[2] * acc_q[1];
    acc_v[1] += vi[2] * acc_q[0] - vi[0] * acc_q[2];
    acc_v[2] += vi[0] * acc_q[1] - vi[1] * acc_q[0];
    if (q_out) {
      float* qo = q_out + (int64_t)i * 3 * F + f;
      qo[0] = acc_q[0]; qo[F] = acc_q[1]; qo[2 * F] = acc_q[2];
    }
  }
  const int64_t so = (int64_t)i * F + f, vo = (int64_t)i * 3 * F + f;
  out_s[so] = (res_s ? res_s[so] : 0.f) + acc_s;
#pragma unroll
  for (int c = 0; c < 3; ++c) out_v[vo + (int64_t)c * F] = (res_v ? res_v[vo + (int64_t)c * F] : 0.f) + acc_v[c];
  }
}

// ------------------------------------------------------------------------------------------
// backward, 3 or 4 splits: reduce by sender over the transposed CSR
//   B_j[k][r] = sum_{e: sender j} basis[e][r] * gm_k[e]   (gm_k = dL/dm_k without the phi factor)
//   g_phi[j][k] = sum_r W[k][r] B_j[k][r]          dW[k][r] += phi[j][k] B_j[k][r]
// ------------------------------------------------------------------------------------------
template <int KS, int RBQ>
__global__ void __launch_bounds__(kMsgWarps * 32) message_bwd_kernel(
    const float* __restrict__ phi, const float* __restrict__ v_send, const float* __restrict__ v_recv,
    const float* __restrict__ q, const int32_t* __restrict__ rowptr_t, const int32_t* __restrict__ col_t,
    const int32_t* __restrict__ perm_t, const float* __restrict__ basis, const float* __restrict__ unit,
    const float* __restrict__ Wf, const float* __restrict__ bf, int64_t n_send, int F, int R,
    const float* __restrict__ g_out_s, const float* __restrict__ g_out_v, int residual, int v_is_zero,
    float* __restrict__ g_phi, float* __restrict__ g_v_send, float* __restrict__ partial, int senders_per_cta) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int RB = 4 * RBQ;
  __shared__ float Wsm[KS][RB][32];
  __shared__ float dWsm[kMsgWarps][KS][RB][32];
  constexpr int CH = (KS * RBQ >= 16) ? 16 : 32;    // edges staged per refill (static shared memory stays below 48 KB)
  __shared__ float4 sbasis[kMsgWarps][CH * RBQ];
  __shared__ float4 sunit[kMsgWarps][CH];
  __shared__ int srecv[kMsgWarps][CH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int f = blockIdx.y * 32 + lane;
  const bool active = f < F;
  const int fc = active ? f : F - 1;
  for (int idx = threadIdx.x; idx < KS * RB * 32; idx += kMsgWarps * 32) {
    const int l = idx & 31, r = (idx >> 5) % RB, k = idx / (32 * RB);
    const int ff = min(blockIdx.y * 32 + l, F - 1);
    Wsm[k][r][l] = filter_entry(Wf, bf, F, R, k, ff, r);
  }
#pragma unroll
  for (int k = 0; k < KS; ++k)
#pragma unroll
    for (int r = 0; r < RB; ++r) dWsm[warp][k][r][lane] = 0.f;
  __syncthreads();
  float W0[RB], W3[KS == 4 ? RB : 1];
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    W0[r] = Wsm[0][r][lane];
    if constexpr (KS == 4) W3[r] = Wsm[3][r][lane];
  }

  const int64_t j_beg = (int64_t)blockIdx.x * senders_per_cta;
  const int64_t j_end = min(n_send, j_beg + senders_per_cta);
  for (int64_t j = j_beg + warp; j < j_end; j += kMsgWarps) {
    float ph[KS], vj[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < KS; ++k) ph[k] = phi[((int64_t)j * KS + k) * F + fc];
    if (!v_is_zero) {
      const float* p = v_send + (int64_t)j * 3 * F + fc;
      vj[0] = p[0]; vj[1] = p[F]; vj[2] = p[2 * F];
    }
    float B[KS][RB];
#pragma unroll
    for (int k = 0; k < KS; ++k)
#pragma unroll
      for (int r = 0; r < RB; ++r) B[k][r] = 0.f;
    float gvj[3] = {0.f, 0.f, 0.f};
    const int beg = rowptr_t[j], end = rowptr_t[j + 1];
    // 32 transposed-CSR slots at a time: receiver index and edge id come in coalesced, every lane fetches the basis row
    // and unit vector of ITS edge, all of it is parked in shared memory -- the per-edge chain perm_t -> basis[e] -> math
    // of the plain loop was two dependent L2 round trips per edge
    int p_i = 0, p_e = 0;
    int n = min(CH, end - beg);
    if (lane < n) { p_i = __ldg(col_t + beg + lane); p_e = __ldg(perm_t + beg + lane); }
    for (int t0 = beg; t0 < end; t0 += CH) {
      __syncwarp();
      if (lane < n) {
        srecv[warp][lane] = p_i;
        sunit[warp][lane] = __ldg(reinterpret_cast<const float4*>(unit) + p_e);
        const float4* brow = reinterpret_cast<const float4*>(basis) + (int64_t)p_e * RBQ;
#pragma unroll
        for (int q = 0; q < RBQ; ++q) sbasis[warp][lane * RBQ + q] = __ldg(brow + q);
      }
      __syncwarp();
      const int n_cur = n;
      n = min(CH, end - (t0 + CH));
      if (lane < n) { p_i = __ldg(col_t + t0 + CH + lane); p_e = __ldg(perm_t + t0 + CH + lane); }
#pragma unroll 2
    for (int tt = 0; tt < n_cur; ++tt) {
      const int i = srecv[warp][tt];
      float b[RB];
#pragma unroll
      for (int q = 0; q < RBQ; ++q) {
        const float4 x = sbasis[warp][tt * RBQ + q];
        b[4 * q + 0] = x.x; b[4 * q + 1] = x.y; b[4 * q + 2] = x.z; b[4 * q + 3] = x.w;
      }
      const float4 u = sunit[warp][tt];
      const float gs = __ldg(g_out_s + (int64_t)i * F + fc);
      const float* gp = g_out_v + (int64_t)i * 3 * F + fc;
      const float g0 = __ldg(gp), g1 = __ldg(gp + F), g2 = __ldg(gp + 2 * F);
      float gm[KS];
      gm[1] = gs;
      gm[2] = g0 * u.x + g1 * u.y + g2 * u.z;
      gm[0] = g0 * vj[0] + g1 * vj[1] + g2 * vj[2];
      float w0 = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) w0 = fmaf(b[r], W0[r], w0);
      const float m0 = ph[0] * w0;
      gvj[0] = fmaf(m0, g0, gvj[0]);
      gvj[1] = fmaf(m0, g1, gvj[1]);
      gvj[2] = fmaf(m0, g2, gvj[2]);
      if constexpr (KS == 4) {
        float x0 = 0.f, x1 = 0.f, x2 = 0.f;  // gq = g x v_i  (dL/dq_i)
        if (!v_is_zero) {
          const float* vp = v_recv + (int64_t)i * 3 * F + fc;
          const float a0 = __ldg(vp), a1 = __ldg(vp + F), a2 = __ldg(vp + 2 * F);
          x0 = g1 * a2 - g2 * a1;
          x1 = g2 * a0 - g0 * a2;
          x2 = g0 * a1 - g1 * a0;
        }
        gm[KS - 1] = x0 * vj[0] + x1 * vj[1] + x2 * vj[2];
        float w3 = 0.f;
#pragma unroll
        for (int r = 0; r < RB; ++r) w3 = fmaf(b[r], W3[r], w3);
        const float m3 = ph[KS - 1] * w3;
        gvj[0] = fmaf(m3, x0, gvj[0]);
        gvj[1] = fmaf(m3, x1, gvj[1]);
        gvj[2] = fmaf(m3, x2, gvj[2]);
      }
#pragma unroll
      for (int k = 0; k < KS; ++k)
#pragma unroll
        for (int r = 0; r < RB; ++r) B[k][r] = fmaf(b[r], gm[k], B[k][r]);
    }
    }
    // sender epilogue
#pragma unroll
    for (int k = 0; k < KS; ++k) {
      float gph = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        gph = fmaf(Wsm[k][r][lane], B[k][r], gph);
        dWsm[warp][k][r][lane] = fmaf(ph[k], B[k][r], dWsm[warp][k][r][lane]);
      }
      if (active) g_phi[((int64_t)j * KS + k) * F + f] = gph;
    }
    if (active) {
      const int64_t vo = (int64_t)j * 3 * F + f;
      if (residual || (KS == 4 && q != nullptr && !v_is_zero)) {
        // both need this node's own output gradient (homogeneous graph: node j is also a receiver)
        const float r0 = g_out_v[vo], r1 = g_out_v[vo + F], r2 = g_out_v[vo + 2 * (int64_t)F];
        if (residual) { gvj[0] += r0; gvj[1] += r1; gvj[2] += r2; }
        if (KS == 4 && q != nullptr && !v_is_zero) {
          // receiver-side term of v_j x q_j: dL/dv_j += q_j x g_j
          const float q0 = q[vo], q1 = q[vo + F], q2 = q[vo + 2 * (int64_t)F];
          gvj[0] += q1 * r2 - q2 * r1;
          gvj[1] += q2 * r0 - q0 * r2;
          gvj[2] += q0 * r1 - q1 * r0;
        }
      }
      g_v_send[vo] = gvj[0];
      g_v_send[vo + F] = gvj[1];
      g_v_send[vo + 2 * (int64_t)F] = gvj[2];
    }
  }
  __syncthreads();
  // CTA partial of dW in fixed warp order -> partial[chunk][k][r][f]
  for (int idx = threadIdx.x; idx < KS * RB * 32; idx += kMsgWarps * 32) {
    const int l = idx & 31, r = (idx >> 5) % RB, k = idx / (32 * RB);
    const int ff = blockIdx.y * 32 + l;
    if (ff < F) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kMsgWarps; ++w) s += dWsm[w][k][r][l];
      partial[(((int64_t)blockIdx.x * KS + k) * RB + r) * F + ff] = s;
    }
  }
}

// dWf[(k*F+f)][r] = sum_chunks partial[chunk][k][r][f] (r < R); dbf[k*F+f] = same at r == R
__global__ void __launch_bounds__(256) filter_grad_finalize_kernel(const float* __restrict__ partial, int n_chunks, int KS, int RB,
                                                                   int F, int R, float* __restrict__ dWf, float* __restrict__ dbf) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // over KS*(R+1)*F, f fastest
  if (idx >= (int64_t)KS * (R + 1) * F) return;
  const int f = (int)(idx % F);
  const int r = (int)((idx / F) % (R + 1));
  const int k = (int)(idx / ((int64_t)F * (R + 1)));
  float s = 0.f;
  for (int c = 0; c < n_chunks; ++c) s += partial[(((int64_t)c * KS + k) * RB + r) * F + f];
  if (r < R) dWf[((int64_t)k * F + f) * R + r] = s;
  else dbf[(int64_t)k * F + f] = s;
}

// ------------------------------------------------------------------------------------------
// 9 splits (EquiMessagePsuedo): decoder graphs of the molecule configs have 12..96 nodes; clarity first
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cross3(const float* a, const float* b, float* o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ float dot3(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void load3(const float* __restrict__ base, int64_t node, int F, int f, float* o) {
  const float* p = base + node * 3 * F + f;
  o[0] = p[0]; o[1] = p[F]; o[2] = p[2 * (int64_t)F];
}

constexpr int kMaxRB9 = 16;

// The slice of split k is the contiguous chunk Wf[(k*F+f0)*R ... +nch*R): read it coalesced and transpose into
// Wsm[k][r][lane].  All global loads are issued before the first shared store (fully unrolled, predicated), otherwise
// the ~36 dependent-latency round trips dominate these tiny-graph kernels.  blockDim.x == kMsgWarps*32.
__device__ __forceinline__ void stage_filter9(float (*Wsm)[kMaxRB9][32], const float* __restrict__ Wf,
                                              const float* __restrict__ bf, int F, int R, int RB, int f0) {
  constexpr int NTH = kMsgWarps * 32;
  constexpr int ITERS = (32 * (kMaxRB9 - 1) + NTH - 1) / NTH;   // R <= 15
  const int nch = min(32, F - f0);
  const int tid = threadIdx.x;
  int ls[ITERS], rs[ITERS];
  bool ok[ITERS];
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int idx = tid + it * NTH;
    ls[it] = idx / R;
    rs[it] = idx - ls[it] * R;
    ok[it] = idx < 32 * R && ls[it] < nch;
  }
  float tmp[9][ITERS], bias[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const float* src = Wf + ((int64_t)k * F + f0) * R;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) tmp[k][it] = ok[it] ? __ldg(src + tid + it * NTH) : 0.f;
    bias[k] = (tid < nch) ? __ldg(bf + (int64_t)k * F + f0 + tid) : 0.f;
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) {
#pragma unroll
    for (int it = 0; it < ITERS; ++it)
      if (tid + it * NTH < 32 * R) Wsm[k][rs[it]][ls[it]] = tmp[k][it];
    if (tid < 32) {
      Wsm[k][R][tid] = bias[k];
      for (int r = R + 1; r < RB; ++r) Wsm[k][r][tid] = 0.f;
    }
  }
}

// RB is a template parameter (RBQ float4 per basis row): the per-edge basis row sits in registers and the 9 x RB filter
// contraction is fully unrolled.  With a run-time RB the loop was a chain of dependent L1 loads (~50 cycles per term,
// 108 terms per edge): 23 us per launch on the 12-bead decoder graphs, almost all of it latency.
// UNR: edges of a node processed per unrolled group.  The decoder graphs of the molecule configs are tiny (12 beads, 5
// edges each, 57 CTAs): the kernel is a chain of dependent round trips (edge -> sender index -> gathers), and with
// UNR = 4 the loads of four edges are in flight together.  Large graphs (PCN: 16 000 residues) use UNR = 1: 64 registers.
template <int RBQ, int UNR>
__global__ void __launch_bounds__(kMsgWarps * 32) message9_fwd_kernel(
    const float* __restrict__ phi, const float* __restrict__ s, const float* __restrict__ sbar, const float* __restrict__ v,
    const float* __restrict__ vbar, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
    const float* __restrict__ basis, const float* __restrict__ unit, const float* __restrict__ Wf, const float* __restrict__ bf,
    int64_t n, int F, int R, int residual, float* __restrict__ out_s, float* __restrict__ out_sbar,
    float* __restrict__ out_v, float* __restrict__ out_vbar) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int RB = 4 * RBQ;
  __shared__ float Wsm[9][kMaxRB9][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  stage_filter9(Wsm, Wf, bf, F, R, RB, blockIdx.y * 32);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * kMsgWarps + warp;
  const int f = blockIdx.y * 32 + lane;
  if (i >= n || f >= F) return;
  const float s_i = s[i * F + f], sb_i = sbar[i * F + f];
  float v_i[3], vb_i[3];
  load3(v, i, F, f, v_i);
  load3(vbar, i, F, f, vb_i);
  float a_s = 0.f, a_sb = 0.f, a_v[3] = {0.f, 0.f, 0.f}, a_vb[3] = {0.f, 0.f, 0.f};
#pragma unroll UNR
  for (int e = rowptr[i]; e < rowptr[i + 1]; ++e) {
    const int j = col[e];
    float b[RB];
    load_basis<RBQ>(basis, e, b);
    const float4 u4 = reinterpret_cast<const float4*>(unit)[e];
    const float u[3] = {u4.x, u4.y, u4.z};
    float m[9], v_j[3], vb_j[3], c1[3], c2[3], c3[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) m[k] = __ldg(phi + ((int64_t)j * 9 + k) * F + f);   // all gathers in flight before the math
    load3(v, j, F, f, v_j);
    load3(vbar, j, F, f, vb_j);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      float w = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) w = fmaf(b[r], Wsm[k][r][lane], w);
      m[k] *= w;
    }
    cross3(v_i, vb_j, c1);
    cross3(v_i, v_j, c2);
    cross3(vb_i, vb_j, c3);
    a_s += m[0] * s_i;                         // conv.py:205
    a_sb += dot3(v_i, vb_j);                   // conv.py:206
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      a_v[c] += m[1] * u[c] + m[2] * v_j[c] + m[3] * c1[c] + m[4] * sb_i * vb_j[c];          // conv.py:209-212
      a_vb[c] += m[5] * vb_j[c] + m[6] * sb_i * v_j[c] + m[7] * c2[c] + m[8] * c3[c];        // conv.py:214-217
    }
  }
  const float rs = residual ? 1.f : 0.f;
  out_s[i * F + f] = rs * s_i + a_s;
  out_sbar[i * F + f] = rs * sb_i + a_sb;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    out_v[(i * 3 + c) * F + f] = rs * v_i[c] + a_v[c];
    out_vbar[(i * 3 + c) * F + f] = rs * vb_i[c] + a_vb[c];
  }
}

template <int RBQ, int UNR>
__global__ void __launch_bounds__(kMsgWarps * 32) message9_bwd_kernel(
    const float* __restrict__ phi, const float* __restrict__ s, const float* __restrict__ sbar, const float* __restrict__ v,
    const float* __restrict__ vbar, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
    const int32_t* __restrict__ rowptr_t, const int32_t* __restrict__ col_t, const int32_t* __restrict__ perm_t,
    const float* __restrict__ basis, const float* __restrict__ unit, const float* __restrict__ Wf, const float* __restrict__ bf,
    int64_t n, int F, int R, int residual, const float* __restrict__ g_s, const float* __restrict__ g_sbar,
    const float* __restrict__ g_v, const float* __restrict__ g_vbar, float* __restrict__ gi_s, float* __restrict__ gi_sbar,
    float* __restrict__ gi_v, float* __restrict__ gi_vbar, float* __restrict__ g_phi, float* __restrict__ gw) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int RB = 4 * RBQ;
  __shared__ float Wsm[9][kMaxRB9][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  stage_filter9(Wsm, Wf, bf, F, R, RB, blockIdx.y * 32);
  __syncthreads();
  const int64_t nd = (int64_t)blockIdx.x * kMsgWarps + warp;
  const int f = blockIdx.y * 32 + lane;
  if (nd >= n || f >= F) return;
  // this node's own state and output gradients
  const float gs_n = g_s[nd * F + f], gsb_n = g_sbar[nd * F + f];
  float v_n[3], vb_n[3], gv_n[3], gvb_n[3];
  load3(v, nd, F, f, v_n);
  load3(vbar, nd, F, f, vb_n);
  load3(g_v, nd, F, f, gv_n);
  load3(g_vbar, nd, F, f, gvb_n);
  const float rs = residual ? 1.f : 0.f;
  float d_s = rs * gs_n, d_sb = rs * gsb_n, d_v[3], d_vb[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) { d_v[c] = rs * gv_n[c]; d_vb[c] = rs * gvb_n[c]; }

  // ---- node as SENDER j = nd: edges (i <- nd)
  float ph[9], gph[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { ph[k] = phi[((int64_t)nd * 9 + k) * F + f]; gph[k] = 0.f; }
#pragma unroll UNR
  for (int t = rowptr_t[nd]; t < rowptr_t[nd + 1]; ++t) {
    const int i = col_t[t], e = perm_t[t];
    float b[RB];
    load_basis<RBQ>(basis, e, b);
    const float4 u4 = reinterpret_cast<const float4*>(unit)[e];
    const float u[3] = {u4.x, u4.y, u4.z};
    const float s_i = s[(int64_t)i * F + f], sb_i = sbar[(int64_t)i * F + f];
    const float gs_i = g_s[(int64_t)i * F + f], gsb_i = g_sbar[(int64_t)i * F + f];
    float v_i[3], vb_i[3], gv_i[3], gvb_i[3], c1[3], c2[3], c3[3];
    load3(v, i, F, f, v_i);
    load3(vbar, i, F, f, vb_i);
    load3(g_v, i, F, f, gv_i);
    load3(g_vbar, i, F, f, gvb_i);
    float w[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      float a = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) a = fmaf(b[r], Wsm[k][r][lane], a);
      w[k] = a;
    }
    cross3(v_i, vb_n, c1);     // v_i x vbar_j
    cross3(v_i, v_n, c2);      // v_i x v_j
    cross3(vb_i, vb_n, c3);    // vbar_i x vbar_j
    float gm[9];
    gm[0] = gs_i * s_i;
    gm[1] = dot3(gv_i, u);
    gm[2] = dot3(gv_i, v_n);
    gm[3] = dot3(gv_i, c1);
    gm[4] = sb_i * dot3(gv_i, vb_n);
    gm[5] = dot3(gvb_i, vb_n);
    gm[6] = sb_i * dot3(gvb_i, v_n);
    gm[7] = dot3(gvb_i, c2);
    gm[8] = dot3(gvb_i, c3);
    float* gwe = gw + ((int64_t)e * 9) * F + f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      gph[k] = fmaf(gm[k], w[k], gph[k]);
      gwe[(int64_t)k * F] = gm[k] * ph[k];
    }
    const float m2 = ph[2] * w[2], m3 = ph[3] * w[3], m4 = ph[4] * w[4], m5 = ph[5] * w[5];
    const float m6 = ph[6] * w[6], m7 = ph[7] * w[7], m8 = ph[8] * w[8];
    float x1[3], x2[3], x3[3];
    cross3(gvb_i, v_i, x1);    // d/dv_j of m7 (v_i x v_j)
    cross3(gv_i, v_i, x2);     // d/dvbar_j of m3 (v_i x vbar_j)
    cross3(gvb_i, vb_i, x3);   // d/dvbar_j of m8 (vbar_i x vbar_j)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      d_v[c] += m2 * gv_i[c] + m6 * sb_i * gvb_i[c] + m7 * x1[c];
      d_vb[c] += gsb_i * v_i[c] + m3 * x2[c] + m4 * sb_i * gv_i[c] + m5 * gvb_i[c] + m8 * x3[c];
    }
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) g_phi[((int64_t)nd * 9 + k) * F + f] = gph[k];

  // ---- node as RECEIVER i = nd: edges (nd <- j)
#pragma unroll UNR
  for (int e = rowptr[nd]; e < rowptr[nd + 1]; ++e) {
    const int j = col[e];
    float b[RB];
    load_basis<RBQ>(basis, e, b);
    float m[9], v_j[3], vb_j[3], y1[3], y2[3], y3[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) m[k] = (k == 1 || k == 2 || k == 5) ? 0.f : __ldg(phi + ((int64_t)j * 9 + k) * F + f);
    load3(v, j, F, f, v_j);
    load3(vbar, j, F, f, vb_j);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      if (k == 1 || k == 2 || k == 5) continue;
      float a = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) a = fmaf(b[r], Wsm[k][r][lane], a);
      m[k] *= a;
    }
    d_s += gs_n * m[0];
    d_sb += m[4] * dot3(gv_n, vb_j) + m[6] * dot3(gvb_n, v_j);
    cross3(vb_j, gv_n, y1);    // d/dv_i of m3 (v_i x vbar_j)
    cross3(v_j, gvb_n, y2);    // d/dv_i of m7 (v_i x v_j)
    cross3(vb_j, gvb_n, y3);   // d/dvbar_i of m8 (vbar_i x vbar_j)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      d_v[c] += gsb_n * vb_j[c] + m[3] * y1[c] + m[7] * y2[c];
      d_vb[c] += m[8] * y3[c];
    }
  }
  gi_s[nd * F + f] = d_s;
  gi_sbar[nd * F + f] = d_sb;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    gi_v[(nd * 3 + c) * F + f] = d_v[c];
    gi_vbar[(nd * 3 + c) * F + f] = d_vb[c];
  }
}

static int bwd_chunks(int64_t n_send, int F, int* senders_per_cta) {
  const int64_t fy = ceil_div(F, 32);
  int64_t chunks = (4 * (int64_t)kNumSM) / fy;  // about four CTAs per SM over the whole grid
  if (chunks < 1) chunks = 1;
  const int64_t max_chunks = ceil_div(n_send, kMsgWarps);
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  int64_t per = ceil_div(n_send, chunks);
  per = ceil_div(per, kMsgWarps) * kMsgWarps;
  if (per < kMsgWarps) per = kMsgWarps;
  *senders_per_cta = (int)per;
  return (int)std::max<int64_t>(1, ceil_div(n_send, per));
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

int cgvae_message_fwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const int32_t* rowptr,
                      const int32_t* col, const float* basis, const float* unit, const float* Wf, const float* bf,
                      int64_t n_recv, int64_t n_send, int F, int R, int RB, const float* res_s, const float* res_v,
                      int v_is_zero, float* out_s, float* out_v, float* q, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n_split == 3 || n_split == 4, "message_fwd: n_split must be 3 or 4 (got %d)", n_split);
  CGVAE_REQUIRE(RB == 8 || RB == 12 || RB == 16, "message_fwd: RB must be 8, 12 or 16 (got %d)", RB);
  CGVAE_REQUIRE(R + 1 <= RB && F >= 1, "message_fwd: need R+1 <= RB");
  if (n_recv == 0) return 0;
  CGVAE_REQUIRE(phi && rowptr && col && basis && unit && Wf && bf && out_s && out_v, "message_fwd: null pointer");
  CGVAE_REQUIRE(v_is_zero || v_send, "message_fwd: v_send missing");
  CGVAE_REQUIRE(n_split != 4 || v_is_zero || v_recv, "message_fwd: v_recv missing for the cross block");
  CGVAE_REQUIRE(aligned16(basis) && aligned16(unit), "message_fwd: edge data must be 16-byte aligned");
  const int64_t fy = ceil_div(F, 32);
  const int recv_per_cta = kFwdWarps;
  dim3 grid((unsigned)ceil_div(n_recv, recv_per_cta), (unsigned)fy);
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_FWD(KS, RBQ)                                                                                            \
  launch_kernel(message_fwd_kernel<KS, RBQ>, dim3(grid), dim3(kFwdWarps * 32), 0, st, phi, v_send, v_recv, rowptr, col, basis, unit, Wf, bf, \
                n_recv, F, R, res_s, res_v, v_is_zero, out_s, out_v, q, recv_per_cta)
  if (n_split == 3) {
    if (RB == 8) LAUNCH_FWD(3, 2); else if (RB == 12) LAUNCH_FWD(3, 3); else LAUNCH_FWD(3, 4);
  } else {
    if (RB == 8) LAUNCH_FWD(4, 2); else if (RB == 12) LAUNCH_FWD(4, 3); else LAUNCH_FWD(4, 4);
  }
#undef LAUNCH_FWD
  (void)n_send;
  return launched("message_fwd");
}

size_t cgvae_message_bwd_ws_bytes(int n_split, int F, int RB, int64_t n_send) {
  int per = 0;
  const int chunks = bwd_chunks(n_send > 0 ? n_send : 1, F, &per);
  return sizeof(float) * (size_t)chunks * (size_t)n_split * (size_t)RB * (size_t)F + 256;
}

int cgvae_message_bwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const float* q,
                      const int32_t* rowptr_t, const int32_t* col_t, const int32_t* perm_t, const float* basis,
                      const float* unit, const float* Wf, const float* bf, int64_t n_recv, int64_t n_send, int F, int R, int RB,
                      const float* g_out_s, const float* g_out_v, int residual, int v_is_zero, float* g_phi, float* g_v_send,
                      float* dWf, float* dbf, void* ws, size_t ws_bytes, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n_split == 3 || n_split == 4, "message_bwd: n_split must be 3 or 4 (got %d)", n_split);
  CGVAE_REQUIRE(RB == 8 || RB == 12 || RB == 16, "message_bwd: RB must be 8, 12 or 16 (got %d)", RB);
  CGVAE_REQUIRE(phi && rowptr_t && col_t && perm_t && basis && unit && Wf && bf && g_out_s && g_out_v && g_phi && g_v_send &&
                    dWf && dbf, "message_bwd: null pointer");
  CGVAE_REQUIRE(!residual || n_recv == n_send, "message_bwd: residual needs one node set");
  CGVAE_REQUIRE(n_split != 4 || n_recv == n_send, "message_bwd: the cross block needs one node set");
  CGVAE_REQUIRE(ws && ws_bytes >= cgvae_message_bwd_ws_bytes(n_split, F, RB, n_send), "message_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int per = 0;
  const int chunks = bwd_chunks(n_send > 0 ? n_send : 1, F, &per);
  float* partial = reinterpret_cast<float*>(ws);
  if (n_send == 0) {
    CGVAE_ZERO(partial, sizeof(float) * (size_t)n_split * RB * F, st);
  } else {
    dim3 grid((unsigned)chunks, (unsigned)ceil_div(F, 32));
    // (forcing 5 CTAs per SM -- 96 registers, 24 bytes of spills -- measured no faster on B200: 186 vs 183 us at chignolin)
#define LAUNCH_BWD(KS, RBQ)                                                                                               \
  launch_kernel(message_bwd_kernel<KS, RBQ>, dim3(grid), dim3(kMsgWarps * 32), 0, st, phi, v_send, v_recv, q, rowptr_t, col_t, perm_t, basis, unit, \
                                                               Wf, bf, n_send, F, R, g_out_s, g_out_v, residual, v_is_zero,  \
                                                               g_phi, g_v_send, partial, per)
    if (n_split == 3) {
      if (RB == 8) LAUNCH_BWD(3, 2); else if (RB == 12) LAUNCH_BWD(3, 3); else LAUNCH_BWD(3, 4);
    } else {
      if (RB == 8) LAUNCH_BWD(4, 2); else if (RB == 12) LAUNCH_BWD(4, 3); else LAUNCH_BWD(4, 4);
    }
#undef LAUNCH_BWD
    if (int rc = launched("message_bwd")) return rc;
  }
  const int64_t total = (int64_t)n_split * (R + 1) * F;
  launch_kernel(filter_grad_finalize_kernel, dim3((unsigned)ceil_div(total, 256)), dim3(256), 0, st, partial, n_send == 0 ? 1 : chunks, n_split, RB, F, R,
                                                                               dWf, dbf);
  return launched("filter_grad_finalize");
}

int cgvae_message9_fwd(const float* phi, const float* s, const float* sbar, const float* v, const float* vbar,
                       const int32_t* rowptr, const int32_t* col, const float* basis, const float* unit, const float* Wf,
                       const float* bf, int64_t n, int F, int R, int RB, int residual, float* out_s, float* out_sbar,
                       float* out_v, float* out_vbar, cgvae_stream_t stream) {
  CGVAE_REQUIRE((RB == 8 || RB == 12 || RB == 16) && R + 1 <= RB, "message9_fwd: bad RB=%d R=%d", RB, R);
  if (n == 0) return 0;
  CGVAE_REQUIRE(phi && s && sbar && v && vbar && rowptr && col && basis && unit && Wf && bf && out_s && out_sbar && out_v && out_vbar,
                "message9_fwd: null pointer");
  dim3 grid((unsigned)ceil_div(n, kMsgWarps), (unsigned)ceil_div(F, 32));
  CGVAE_REQUIRE(aligned16(basis) && aligned16(unit), "message9_fwd: edge data must be 16-byte aligned");
  const bool tiny = n <= 512;
#define LAUNCH_FWD9(RBQ)                                                                                                        \
  do {                                                                                                                          \
    if (tiny)                                                                                                                   \
      launch_kernel(message9_fwd_kernel<RBQ, 4>, dim3(grid), dim3(kMsgWarps * 32), 0, (cudaStream_t)stream, phi, s, sbar, v, vbar, rowptr, \
                    col, basis, unit, Wf, bf, n, F, R, residual, out_s, out_sbar, out_v, out_vbar);                              \
    else                                                                                                                        \
      launch_kernel(message9_fwd_kernel<RBQ, 1>, dim3(grid), dim3(kMsgWarps * 32), 0, (cudaStream_t)stream, phi, s, sbar, v, vbar, rowptr, \
                    col, basis, unit, Wf, bf, n, F, R, residual, out_s, out_sbar, out_v, out_vbar);                              \
  } while (0)
  if (RB == 8) LAUNCH_FWD9(2); else if (RB == 12) LAUNCH_FWD9(3); else LAUNCH_FWD9(4);
#undef LAUNCH_FWD9
  return launched("message9_fwd");
}

int cgvae_message9_bwd(const float* phi, const float* s, const float* sbar, const float* v, const float* vbar,
                       const int32_t* rowptr, const int32_t* col, const int32_t* rowptr_t, const int32_t* col_t,
                       const int32_t* perm_t, const float* basis, const float* unit, const float* Wf, const float* bf, int64_t n,
                       int64_t n_edge_slots, int F, int R, int RB, int residual, const float* g_s, const float* g_sbar, const float* g_v,
                       const float* g_vbar, float* gi_s, float* gi_sbar, float* gi_v, float* gi_vbar, float* g_phi, float* gw,
                       cgvae_stream_t stream) {
  CGVAE_REQUIRE((RB == 8 || RB == 12 || RB == 16) && R + 1 <= RB, "message9_bwd: bad RB=%d R=%d", RB, R);
  if (n == 0) return 0;
  CGVAE_REQUIRE(phi && s && sbar && v && vbar && rowptr && col && rowptr_t && col_t && perm_t && basis && unit && Wf && bf && g_s &&
                    g_sbar && g_v && g_vbar && gi_s && gi_sbar && gi_v && gi_vbar && g_phi && gw, "message9_bwd: null pointer");
  dim3 grid((unsigned)ceil_div(n, kMsgWarps), (unsigned)ceil_div(F, 32));
  // gw rows of unused (padded) edge slots must read as zero in the dWf = gw^T basis contraction
  CGVAE_ZERO(gw, sizeof(float) * (size_t)n_edge_slots * 9 * (size_t)F, (cudaStream_t)stream);
  CGVAE_REQUIRE(aligned16(basis) && aligned16(unit), "message9_bwd: edge data must be 16-byte aligned");
  const bool tiny = n <= 512;
#define LAUNCH_BWD9(RBQ)                                                                                                        \
  do {                                                                                                                          \
    if (tiny)                                                                                                                   \
      launch_kernel(message9_bwd_kernel<RBQ, 3>, dim3(grid), dim3(kMsgWarps * 32), 0, (cudaStream_t)stream, phi, s, sbar, v, vbar, rowptr, \
                    col, rowptr_t, col_t, perm_t, basis, unit, Wf, bf, n, F, R, residual, g_s, g_sbar, g_v, g_vbar, gi_s, gi_sbar, \
                    gi_v, gi_vbar, g_phi, gw);                                                                                  \
    else                                                                                                                        \
      launch_kernel(message9_bwd_kernel<RBQ, 1>, dim3(grid), dim3(kMsgWarps * 32), 0, (cudaStream_t)stream, phi, s, sbar, v, vbar, rowptr, \
                    col, rowptr_t, col_t, perm_t, basis, unit, Wf, bf, n, F, R, residual, g_s, g_sbar, g_v, g_vbar, gi_s, gi_sbar, \
                    gi_v, gi_vbar, g_phi, gw);                                                                                  \
  } while (0)
  if (RB == 8) LAUNCH_BWD9(2); else if (RB == 12) LAUNCH_BWD9(3); else LAUNCH_BWD9(4);
#undef LAUNCH_BWD9
  return launched("message9_bwd");
}

}  // extern "C"
