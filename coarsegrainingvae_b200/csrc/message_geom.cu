// Geometry cotangents of the message layers: the part of the message-layer backward that only runs when a coordinate
// requires grad.  For an edge e = (i <- j) of the receiver CSR, with w_e[k][f] = sum_r basis_e[r] Wf'[kF+f][r]:
//   3 / 4 splits:  gm0 = <gv_i, v_j>, gm1 = gs_i, gm2 = <gv_i, u_e>, gm3 = <gv_i, v_i x v_j> (4 splits)
//                  d_basis_e[r] = sum_k sum_f gm_k[f] phi_j[k][f] Wf'[kF+f][r]
//                  d_unit_e[c]  = sum_f phi_j[2][f] w_e[2][f] gv_i[c][f]
//   9 splits (unit-only form; d_basis comes from the filter gradient gw of cgvae_message9_bwd):
//                  d_unit_e[c]  = sum_f phi_j[1][f] w_e[1][f] gv_i[c][f]
// A CTA takes 32 consecutive edge slots and all F/32 channel slices; warp w walks slices w, w + nw, ... with the slice's
// filter in registers and reduces its RB + 3 per-edge partials across lanes with a transposing butterfly (31 shuffles for
// 32 values).  The warps' partials are added in warp order in shared memory and every edge is stored once: no atomics,
// a fixed summation order, bitwise repeatable.
#include "common.cuh"

namespace cgvae {

constexpr int kGeomEdges = 32;     // edge slots per CTA
constexpr int kGeomMaxWarps = 8;   // channel-slice warps per CTA

// v[0..31] summed over the warp's 32 lanes; on return v[0] of lane L holds the total of value L
__device__ __forceinline__ void transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16, n = 16; o >= 1; o >>= 1, n >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int t = 0; t < n; ++t) {
      const float send = upper ? v[t] : v[t + n];
      const float keep = upper ? v[t + n] : v[t];
      v[t] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
}

// KS = 3, 4: full form; KS = 9: unit-only form (split 1 carries u)
template <int KS, int RBQ>
__global__ void __launch_bounds__(kGeomMaxWarps * 32) message_geom_bwd_kernel(
    const float* __restrict__ phi, const float* __restrict__ v_send, const float* __restrict__ v_recv,
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_recv, int64_t n_edges,
    const float* __restrict__ basis, const float* __restrict__ unit, const float* __restrict__ Wf, const float* __restrict__ bf,
    int F, int R, const float* __restrict__ g_out_s, const float* __restrict__ g_out_v, int v_is_zero,
    float* __restrict__ d_basis, float* __restrict__ d_unit) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int RB = 4 * RBQ;
  constexpr bool kUnitOnly = KS == 9;
  constexpr int KW = kUnitOnly ? 1 : KS;       // filter splits held in registers
  constexpr int kU = kUnitOnly ? 1 : 2;        // split that multiplies the unit vector
  __shared__ float part[kGeomMaxWarps][kGeomEdges][32];
  __shared__ float4 sbasis[kGeomEdges * RBQ];
  __shared__ float4 sunit[kGeomEdges];
  __shared__ int scol[kGeomEdges], srecv[kGeomEdges];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int64_t e0 = (int64_t)blockIdx.x * kGeomEdges;
  const int64_t live = rowptr[n_recv];
  const int n = (int)max((int64_t)0, min((int64_t)kGeomEdges, min(n_edges, live) - e0));   // live slots of this CTA
  if (threadIdx.x < n) {
    const int64_t e = e0 + threadIdx.x;
    scol[threadIdx.x] = col[e];
    srecv[threadIdx.x] = row_of_slot(rowptr, n_recv, (int)e);
    sunit[threadIdx.x] = __ldg(reinterpret_cast<const float4*>(unit) + e);
  }
  for (int q = threadIdx.x; q < n * RBQ; q += blockDim.x) sbasis[q] = __ldg(reinterpret_cast<const float4*>(basis) + e0 * RBQ + q);
  __syncthreads();

  const int n_slices = (F + 31) / 32;
  for (int sl = warp; sl < n_slices; sl += nw) {
    const int f = sl * 32 + lane;
    const bool active = f < F;
    const int fc = active ? f : F - 1;
    float W[KW][RB];
#pragma unroll
    for (int k = 0; k < KW; ++k)
#pragma unroll
      for (int r = 0; r < RB; ++r) W[k][r] = filter_entry(Wf, bf, F, R, kUnitOnly ? kU : k, fc, r);
    for (int t = 0; t < n; ++t) {
      const int i = srecv[t], j = scol[t];
      float b[RB];
#pragma unroll
      for (int q = 0; q < RBQ; ++q) {
        const float4 x = sbasis[t * RBQ + q];
        b[4 * q + 0] = x.x; b[4 * q + 1] = x.y; b[4 * q + 2] = x.z; b[4 * q + 3] = x.w;
      }
      const float4 u = sunit[t];
      // inactive lanes read zero output gradients: every partial they form is zero
      float gv[3] = {0.f, 0.f, 0.f}, gs = 0.f;
      if (active) {
        const float* gp = g_out_v + (int64_t)i * 3 * F + f;
        gv[0] = __ldg(gp); gv[1] = __ldg(gp + F); gv[2] = __ldg(gp + 2 * F);
        if (!kUnitOnly) gs = __ldg(g_out_s + (int64_t)i * F + f);
      }
      const float* pj = phi + (int64_t)j * KS * F + fc;
      float wu = 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) wu = fmaf(b[r], W[kUnitOnly ? 0 : kU][r], wu);
      const float au = __ldg(pj + (int64_t)kU * F) * wu;
      float val[32];
#pragma unroll
      for (int x = 0; x < 32; ++x) val[x] = 0.f;
      if constexpr (!kUnitOnly) {
        float a[KS];
        a[1] = gs * __ldg(pj + F);
        a[2] = (gv[0] * u.x + gv[1] * u.y + gv[2] * u.z) * __ldg(pj + 2 * F);
        a[0] = 0.f;
        if constexpr (KS == 4) a[3] = 0.f;
        if (!v_is_zero) {
          const float* vp = v_send + (int64_t)j * 3 * F + fc;
          const float vj0 = __ldg(vp), vj1 = __ldg(vp + F), vj2 = __ldg(vp + 2 * F);
          a[0] = (gv[0] * vj0 + gv[1] * vj1 + gv[2] * vj2) * __ldg(pj);
          if constexpr (KS == 4) {
            const float* wp = v_recv + (int64_t)i * 3 * F + fc;
            const float vi0 = __ldg(wp), vi1 = __ldg(wp + F), vi2 = __ldg(wp + 2 * F);
            const float c0 = vi1 * vj2 - vi2 * vj1, c1 = vi2 * vj0 - vi0 * vj2, c2 = vi0 * vj1 - vi1 * vj0;
            a[3] = (gv[0] * c0 + gv[1] * c1 + gv[2] * c2) * __ldg(pj + 3 * F);
          }
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          float s = 0.f;
#pragma unroll
          for (int k = 0; k < KS; ++k) s = fmaf(a[k], W[k][r], s);
          val[r] = s;
        }
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) val[RB + c] = au * gv[c];
      transpose_reduce32(val, lane);
      part[warp][t][lane] = (sl == warp) ? val[0] : part[warp][t][lane] + val[0];
    }
  }
  __syncthreads();
  // one store per edge value, warps added in warp order; padded tail slots get zero
  const int nw_used = min(nw, n_slices);
  const int n_all = (int)min((int64_t)kGeomEdges, n_edges - e0);
  for (int idx = threadIdx.x; idx < n_all * 32; idx += blockDim.x) {
    const int t = idx >> 5, x = idx & 31;
    float s = 0.f;
    if (t < n)
      for (int w = 0; w < nw_used; ++w) s += part[w][t][x];
    const int64_t e = e0 + t;
    if (x < RB) {
      if (!kUnitOnly) d_basis[e * RB + x] = s;
    } else if (x < RB + 4) {
      d_unit[e * 4 + (x - RB)] = (x < RB + 3) ? s : 0.f;
    }
  }
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

int cgvae_message_geom_bwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const int32_t* rowptr,
                           const int32_t* col, int64_t n_recv, int64_t n_edges, const float* basis, const float* unit,
                           const float* Wf, const float* bf, int F, int R, int RB, const float* g_out_s, const float* g_out_v,
                           int v_is_zero, float* d_basis, float* d_unit, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n_split == 3 || n_split == 4 || n_split == 9, "message_geom_bwd: n_split must be 3, 4 or 9 (got %d)", n_split);
  CGVAE_REQUIRE((RB == 8 || RB == 12 || RB == 16) && R + 1 <= RB && F >= 1, "message_geom_bwd: bad RB=%d R=%d F=%d", RB, R, F);
  if (n_edges == 0) return 0;
  CGVAE_REQUIRE(phi && rowptr && col && basis && unit && Wf && bf && g_out_v && d_unit && (n_split == 9 || (g_out_s && d_basis)),
                "message_geom_bwd: null pointer");
  CGVAE_REQUIRE(n_split == 9 || v_is_zero || v_send, "message_geom_bwd: v_send missing");
  CGVAE_REQUIRE(n_split != 4 || v_is_zero || v_recv, "message_geom_bwd: v_recv missing for the cross block");
  CGVAE_REQUIRE(aligned16(basis) && aligned16(unit), "message_geom_bwd: edge data must be 16-byte aligned");
  const int nw = (int)std::min<int64_t>(kGeomMaxWarps, ceil_div(F, 32));
  const dim3 grid((unsigned)ceil_div(n_edges, kGeomEdges));
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_GEOM(KS, RBQ)                                                                                                 \
  launch_kernel(message_geom_bwd_kernel<KS, RBQ>, grid, dim3(nw * 32), 0, st, phi, v_send, v_recv, rowptr, col, n_recv, n_edges, \
                basis, unit, Wf, bf, F, R, g_out_s, g_out_v, v_is_zero, d_basis, d_unit)
  if (n_split == 3) {
    if (RB == 8) LAUNCH_GEOM(3, 2); else if (RB == 12) LAUNCH_GEOM(3, 3); else LAUNCH_GEOM(3, 4);
  } else if (n_split == 4) {
    if (RB == 8) LAUNCH_GEOM(4, 2); else if (RB == 12) LAUNCH_GEOM(4, 3); else LAUNCH_GEOM(4, 4);
  } else {
    if (RB == 8) LAUNCH_GEOM(9, 2); else if (RB == 12) LAUNCH_GEOM(9, 3); else LAUNCH_GEOM(9, 4);
  }
#undef LAUNCH_GEOM
  return launched("message_geom_bwd");
}

}  // extern "C"
