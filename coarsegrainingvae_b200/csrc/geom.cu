// Edge geometry: distance, unit vector, sinc radial basis x cosine envelope, once per graph
// (the reference recomputes these ~12 element-wise launches in every layer).
#include "common.cuh"

namespace cgvae {

__global__ void __launch_bounds__(256) edge_geometry_kernel(
    const float* __restrict__ xs, const float* __restrict__ xr, const float* __restrict__ r_edge,
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_recv, int64_t E,
    const float* __restrict__ coef, int R, int RB,
    float cutoff, const float* __restrict__ edge_wgt, const int32_t* __restrict__ eid, float* __restrict__ basis,
    float* __restrict__ unit) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  if (e >= rowptr[n_recv]) {
    // tail of a static-capacity graph (CUDA-graph replay): neutral records, so padded rows contribute exact zeros
    reinterpret_cast<float4*>(unit)[e] = make_float4(0.f, 0.f, 0.f, 1.f);
    for (int r = 0; r < RB; ++r) basis[e * RB + r] = 0.f;
    return;
  }
  float rx, ry, rz;
  if (r_edge != nullptr) {
    // block-level API: the caller supplies r_ij per edge in its original edge order
    const int64_t o = eid ? eid[e] : e;
    rx = r_edge[o * 3 + 0]; ry = r_edge[o * 3 + 1]; rz = r_edge[o * 3 + 2];
  } else {
    // r_ij = x_j - x_i (cgvae.py:276)
    const int i = row_of_slot(rowptr, n_recv, (int)e);
    const int j = col[e];
    rx = __fsub_rn(xs[(int64_t)j * 3 + 0], xr[(int64_t)i * 3 + 0]);
    ry = __fsub_rn(xs[(int64_t)j * 3 + 1], xr[(int64_t)i * 3 + 1]);
    rz = __fsub_rn(xs[(int64_t)j * 3 + 2], xr[(int64_t)i * 3 + 2]);
  }
  // d = sqrt(sum_c (r_c^2 + 1e-8)) (conv.py:26), fp32, unfused
  const float ax = __fadd_rn(__fmul_rn(rx, rx), 1e-8f);
  const float ay = __fadd_rn(__fmul_rn(ry, ry), 1e-8f);
  const float az = __fadd_rn(__fmul_rn(rz, rz), 1e-8f);
  const float d = __fsqrt_rn(__fadd_rn(__fadd_rn(ax, ay), az));
  float4 u;
  u.x = __fdiv_rn(rx, d);
  u.y = __fdiv_rn(ry, d);
  u.z = __fdiv_rn(rz, d);
  u.w = d;
  reinterpret_cast<float4*>(unit)[e] = u;
  const bool outside = d >= cutoff;
  // CosineEnvelope modules.py:54-56: 0.5 * (cos(pi * d / cutoff) + 1), fp32 pi
  float env = 0.f;
  if (!outside) env = 0.5f * (cosf(__fdiv_rn(__fmul_rn(3.14159265358979323846f, d), cutoff)) + 1.0f);
  float wgt = 1.0f;
  if (edge_wgt != nullptr) wgt = edge_wgt[eid ? eid[e] : e];
  float* b = basis + e * RB;
  for (int r = 0; r < RB; ++r) {
    float val = 0.f;
    if (r < R) {
      // PainnRadialBasis modules.py:161-170
      if (!outside) {
        const float c = coef[r];
        const float num = (d == 0.f) ? c : sinf(__fmul_rn(c, d));
        const float den = (d == 0.f) ? 1.0f : d;
        val = __fmul_rn(__fdiv_rn(num, den), env);
      }
    } else if (r == R) {
      val = env;  // bias column of DistanceEmbed (modules.py:192-197)
    }
    b[r] = val * wgt;
  }
}

// Backward of edge_geometry_kernel, the autograd of the reference's expressions (conv.py:25-29, modules.py:52-58,148-172):
//   d = sqrt(sum_c (r_c^2 + 1e-8)), dd/dr = u;  rbf_n' = (c_n cos(c_n d) - sin(c_n d) / d) / d;
//   env' = -1/2 (pi / cutoff) sin(pi d / cutoff); basis derivatives vanish for d >= cutoff; edge_wgt multiplies;
//   dr = dd u + (du - <u, du> u) / d.
// d_basis / d_unit (nullable = zero) are the cotangents of basis / unit.  Writes dr[e] per CSR slot (padded tail slots of a
// static-capacity graph: zero), or, with r_edge, d_r_edge[eid[e]] (every original edge owns exactly one slot).
__global__ void __launch_bounds__(256) edge_geometry_bwd_kernel(
    const float* __restrict__ xs, const float* __restrict__ xr, const float* __restrict__ r_edge,
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_recv, int64_t E,
    const float* __restrict__ coef, int R, int RB, float cutoff, const float* __restrict__ edge_wgt, const int32_t* __restrict__ eid,
    const float* __restrict__ d_basis, const float* __restrict__ d_unit, float* __restrict__ dr) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t o = (r_edge != nullptr && eid != nullptr) ? eid[e] : e;
  if (e >= rowptr[n_recv]) {
    dr[o * 3 + 0] = 0.f; dr[o * 3 + 1] = 0.f; dr[o * 3 + 2] = 0.f;
    return;
  }
  float rx, ry, rz;
  if (r_edge != nullptr) {
    rx = r_edge[o * 3 + 0]; ry = r_edge[o * 3 + 1]; rz = r_edge[o * 3 + 2];
  } else {
    const int i = row_of_slot(rowptr, n_recv, (int)e);
    const int j = col[e];
    rx = xs[(int64_t)j * 3 + 0] - xr[(int64_t)i * 3 + 0];
    ry = xs[(int64_t)j * 3 + 1] - xr[(int64_t)i * 3 + 1];
    rz = xs[(int64_t)j * 3 + 2] - xr[(int64_t)i * 3 + 2];
  }
  const float d = sqrtf((rx * rx + 1e-8f) + (ry * ry + 1e-8f) + (rz * rz + 1e-8f));
  const float ux = rx / d, uy = ry / d, uz = rz / d;
  float gd = 0.f, gux = 0.f, guy = 0.f, guz = 0.f;
  if (d_unit != nullptr) {
    const float4 g = reinterpret_cast<const float4*>(d_unit)[e];
    gux = g.x; guy = g.y; guz = g.z; gd = g.w;
  }
  if (d_basis != nullptr && d < cutoff) {
    const float wgt = edge_wgt != nullptr ? edge_wgt[eid ? eid[e] : e] : 1.0f;
    const float a = 3.14159265358979323846f / cutoff;
    const float env = 0.5f * (cosf(a * d) + 1.0f);
    const float denv = -0.5f * a * sinf(a * d);
    const float* gb = d_basis + e * RB;
    float acc = gb[R] * denv;
    for (int r = 0; r < R; ++r) {
      const float c = coef[r];
      float sn, cs;
      sincosf(c * d, &sn, &cs);
      const float rbf = sn / d;
      const float drbf = (c * cs - rbf) / d;
      acc = fmaf(gb[r], fmaf(drbf, env, rbf * denv), acc);
    }
    gd = fmaf(acc, wgt, gd);
  }
  const float ug = ux * gux + uy * guy + uz * guz;
  dr[o * 3 + 0] = fmaf(gd, ux, (gux - ug * ux) / d);
  dr[o * 3 + 1] = fmaf(gd, uy, (guy - ug * uy) / d);
  dr[o * 3 + 2] = fmaf(gd, uz, (guz - ug * uz) / d);
}

// Coordinate gradients from the per-slot dr (r_e = x_send[j] - x_recv[i]): g_send[j] = sum of dr over the sender CSR row,
// g_recv[i] = -sum of dr over the receiver CSR row, each in CSR order.  same != 0 (one node set, one coordinate tensor):
// g_send[n] = send sum - receive sum, g_recv unused.
__global__ void __launch_bounds__(256) edge_coord_reduce_kernel(
    const float* __restrict__ dr, const int32_t* __restrict__ rowptr, int64_t n_recv, const int32_t* __restrict__ rowptr_t,
    const int32_t* __restrict__ perm_t, int64_t n_send, int same, float* __restrict__ g_send, float* __restrict__ g_recv) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  if (n < n_send) {
    for (int t = rowptr_t[n]; t < rowptr_t[n + 1]; ++t) {
      const int64_t e = perm_t[t];
      sx += dr[e * 3 + 0]; sy += dr[e * 3 + 1]; sz += dr[e * 3 + 2];
    }
  }
  float qx = 0.f, qy = 0.f, qz = 0.f;
  if (n < n_recv) {
    for (int e = rowptr[n]; e < rowptr[n + 1]; ++e) {
      qx += dr[(int64_t)e * 3 + 0]; qy += dr[(int64_t)e * 3 + 1]; qz += dr[(int64_t)e * 3 + 2];
    }
  }
  if (same) {
    if (n < n_send) {
      g_send[n * 3 + 0] = sx - qx; g_send[n * 3 + 1] = sy - qy; g_send[n * 3 + 2] = sz - qz;
    }
    return;
  }
  if (n < n_send) {
    g_send[n * 3 + 0] = sx; g_send[n * 3 + 1] = sy; g_send[n * 3 + 2] = sz;
  }
  if (n < n_recv) {
    g_recv[n * 3 + 0] = -qx; g_recv[n * 3 + 1] = -qy; g_recv[n * 3 + 2] = -qz;
  }
}

// reference layout v[N][F][3] <-> planar v[N][3][F]
__global__ void vec_to_planar_kernel(const float* __restrict__ in, int64_t N, int F, float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // over N*3*F outputs
  if (idx >= N * 3 * (int64_t)F) return;
  const int f = (int)(idx % F);
  const int c = (int)((idx / F) % 3);
  const int64_t n = idx / (3 * (int64_t)F);
  out[idx] = in[(n * F + f) * 3 + c];
}
__global__ void vec_from_planar_kernel(const float* __restrict__ in, int64_t N, int F, float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // over N*F*3 outputs
  if (idx >= N * 3 * (int64_t)F) return;
  const int c = (int)(idx % 3);
  const int f = (int)((idx / 3) % F);
  const int64_t n = idx / (3 * (int64_t)F);
  out[idx] = in[(n * 3 + c) * F + f];
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

int cgvae_edge_geometry(const float* xyz_send, const float* xyz_recv, const float* r_edge, const int32_t* rowptr,
                        const int32_t* col, int64_t n_recv, int64_t n_edges, const float* coef, int R, int RB, float cutoff,
                        const float* edge_wgt, const int32_t* eid, float* basis, float* unit, cgvae_stream_t stream) {
  if (n_edges == 0) return 0;
  CGVAE_REQUIRE(((xyz_send && xyz_recv) || r_edge) && rowptr && col && coef && basis && unit, "edge_geometry: null pointer");
  CGVAE_REQUIRE(R >= 1 && RB >= R + 1 && (RB % 4) == 0, "edge_geometry: need RB %% 4 == 0 and RB >= R+1 (R=%d RB=%d)", R, RB);
  CGVAE_REQUIRE(aligned16(unit) && aligned16(basis), "edge_geometry: outputs must be 16-byte aligned");
  launch_kernel(edge_geometry_kernel, dim3((unsigned)ceil_div(n_edges, 256)), dim3(256), 0, (cudaStream_t)stream, 
      xyz_send, xyz_recv, r_edge, rowptr, col, n_recv, n_edges, coef, R, RB, cutoff, edge_wgt, eid, basis, unit);
  return launched("edge_geometry");
}

int cgvae_edge_geometry_bwd(const float* xyz_send, const float* xyz_recv, const float* r_edge, const int32_t* rowptr,
                            const int32_t* col, int64_t n_recv, int64_t n_edges, const float* coef, int R, int RB, float cutoff,
                            const float* edge_wgt, const int32_t* eid, const float* d_basis, const float* d_unit, float* dr,
                            cgvae_stream_t stream) {
  if (n_edges == 0) return 0;
  CGVAE_REQUIRE(((xyz_send && xyz_recv) || r_edge) && rowptr && col && coef && dr && (r_edge == nullptr || eid),
                "edge_geometry_bwd: null pointer");
  CGVAE_REQUIRE(R >= 1 && RB >= R + 1 && (RB % 4) == 0, "edge_geometry_bwd: need RB %% 4 == 0 and RB >= R+1 (R=%d RB=%d)", R, RB);
  CGVAE_REQUIRE(d_unit == nullptr || aligned16(d_unit), "edge_geometry_bwd: d_unit must be 16-byte aligned");
  launch_kernel(edge_geometry_bwd_kernel, dim3((unsigned)ceil_div(n_edges, 256)), dim3(256), 0, (cudaStream_t)stream, xyz_send,
                xyz_recv, r_edge, rowptr, col, n_recv, n_edges, coef, R, RB, cutoff, edge_wgt, eid, d_basis, d_unit, dr);
  return launched("edge_geometry_bwd");
}

int cgvae_edge_coord_reduce(const float* dr, const int32_t* rowptr, int64_t n_recv, const int32_t* rowptr_t,
                            const int32_t* perm_t, int64_t n_send, int same, float* g_send, float* g_recv,
                            cgvae_stream_t stream) {
  CGVAE_REQUIRE(!same || n_recv == n_send, "edge_coord_reduce: same needs one node set (n_recv=%lld n_send=%lld)",
                (long long)n_recv, (long long)n_send);
  const int64_t n = std::max(n_recv, n_send);
  if (n == 0) return 0;
  CGVAE_REQUIRE(dr && rowptr && rowptr_t && perm_t && g_send && (same || g_recv), "edge_coord_reduce: null pointer");
  launch_kernel(edge_coord_reduce_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, dr, rowptr, n_recv,
                rowptr_t, perm_t, n_send, same, g_send, g_recv);
  return launched("edge_coord_reduce");
}

int cgvae_vec_to_planar(const float* v_nf3, int64_t N, int F, float* v_n3f, cgvae_stream_t stream) {
  if (N == 0) return 0;
  launch_kernel(vec_to_planar_kernel, dim3((unsigned)ceil_div(N * 3 * (int64_t)F, 256)), dim3(256), 0, (cudaStream_t)stream, v_nf3, N, F, v_n3f);
  return launched("vec_to_planar");
}
int cgvae_vec_from_planar(const float* v_n3f, int64_t N, int F, float* v_nf3, cgvae_stream_t stream) {
  if (N == 0) return 0;
  launch_kernel(vec_from_planar_kernel, dim3((unsigned)ceil_div(N * 3 * (int64_t)F, 256)), dim3(256), 0, (cudaStream_t)stream, v_n3f, N, F, v_nf3);
  return launched("vec_from_planar");
}

}  // extern "C"
