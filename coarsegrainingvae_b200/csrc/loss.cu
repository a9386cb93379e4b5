// Loss assembly of the training loop (scripts/utils.py:81-141) and the VAE reparametrisation (cgvae.py:445-449,500-507)
// as a handful of fused launches instead of ~100 element-wise / reduction / index launches:
//
//   vae_latent      sigma = 1e-12 + exp(logvar / 2) ; z = eps * sigma + mu                       (one launch, one backward)
//   std_logvar      y = c + exp(x / 2)   (prior std, cgvae.py:401: c = 1e-9)                     (one launch, one backward)
//   loss_fwd        loss = mean((x_rec - x)^2) + beta * KL + gamma * mean_bonds((|x_rec_a - x_rec_b|_e - |x_a - x_b|_e)^2)
//                   KL = 0.5 * mean_beads( sum_f s1^2/s2^2 + (m1-m2)^2/s2 + log s2^2 - log s1^2 - 1 )   (the `/ s2` quirk of
//                   scripts/utils.py:85 is kept; without a prior the standard-normal KL of :82-83)
//   loss_bwd        gradients to x_rec (per atom, over the bond CSR: deterministic, no index_put / sort), mu, sigma and the
//                   prior mean / std
// Reductions: per-block partial sums in a fixed order, re-reduced by ONE block in block order: deterministic.
// The bond term runs over the receiver CSR of the symmetrised bond list (every bond seen from both atoms): the forward
// halves the doubled sum, the backward needs no scatter.
#include "common.cuh"

namespace cgvae {

constexpr float kBondEps = 1e-6f;      // EPS of scripts/utils.py:27
constexpr int kLossBlocks = 256;       // partial-sum slots per term

__global__ void __launch_bounds__(256) vae_latent_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ logvar,
                                                             const float* __restrict__ eps, int64_t n, float* __restrict__ sigma,
                                                             float* __restrict__ z) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = 1e-12f + expf(logvar[i] * 0.5f);          // cgvae.py:502
  sigma[i] = s;
  if (z) z[i] = fmaf(eps[i], s, mu[i]);                     // cgvae.py:447-448
}
// g_mu = g_z ; g_logvar = (g_sigma + g_z * eps) * d sigma / d logvar,  d sigma / d logvar = 0.5 * exp(logvar / 2)
__global__ void __launch_bounds__(256) vae_latent_bwd_kernel(const float* __restrict__ g_z, const float* __restrict__ g_sigma,
                                                             const float* __restrict__ eps, const float* __restrict__ sigma, int64_t n,
                                                             float* __restrict__ g_mu, float* __restrict__ g_logvar) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gz = g_z ? g_z[i] : 0.f;
  const float gs = (g_sigma ? g_sigma[i] : 0.f) + (eps ? gz * eps[i] : 0.f);
  if (g_mu) g_mu[i] = gz;
  g_logvar[i] = gs * 0.5f * (sigma[i] - 1e-12f);
}

__global__ void __launch_bounds__(256) std_logvar_fwd_kernel(const float* __restrict__ x, int64_t n, float c, float* __restrict__ y) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = c + expf(x[i] * 0.5f);
}
__global__ void __launch_bounds__(256) std_logvar_bwd_kernel(const float* __restrict__ gy, const float* __restrict__ y, int64_t n, float c,
                                                             float* __restrict__ gx) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) gx[i] = gy[i] * 0.5f * (y[i] - c);
}

__device__ __forceinline__ float block_sum_256(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
  }
  __syncthreads();
  return t;       // valid in thread 0
}

// partial[0][b] = sum of squared coordinate errors, partial[1][b] = doubled sum of squared bond-length errors,
// partial[2][b] = sum over (bead, channel) of the KL integrand, each over a fixed slice of the index range
__global__ void __launch_bounds__(256) loss_partial_kernel(
    const float* __restrict__ xyz, const float* __restrict__ xyz_rec, int64_t n_atoms, const int32_t* __restrict__ rowptr,
    const int32_t* __restrict__ col, const float* __restrict__ mu, const float* __restrict__ sigma, const float* __restrict__ pmu,
    const float* __restrict__ pstd, int64_t n_lat, float* __restrict__ partial) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ float red[8];
  const int nb = gridDim.x;
  // ---- coordinates and bonds: atoms of this block's slice
  {
    const int64_t per = (n_atoms + nb - 1) / nb;
    const int64_t a0 = (int64_t)blockIdx.x * per, a1 = min(n_atoms, a0 + per);
    float s_rec = 0.f, s_bond = 0.f;
    for (int64_t a = a0 + threadIdx.x; a < a1; a += 256) {
      const float xa = xyz[3 * a], ya = xyz[3 * a + 1], za = xyz[3 * a + 2];
      const float xr = xyz_rec[3 * a], yr = xyz_rec[3 * a + 1], zr = xyz_rec[3 * a + 2];
      s_rec += (xr - xa) * (xr - xa) + (yr - ya) * (yr - ya) + (zr - za) * (zr - za);
      if (rowptr != nullptr) {
        for (int t = rowptr[a]; t < rowptr[a + 1]; ++t) {
          const int64_t b = col[t];
          const float dx = xr - xyz_rec[3 * b], dy = yr - xyz_rec[3 * b + 1], dz = zr - xyz_rec[3 * b + 2];
          const float ex = xa - xyz[3 * b], ey = ya - xyz[3 * b + 1], ez = za - xyz[3 * b + 2];
          const float gen = sqrtf(dx * dx + dy * dy + dz * dz + kBondEps);
          const float dat = sqrtf(ex * ex + ey * ey + ez * ez + kBondEps);
          s_bond += (gen - dat) * (gen - dat);
        }
      }
    }
    const float t0 = block_sum_256(s_rec, red);
    const float t1 = block_sum_256(s_bond, red);
    if (threadIdx.x == 0) {
      partial[blockIdx.x] = t0;
      partial[nb + blockIdx.x] = t1;
    }
  }
  // ---- KL integrand
  {
    const int64_t per = (n_lat + nb - 1) / nb;
    const int64_t i0 = (int64_t)blockIdx.x * per, i1 = min(n_lat, i0 + per);
    float s_kl = 0.f;
    if (mu != nullptr) {
      for (int64_t i = i0 + threadIdx.x; i < i1; i += 256) {
        const float m1 = mu[i], s1 = sigma[i];
        if (pmu != nullptr) {
          const float m2 = pmu[i], s2 = pstd[i];
          const float d = m1 - m2;
          s_kl += (s1 * s1) / (s2 * s2) + d * d / s2 + logf(s2 * s2) - logf(s1 * s1) - 1.0f;      // utils.py:85-86
        } else {
          s_kl += -(1.0f + logf(s1 * s1) - m1 * m1 - s1 * s1);                                     // utils.py:82-83 (x 0.5 below)
        }
      }
    }
    const float t2 = block_sum_256(s_kl, red);
    if (threadIdx.x == 0) partial[2 * nb + blockIdx.x] = t2;
  }
}

// out[0] = loss, out[1] = recon, out[2] = kl, out[3] = graph.  norms (nullable, device float[3]) = denominators (atoms, beads,
// bonds) as GLOBAL count / world for data-parallel training; otherwise the local counts (bond count from the CSR).
__global__ void __launch_bounds__(256) loss_final_kernel(const float* __restrict__ partial, int nb, int64_t n_atoms, int64_t n_beads,
                                                         const int32_t* __restrict__ rowptr, const float* __restrict__ norms,
                                                         float beta, float gamma, int has_kl, float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ float red[8];
  float s[3] = {0.f, 0.f, 0.f};
  for (int t = 0; t < 3; ++t) {
    float v = 0.f;
    for (int b = threadIdx.x; b < nb; b += 256) v += partial[t * nb + b];
    s[t] = block_sum_256(v, red);
  }
  if (threadIdx.x == 0) {
    const float n_at = norms ? norms[0] : (float)n_atoms;
    const float n_bd = norms ? norms[1] : (float)n_beads;
    const float n_bo = norms ? norms[2] : (rowptr ? 0.5f * (float)rowptr[n_atoms] : 1.0f);
    const float recon = s[0] / (3.0f * n_at);
    const float graph = (rowptr && gamma != 0.f) ? 0.5f * s[1] / fmaxf(n_bo, 1e-30f) : 0.f;
    const float kl = has_kl ? 0.5f * s[2] / n_bd : 0.f;
    out[0] = recon + kl * beta + graph * gamma;
    out[1] = recon;
    out[2] = kl;
    out[3] = graph;
  }
}

// g_xyz_rec[a] = g * ( 2 (x_rec_a - x_a) / (3 n_atoms) + gamma / n_bonds * sum_b 2 (gen - dat) / gen * (x_rec_a - x_rec_b) )
__global__ void __launch_bounds__(256) loss_bwd_xyz_kernel(const float* __restrict__ g_loss, const float* __restrict__ xyz,
                                                           const float* __restrict__ xyz_rec, int64_t n_atoms,
                                                           const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                           const float* __restrict__ norms, float gamma, float* __restrict__ g_rec) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_atoms) return;
  const float g = g_loss[0];
  const float n_at = norms ? norms[0] : (float)n_atoms;
  const float xa = xyz[3 * a], ya = xyz[3 * a + 1], za = xyz[3 * a + 2];
  const float xr = xyz_rec[3 * a], yr = xyz_rec[3 * a + 1], zr = xyz_rec[3 * a + 2];
  const float cr = 2.0f / (3.0f * n_at);
  float gx = cr * (xr - xa), gy = cr * (yr - ya), gz = cr * (zr - za);
  if (rowptr != nullptr && gamma != 0.f) {
    const float n_bo = norms ? norms[2] : 0.5f * (float)rowptr[n_atoms];
    const float cb = gamma / fmaxf(n_bo, 1e-30f);
    float bx = 0.f, by = 0.f, bz = 0.f;
    for (int t = rowptr[a]; t < rowptr[a + 1]; ++t) {
      const int64_t b = col[t];
      const float dx = xr - xyz_rec[3 * b], dy = yr - xyz_rec[3 * b + 1], dz = zr - xyz_rec[3 * b + 2];
      const float ex = xa - xyz[3 * b], ey = ya - xyz[3 * b + 1], ez = za - xyz[3 * b + 2];
      const float gen = sqrtf(dx * dx + dy * dy + dz * dz + kBondEps);
      const float dat = sqrtf(ex * ex + ey * ey + ez * ez + kBondEps);
      const float k = 2.0f * (gen - dat) / gen;
      bx = fmaf(k, dx, bx); by = fmaf(k, dy, by); bz = fmaf(k, dz, bz);
    }
    gx = fmaf(cb, bx, gx); gy = fmaf(cb, by, gy); gz = fmaf(cb, bz, gz);
  }
  g_rec[3 * a] = g * gx;
  g_rec[3 * a + 1] = g * gy;
  g_rec[3 * a + 2] = g * gz;
}

// gradient to the TARGET coordinates (xyz is also the encoder input when coordinates are differentiated):
// g_xyz[a] = g * ( -2 (x_rec_a - x_a) / (3 n_atoms) - gamma / n_bonds * sum_b 2 (gen - dat) / dat * (x_a - x_b) )
__global__ void __launch_bounds__(256) loss_bwd_target_kernel(const float* __restrict__ g_loss, const float* __restrict__ xyz,
                                                              const float* __restrict__ xyz_rec, int64_t n_atoms,
                                                              const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                              const float* __restrict__ norms, float gamma, float* __restrict__ g_xyz) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_atoms) return;
  const float g = g_loss[0];
  const float n_at = norms ? norms[0] : (float)n_atoms;
  const float xa = xyz[3 * a], ya = xyz[3 * a + 1], za = xyz[3 * a + 2];
  const float xr = xyz_rec[3 * a], yr = xyz_rec[3 * a + 1], zr = xyz_rec[3 * a + 2];
  const float cr = 2.0f / (3.0f * n_at);
  float gx = cr * (xa - xr), gy = cr * (ya - yr), gz = cr * (za - zr);
  if (rowptr != nullptr && gamma != 0.f) {
    const float n_bo = norms ? norms[2] : 0.5f * (float)rowptr[n_atoms];
    const float cb = gamma / fmaxf(n_bo, 1e-30f);
    float bx = 0.f, by = 0.f, bz = 0.f;
    for (int t = rowptr[a]; t < rowptr[a + 1]; ++t) {
      const int64_t b = col[t];
      const float dx = xr - xyz_rec[3 * b], dy = yr - xyz_rec[3 * b + 1], dz = zr - xyz_rec[3 * b + 2];
      const float ex = xa - xyz[3 * b], ey = ya - xyz[3 * b + 1], ez = za - xyz[3 * b + 2];
      const float gen = sqrtf(dx * dx + dy * dy + dz * dz + kBondEps);
      const float dat = sqrtf(ex * ex + ey * ey + ez * ez + kBondEps);
      const float k = 2.0f * (dat - gen) / dat;
      bx = fmaf(k, ex, bx); by = fmaf(k, ey, by); bz = fmaf(k, ez, bz);
    }
    gx = fmaf(cb, bx, gx); gy = fmaf(cb, by, gy); gz = fmaf(cb, bz, gz);
  }
  g_xyz[3 * a] = g * gx;
  g_xyz[3 * a + 1] = g * gy;
  g_xyz[3 * a + 2] = g * gz;
}

// gradients of beta * KL to (mu, sigma, prior mean, prior std)
__global__ void __launch_bounds__(256) loss_bwd_kl_kernel(const float* __restrict__ g_loss, const float* __restrict__ mu,
                                                          const float* __restrict__ sigma, const float* __restrict__ pmu,
                                                          const float* __restrict__ pstd, int64_t n_lat, int64_t n_beads,
                                                          const float* __restrict__ norms, float beta, float* __restrict__ g_mu,
                                                          float* __restrict__ g_sigma, float* __restrict__ g_pmu, float* __restrict__ g_pstd) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_lat) return;
  const float n_bd = norms ? norms[1] : (float)n_beads;
  const float c = g_loss[0] * beta * 0.5f / n_bd;
  const float m1 = mu[i], s1 = sigma[i];
  if (pmu != nullptr) {
    const float m2 = pmu[i], s2 = pstd[i];
    const float d = m1 - m2;
    g_mu[i] = c * 2.0f * d / s2;
    g_sigma[i] = c * (2.0f * s1 / (s2 * s2) - 2.0f / s1);
    g_pmu[i] = -c * 2.0f * d / s2;
    g_pstd[i] = c * (-2.0f * s1 * s1 / (s2 * s2 * s2) - d * d / (s2 * s2) + 2.0f / s2);
  } else {
    g_mu[i] = c * 2.0f * m1;
    g_sigma[i] = c * (2.0f * s1 - 2.0f / s1);
  }
}

__global__ void __launch_bounds__(256) fill_kernel(float* __restrict__ p, int64_t n, float value) {
  CGVAE_KERNEL_PROLOGUE();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = value;
}

// ---- dihedral loss of the PCN loop (scripts/pcn_utils.py:114-132,178-180) ------------------------------------------------------
// theta(x; i0..i3) = atan(p1 / (p2 + EPS)),  b1 = x1 - x0, b2 = x2 - x1, b3 = x3 - x2, c1 = b2 x b3, c2 = b1 x b2,
// p1 = (b1 . c1) * sqrt(b2 . b2 + EPS),  p2 = c1 . c2  -- the reference's formula, EPS quirks included (arctan, not atan2).
struct Vec3 {
  float x, y, z;
};
__device__ __forceinline__ Vec3 v3(const float* p) { return Vec3{p[0], p[1], p[2]}; }
__device__ __forceinline__ Vec3 operator-(Vec3 a, Vec3 b) { return Vec3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ Vec3 operator+(Vec3 a, Vec3 b) { return Vec3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ Vec3 operator*(float s, Vec3 a) { return Vec3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ float dot3(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ Vec3 cross3(Vec3 a, Vec3 b) { return Vec3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

// angle and (optionally) its gradient with respect to the four positions
__device__ __forceinline__ float dihedral(const float* __restrict__ xyz, const int64_t* __restrict__ q, Vec3* g) {
  constexpr float EPS = 1e-6f;
  const Vec3 x0 = v3(xyz + 3 * q[0]), x1 = v3(xyz + 3 * q[1]), x2 = v3(xyz + 3 * q[2]), x3 = v3(xyz + 3 * q[3]);
  const Vec3 b1 = x1 - x0, b2 = x2 - x1, b3 = x3 - x2;
  const Vec3 c1 = cross3(b2, b3), c2 = cross3(b1, b2);
  const float u = dot3(b1, c1), nrm = sqrtf(dot3(b2, b2) + EPS);
  const float p1 = u * nrm, p2 = dot3(c1, c2), den = p2 + EPS, t = p1 / den;
  if (g != nullptr) {
    const float dt = 1.0f / (1.0f + t * t);
    const float g_p1 = dt / den, g_p2 = -dt * p1 / (den * den);
    // p1 = u * nrm ; u = b1 . c1 ; nrm = sqrt(b2 . b2 + EPS) ; p2 = c1 . c2
    const float g_u = g_p1 * nrm, g_n = g_p1 * u;
    Vec3 g_b1 = g_u * c1, g_c1 = g_u * b1 + g_p2 * c2, g_c2 = g_p2 * c1;
    Vec3 g_b2 = (g_n / nrm) * b2;
    // c1 = b2 x b3 : g_b2 += b3 x g_c1, g_b3 = g_c1 x b2 ;  c2 = b1 x b2 : g_b1 += b2 x g_c2, g_b2 += g_c2 x b1
    g_b2 = g_b2 + cross3(b3, g_c1) + cross3(g_c2, b1);
    const Vec3 g_b3 = cross3(g_c1, b2);
    g_b1 = g_b1 + cross3(b2, g_c2);
    g[0] = -1.0f * g_b1;
    g[1] = g_b1 - g_b2;
    g[2] = g_b2 - g_b3;
    g[3] = g_b3;
  }
  return atanf(t);
}

// per dihedral: diff = theta(rec) - theta(xyz); contrib[d][slot] = 2 diff dtheta/dx_slot (unscaled); block partial of diff^2
__global__ void __launch_bounds__(256) dihedral_fwd_kernel(const float* __restrict__ xyz, const float* __restrict__ rec,
                                                           const int64_t* __restrict__ idx, int64_t n_dihe, const int64_t* __restrict__ n_live,
                                                           float* __restrict__ contrib, float* __restrict__ partial) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ float red[8];
  const int64_t n = n_live ? min(*n_live, n_dihe) : n_dihe;
  float acc = 0.f;
  for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d < n_dihe; d += (int64_t)gridDim.x * blockDim.x) {
    Vec3 g[4] = {Vec3{0.f, 0.f, 0.f}, Vec3{0.f, 0.f, 0.f}, Vec3{0.f, 0.f, 0.f}, Vec3{0.f, 0.f, 0.f}};
    if (d < n) {
      const float diff = dihedral(rec, idx + 4 * d, g) - dihedral(xyz, idx + 4 * d, nullptr);
      acc += diff * diff;
#pragma unroll
      for (int s = 0; s < 4; ++s) g[s] = (2.0f * diff) * g[s];
    }
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      contrib[(d * 4 + s) * 3 + 0] = g[s].x;
      contrib[(d * 4 + s) * 3 + 1] = g[s].y;
      contrib[(d * 4 + s) * 3 + 2] = g[s].z;
    }
  }
  acc = block_sum_256(acc, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
// out[0] = mean over the live dihedrals (fixed-order sum of the block partials)
__global__ void __launch_bounds__(256) dihedral_final_kernel(const float* __restrict__ partial, int nb, int64_t n_dihe,
                                                             const int64_t* __restrict__ n_live, const float* __restrict__ norm,
                                                             float* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ float red[8];
  float v = 0.f;
  for (int i = threadIdx.x; i < nb; i += 256) v += partial[i];
  v = block_sum_256(v, red);
  if (threadIdx.x == 0) {
    const float n = norm ? *norm : (float)(n_live ? min(*n_live, n_dihe) : n_dihe);
    out[0] = v / fmaxf(n, 1.0f);
  }
}
// per atom: g_rec[a] = g_loss / n * sum over the (dihedral, slot) entries that name atom a (CSR of the flattened index list)
__global__ void __launch_bounds__(256) dihedral_bwd_kernel(const float* __restrict__ g_loss, const float* __restrict__ contrib,
                                                           const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                           int64_t n_atoms, int64_t n_dihe, const int64_t* __restrict__ n_live,
                                                           const float* __restrict__ norm, float* __restrict__ g_rec) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_atoms) return;
  const float n = norm ? *norm : (float)(n_live ? min(*n_live, n_dihe) : n_dihe);
  const float scale = g_loss[0] / fmaxf(n, 1.0f);
  float gx = 0.f, gy = 0.f, gz = 0.f;
  for (int j = rowptr[a]; j < rowptr[a + 1]; ++j) {
    const int64_t e = col[j];
    gx += contrib[e * 3 + 0];
    gy += contrib[e * 3 + 1];
    gz += contrib[e * 3 + 2];
  }
  g_rec[a * 3 + 0] = scale * gx;
  g_rec[a * 3 + 1] = scale * gy;
  g_rec[a * 3 + 2] = scale * gz;
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

int cgvae_vae_latent_fwd(const float* mu, const float* logvar, const float* eps, int64_t n, float* sigma, float* z,
                         cgvae_stream_t stream) {
  if (n == 0) return 0;
  CGVAE_REQUIRE(logvar && sigma && (!z || (mu && eps)), "vae_latent_fwd: null pointer");
  launch_kernel(vae_latent_fwd_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, mu, logvar, eps, n, sigma, z);
  return launched("vae_latent_fwd");
}
int cgvae_vae_latent_bwd(const float* g_z, const float* g_sigma, const float* eps, const float* sigma, int64_t n, float* g_mu,
                         float* g_logvar, cgvae_stream_t stream) {
  if (n == 0) return 0;
  CGVAE_REQUIRE(sigma && g_logvar, "vae_latent_bwd: null pointer");
  launch_kernel(vae_latent_bwd_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, g_z, g_sigma, eps, sigma, n, g_mu,
                g_logvar);
  return launched("vae_latent_bwd");
}
int cgvae_std_logvar_fwd(const float* x, int64_t n, float c, float* y, cgvae_stream_t stream) {
  if (n == 0) return 0;
  CGVAE_REQUIRE(x && y, "std_logvar_fwd: null pointer");
  launch_kernel(std_logvar_fwd_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, x, n, c, y);
  return launched("std_logvar_fwd");
}
int cgvae_std_logvar_bwd(const float* gy, const float* y, int64_t n, float c, float* gx, cgvae_stream_t stream) {
  if (n == 0) return 0;
  CGVAE_REQUIRE(gy && y && gx, "std_logvar_bwd: null pointer");
  launch_kernel(std_logvar_bwd_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, gy, y, n, c, gx);
  return launched("std_logvar_bwd");
}

int cgvae_fill(float* p, int64_t n, float value, cgvae_stream_t stream) {
  if (n == 0) return 0;
  CGVAE_REQUIRE(p, "fill: null pointer");
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(n, 256), (int64_t)kNumSM * 8);
  launch_kernel(fill_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, p, n, value);
  return launched("fill");
}

size_t cgvae_loss_ws_bytes(void) { return sizeof(float) * 3 * kLossBlocks; }

int cgvae_loss_fwd(const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr, const int32_t* bond_col,
                   const float* mu, const float* sigma, const float* pmu, const float* pstd, int64_t n_beads, int F,
                   const float* norms, float beta, float gamma, float* out4, void* ws, size_t ws_bytes, cgvae_stream_t stream) {
  CGVAE_REQUIRE(xyz && xyz_rec && out4 && n_atoms > 0, "loss_fwd: null pointer / no atoms");
  CGVAE_REQUIRE((mu == nullptr) == (sigma == nullptr) && (pmu == nullptr) == (pstd == nullptr), "loss_fwd: mu / sigma and prior mean / std come in pairs");
  CGVAE_REQUIRE(ws && ws_bytes >= cgvae_loss_ws_bytes(), "loss_fwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = reinterpret_cast<float*>(ws);
  const int nb = kLossBlocks;
  launch_kernel(loss_partial_kernel, dim3(nb), dim3(256), 0, st, xyz, xyz_rec, n_atoms, bond_rowptr, bond_col, mu, sigma, pmu, pstd,
                (int64_t)n_beads * F, partial);
  if (int rc = launched("loss_partial")) return rc;
  launch_kernel(loss_final_kernel, dim3(1), dim3(256), 0, st, (const float*)partial, nb, n_atoms, n_beads, bond_rowptr, norms, beta, gamma,
                mu != nullptr ? 1 : 0, out4);
  return launched("loss_final");
}

int cgvae_loss_bwd(const float* g_loss, const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr,
                   const int32_t* bond_col, const float* mu, const float* sigma, const float* pmu, const float* pstd,
                   int64_t n_beads, int F, const float* norms, float beta, float gamma, float* g_xyz_rec, float* g_mu,
                   float* g_sigma, float* g_pmu, float* g_pstd, cgvae_stream_t stream) {
  CGVAE_REQUIRE(g_loss && xyz && xyz_rec && g_xyz_rec && n_atoms > 0, "loss_bwd: null pointer / no atoms");
  cudaStream_t st = (cudaStream_t)stream;
  launch_kernel(loss_bwd_xyz_kernel, dim3((unsigned)ceil_div(n_atoms, 256)), dim3(256), 0, st, g_loss, xyz, xyz_rec, n_atoms, bond_rowptr,
                bond_col, norms, gamma, g_xyz_rec);
  if (int rc = launched("loss_bwd_xyz")) return rc;
  if (mu != nullptr) {
    CGVAE_REQUIRE(sigma && g_mu && g_sigma && (pmu == nullptr || (pstd && g_pmu && g_pstd)), "loss_bwd: null pointer (KL term)");
    const int64_t n_lat = (int64_t)n_beads * F;
    launch_kernel(loss_bwd_kl_kernel, dim3((unsigned)ceil_div(n_lat, 256)), dim3(256), 0, st, g_loss, mu, sigma, pmu, pstd, n_lat, n_beads,
                  norms, beta, g_mu, g_sigma, g_pmu, g_pstd);
    return launched("loss_bwd_kl");
  }
  return 0;
}


/* Dihedral loss (scripts/pcn_utils.py:114-132,178-180): out[0] = mean_d (theta(rec; idx[d]) - theta(xyz; idx[d]))^2.
 * contrib [n_dihe][4][3]: unscaled per-(dihedral, slot) gradients kept for the backward; ws: 256 floats. */
int cgvae_loss_bwd_target(const float* g_loss, const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr,
                          const int32_t* bond_col, const float* norms, float gamma, float* g_xyz, cgvae_stream_t stream) {
  CGVAE_REQUIRE(g_loss && xyz && xyz_rec && g_xyz && n_atoms > 0, "loss_bwd_target: null pointer / no atoms");
  launch_kernel(loss_bwd_target_kernel, dim3((unsigned)ceil_div(n_atoms, 256)), dim3(256), 0, (cudaStream_t)stream, g_loss, xyz,
                xyz_rec, n_atoms, bond_rowptr, bond_col, norms, gamma, g_xyz);
  return launched("loss_bwd_target");
}

int cgvae_dihedral_loss_fwd(const float* xyz, const float* xyz_rec, const int64_t* idx, int64_t n_dihe, const int64_t* n_live,
                            const float* norm, float* contrib, float* out, void* ws, size_t ws_bytes, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CGVAE_REQUIRE(out && ws && ws_bytes >= sizeof(float) * kLossBlocks, "dihedral_loss_fwd: workspace too small");
  CGVAE_REQUIRE(n_dihe == 0 || (xyz && xyz_rec && idx && contrib), "dihedral_loss_fwd: null pointer");
  const int nb = (int)std::max<int64_t>(1, std::min<int64_t>(kLossBlocks, ceil_div(n_dihe, 256)));
  float* partial = reinterpret_cast<float*>(ws);
  launch_kernel(dihedral_fwd_kernel, dim3(nb), dim3(256), 0, st, xyz, xyz_rec, idx, n_dihe, n_live, contrib, partial);
  launch_kernel(dihedral_final_kernel, dim3(1), dim3(256), 0, st, (const float*)partial, nb, n_dihe, n_live, norm, out);
  return launched("dihedral_loss_fwd");
}
int cgvae_dihedral_loss_bwd(const float* g_loss, const float* contrib, const int32_t* rowptr, const int32_t* col, int64_t n_atoms,
                            int64_t n_dihe, const int64_t* n_live, const float* norm, float* g_xyz_rec, cgvae_stream_t stream) {
  if (n_atoms == 0) return 0;
  CGVAE_REQUIRE(g_loss && rowptr && g_xyz_rec && (n_dihe == 0 || (contrib && col)), "dihedral_loss_bwd: null pointer");
  launch_kernel(dihedral_bwd_kernel, dim3((unsigned)ceil_div(n_atoms, 256)), dim3(256), 0, (cudaStream_t)stream, g_loss, contrib, rowptr,
                col, n_atoms, n_dihe, n_live, norm, g_xyz_rec);
  return launched("dihedral_loss_bwd");
}

}  // extern "C"
