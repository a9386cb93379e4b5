// Integer / index kernels: radius graph (cell list + tiled brute force, bit-exact, sorted),
// scans, CSR construction, segment ranks.  See include/cgvae_b200.h for the contract.
#include "common.cuh"
#include <limits.h>

namespace cgvae {

thread_local char g_err[512] = {0};
std::atomic<unsigned long long> g_launches{0};
std::atomic<int32_t*> g_err_flags[kMaxDevices];

// Programmatic dependent launch: on by default since round 2.  On its own it changed the captured step by < 1 % (dependent-node
// gaps are ~0.35 us already); what pays is what it enables: the weight-streaming GEMMs issue the bulk copies of a registered
// parameter matrix BEFORE their dependency wait (gemm_stream.cu), 2.93 -> 2.81 ms per chignolin step.  It inflates the
// per-kernel durations a profiler reports (a dependent grid is resident while it waits), so bench.py takes its kernel timeline
// from a second capture with cgvae_set_pdl(0).  CGVAE_PDL=0 disables it.
static std::atomic<int> g_pdl{-1};
bool pdl_enabled() {
  int v = g_pdl.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("CGVAE_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
    g_pdl.store(v, std::memory_order_relaxed);
  }
  return v != 0;
}

// Matmul precision of the tensor-core contractions (cgvae_set_matmul_precision): 0 = 3xTF32 (default), 1 = 1xTF32.
// Read by the dispatchers at every launch; a captured CUDA graph keeps the kernels it was captured with.
static std::atomic<int> g_matmul_precision{0};
int matmul_precision() { return g_matmul_precision.load(std::memory_order_relaxed); }

// ------------------------------------------------------------------------------------------
// scans (single CTA, 1024 threads x 8 items per sweep; inputs here are <= a few 1e5 long)
// ------------------------------------------------------------------------------------------
template <typename TOut>
__global__ void __launch_bounds__(1024) scan_kernel(const int32_t* __restrict__ in, int64_t n, TOut* __restrict__ out) {
  CGVAE_KERNEL_PROLOGUE();
  constexpr int ITEMS = 8;
  __shared__ long long warp_tot[32];
  __shared__ long long carry_sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_sh = 0;
  __syncthreads();
  for (int64_t base = 0; base < n; base += 1024 * ITEMS) {
    const int64_t i0 = base + (int64_t)threadIdx.x * ITEMS;
    int v[ITEMS];
    long long tsum = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      v[k] = (i0 + k < n) ? in[i0 + k] : 0;
      tsum += v[k];
    }
    long long x = tsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      long long y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
      long long w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        long long y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    long long excl = carry_sh + (warp ? warp_tot[warp - 1] : 0) + (x - tsum);
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      if (i0 + k < n) out[i0 + k] = (TOut)excl;
      excl += v[k];
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_sh += warp_tot[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = (TOut)carry_sh;
}

// ------------------------------------------------------------------------------------------
// warp-level sorting of short rows in shared memory
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_bitonic(int* a, int P, int lane) {
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < (P >> 1); t += 32) {
        const int i = ((t / j) * 2 * j) + (t % j);
        const int l = i + j;
        const bool up = ((i & k) == 0);
        const int x = a[i], y = a[l];
        if ((x > y) == up) { a[i] = y; a[l] = x; }
      }
      __syncwarp();
    }
  }
}
__device__ __forceinline__ int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

constexpr int kSortCap = 2048;     // ints per warp in shared memory
constexpr int kSortWarps = 4;      // warps per CTA in the sorting kernels

// sort each row (rowptr) of `data` ascending; rows longer than kSortCap fall back to an in-place
// odd-even transposition sort in global memory (correct, slow, not expected in practice).
__global__ void __launch_bounds__(kSortWarps * 32) sort_rows_kernel(const int32_t* __restrict__ rowptr, int64_t n_rows,
                                                                    int32_t* __restrict__ data) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ int buf[kSortWarps][kSortCap];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * kSortWarps + warp;
  if (row >= n_rows) return;
  const int beg = rowptr[row], L = rowptr[row + 1] - beg;
  if (L <= 1) return;
  int32_t* d = data + beg;
  if (L <= kSortCap) {
    const int P = next_pow2(L);
    for (int t = lane; t < P; t += 32) buf[warp][t] = (t < L) ? d[t] : INT_MAX;
    __syncwarp();
    warp_bitonic(buf[warp], P, lane);
    for (int t = lane; t < L; t += 32) d[t] = buf[warp][t];
  } else {
    for (int phase = 0; phase < L; ++phase) {
      for (int t = lane; 2 * t + (phase & 1) + 1 < L; t += 32) {
        const int i = 2 * t + (phase & 1);
        const int x = d[i], y = d[i + 1];
        if (x > y) { d[i] = y; d[i + 1] = x; }
      }
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------------
// radius graph
// ------------------------------------------------------------------------------------------
struct FrameInfo {
  float minx, miny, minz;
  int nx, ny, nz;
  int cell_base;
  int pad;
  double inv_h;
};

// the reference's fp32 recipe (data.py:71-72): ((dx*dx + dy*dy) + dz*dz), IEEE sqrt, no FMA contraction
__device__ __forceinline__ bool within_cutoff(float xi, float yi, float zi, float xj, float yj, float zj, float cutoff) {
  const float dx = __fsub_rn(xj, xi), dy = __fsub_rn(yj, yi), dz = __fsub_rn(zj, zi);
  const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
  return __fsqrt_rn(d2) <= cutoff;
}

__device__ __forceinline__ int frame_of(const int64_t* __restrict__ frame_ptr, int64_t n_frames, int64_t atom) {
  int64_t lo = 0, hi = n_frames;  // largest f with frame_ptr[f] <= atom
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (frame_ptr[mid] <= atom) lo = mid; else hi = mid;
  }
  return (int)lo;
}

struct RadiusWs {
  FrameInfo* frames;
  int32_t* frame_of_atom;
  int32_t* cell_of_atom;
  int32_t* cell_atoms;
  int32_t* cell_start;   // max_cells + 1
  int32_t* cell_count;   // max_cells (count, then cursor)
  int64_t max_cells;
};

static inline size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }

static size_t radius_ws_layout(int64_t n, int64_t n_frames, char* base, RadiusWs* out) {
  const int64_t max_cells = 8 * n + 64 * n_frames;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  size_t o_frames = take(sizeof(FrameInfo) * (size_t)n_frames);
  size_t o_foa = take(4 * (size_t)n);
  size_t o_coa = take(4 * (size_t)n);
  size_t o_ca = take(4 * (size_t)n);
  size_t o_cs = take(4 * (size_t)(max_cells + 1));
  size_t o_cc = take(4 * (size_t)max_cells);
  if (out) {
    out->frames = reinterpret_cast<FrameInfo*>(base + o_frames);
    out->frame_of_atom = reinterpret_cast<int32_t*>(base + o_foa);
    out->cell_of_atom = reinterpret_cast<int32_t*>(base + o_coa);
    out->cell_atoms = reinterpret_cast<int32_t*>(base + o_ca);
    out->cell_start = reinterpret_cast<int32_t*>(base + o_cs);
    out->cell_count = reinterpret_cast<int32_t*>(base + o_cc);
    out->max_cells = max_cells;
  }
  return off;
}

// one CTA per frame: bounding box -> cell grid (edge >= cutoff, total cells <= 8 n_f + 64)
__global__ void __launch_bounds__(256) frame_bounds_kernel(const float* __restrict__ xyz, const int64_t* __restrict__ frame_ptr,
                                                           float cutoff, FrameInfo* __restrict__ frames) {
  CGVAE_KERNEL_PROLOGUE();
  const int f = blockIdx.x;
  const int64_t beg = frame_ptr[f], end = frame_ptr[f + 1];
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t a = beg + threadIdx.x; a < end; a += blockDim.x) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float x = xyz[a * 3 + c];
      mn[c] = fminf(mn[c], x);
      mx[c] = fmaxf(mx[c], x);
    }
  }
  __shared__ float smn[3][8], smx[3][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[c] = fminf(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o));
      mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o));
    }
    if (lane == 0) { smn[c][warp] = mn[c]; smx[c][warp] = mx[c]; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    FrameInfo fi;
    double ext[3];
    float lo[3];
    for (int c = 0; c < 3; ++c) {
      float a = smn[c][0], b = smx[c][0];
      for (int w = 1; w < 8; ++w) { a = fminf(a, smn[c][w]); b = fmaxf(b, smx[c][w]); }
      if (end <= beg) { a = 0.f; b = 0.f; }
      lo[c] = a;
      ext[c] = (double)b - (double)a;
    }
    double h = (double)cutoff * (1.0 + 1e-6);
    if (!(h > 0.0)) h = 1.0;
    const double cap = 8.0 * (double)(end - beg) + 64.0;
    int nx, ny, nz;
    for (;;) {
      nx = (int)floor(ext[0] / h) + 1; ny = (int)floor(ext[1] / h) + 1; nz = (int)floor(ext[2] / h) + 1;
      if ((double)nx * (double)ny * (double)nz <= cap) break;
      h *= 1.2599210498948732;  // doubles the cell volume
    }
    fi.minx = lo[0]; fi.miny = lo[1]; fi.minz = lo[2];
    fi.nx = nx; fi.ny = ny; fi.nz = nz;
    fi.cell_base = nx * ny * nz;  // turned into an offset by frame_offsets_kernel
    fi.pad = 0;
    fi.inv_h = 1.0 / h;
    frames[f] = fi;
  }
}

__global__ void frame_offsets_kernel(FrameInfo* frames, int64_t n_frames) {
  CGVAE_KERNEL_PROLOGUE();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int run = 0;
    for (int64_t f = 0; f < n_frames; ++f) {
      const int c = frames[f].cell_base;
      frames[f].cell_base = run;
      run += c;
    }
  }
}

__device__ __forceinline__ void cell_coords(const FrameInfo& fi, float x, float y, float z, int& cx, int& cy, int& cz) {
  cx = min(fi.nx - 1, max(0, (int)floor(((double)x - (double)fi.minx) * fi.inv_h)));
  cy = min(fi.ny - 1, max(0, (int)floor(((double)y - (double)fi.miny) * fi.inv_h)));
  cz = min(fi.nz - 1, max(0, (int)floor(((double)z - (double)fi.minz) * fi.inv_h)));
}

__global__ void assign_cells_kernel(const float* __restrict__ xyz, int64_t n, const int64_t* __restrict__ frame_ptr,
                                    int64_t n_frames, const FrameInfo* __restrict__ frames, int32_t* __restrict__ frame_of_atom,
                                    int32_t* __restrict__ cell_of_atom, int32_t* __restrict__ cell_count) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n) return;
  const int f = frame_of(frame_ptr, n_frames, a);
  const FrameInfo fi = frames[f];
  int cx, cy, cz;
  cell_coords(fi, xyz[a * 3], xyz[a * 3 + 1], xyz[a * 3 + 2], cx, cy, cz);
  const int cell = fi.cell_base + (cz * fi.ny + cy) * fi.nx + cx;
  frame_of_atom[a] = f;
  cell_of_atom[a] = cell;
  atomicAdd(&cell_count[cell], 1);
}

__global__ void fill_cells_kernel(int64_t n, const int32_t* __restrict__ cell_of_atom, const int32_t* __restrict__ cell_start,
                                  int32_t* __restrict__ cursor, int32_t* __restrict__ cell_atoms) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n) return;
  const int c = cell_of_atom[a];
  cell_atoms[cell_start[c] + atomicAdd(&cursor[c], 1)] = (int32_t)a;
}

constexpr int kRadWarps = 4;

// warp per atom.  FILL=false: deg[i] = number of neighbours.  FILL=true: writes the sorted row.
template <bool FILL, bool CELLS>
__global__ void __launch_bounds__(kRadWarps * 32) radius_query_kernel(
    const float* __restrict__ xyz, int64_t n, const int64_t* __restrict__ frame_ptr, int64_t n_frames, float cutoff,
    int undirected, RadiusWs ws, int32_t* __restrict__ deg, const int64_t* __restrict__ rowptr, int64_t* __restrict__ out_pairs) {
  CGVAE_KERNEL_PROLOGUE();
  __shared__ int buf[FILL ? kRadWarps : 1][FILL ? kSortCap : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * kRadWarps + warp;
  if (i >= n) return;
  const float xi = xyz[i * 3], yi = xyz[i * 3 + 1], zi = xyz[i * 3 + 2];
  const int f = CELLS ? ws.frame_of_atom[i] : frame_of(frame_ptr, n_frames, i);
  const int64_t fbeg = frame_ptr[f], fend = frame_ptr[f + 1];
  int64_t row_beg = 0;
  int L = 0;
  if (FILL) {
    row_beg = rowptr[i];
    L = (int)(rowptr[i + 1] - row_beg);
    if (L == 0) return;
  }
  const unsigned lt_mask = (1u << lane) - 1u;
  int count = 0;
  const bool ordered_scan = !CELLS || (FILL && L > kSortCap);
  if (ordered_scan) {
    // candidates visited in ascending j: ballot-compaction yields the sorted row directly
    for (int64_t j0 = undirected ? i + 1 : fbeg; j0 < fend; j0 += 32) {
      const int64_t j = j0 + lane;
      bool ok = false;
      if (j < fend && j != i) ok = within_cutoff(xi, yi, zi, xyz[j * 3], xyz[j * 3 + 1], xyz[j * 3 + 2], cutoff);
      const unsigned m = __ballot_sync(0xffffffffu, ok);
      if (FILL && ok) {
        const int64_t p = row_beg + count + __popc(m & lt_mask);
        out_pairs[2 * p] = i;
        out_pairs[2 * p + 1] = j;
      }
      count += __popc(m);
    }
  } else {
    const FrameInfo fi = ws.frames[f];
    const int local = ws.cell_of_atom[i] - fi.cell_base;
    const int cx = local % fi.nx, cy = (local / fi.nx) % fi.ny, cz = local / (fi.nx * fi.ny);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, fi.nx - 1);
    for (int dz = -1; dz <= 1; ++dz) {
      const int z = cz + dz;
      if (z < 0 || z >= fi.nz) continue;
      for (int dy = -1; dy <= 1; ++dy) {
        const int y = cy + dy;
        if (y < 0 || y >= fi.ny) continue;
        const int rowc = fi.cell_base + (z * fi.ny + y) * fi.nx;
        const int beg = ws.cell_start[rowc + x0], end = ws.cell_start[rowc + x1 + 1];  // x-adjacent cells are contiguous
        for (int t0 = beg; t0 < end; t0 += 32) {
          const int t = t0 + lane;
          bool ok = false;
          int j = -1;
          if (t < end) {
            j = ws.cell_atoms[t];
            if (j != i && (!undirected || j > i))
              ok = within_cutoff(xi, yi, zi, xyz[(int64_t)j * 3], xyz[(int64_t)j * 3 + 1], xyz[(int64_t)j * 3 + 2], cutoff);
          }
          const unsigned m = __ballot_sync(0xffffffffu, ok);
          if (FILL && ok) buf[warp][count + __popc(m & lt_mask)] = j;
          count += __popc(m);
        }
      }
    }
    if (FILL) {
      const int P = next_pow2(L);
      for (int t = L + lane; t < P; t += 32) buf[warp][t] = INT_MAX;
      __syncwarp();
      warp_bitonic(buf[warp], P, lane);
      for (int t = lane; t < L; t += 32) {
        out_pairs[2 * (row_beg + t)] = i;
        out_pairs[2 * (row_beg + t) + 1] = buf[warp][t];
      }
    }
  }
  if (!FILL && lane == 0) deg[i] = count;
}

// ------------------------------------------------------------------------------------------
// CSR
// ------------------------------------------------------------------------------------------
__global__ void edge_orientation_kernel(const int64_t* __restrict__ pairs, int64_t E, int32_t* __restrict__ flags) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool up = false, down = false;
  if (e < E) {
    const int64_t a = pairs[2 * e], b = pairs[2 * e + 1];
    up = a > b;
    down = b > a;
  }
  if (__any_sync(0xffffffffu, up) && (threadIdx.x & 31) == 0) atomicOr(&flags[0], 1);
  if (__any_sync(0xffffffffu, down) && (threadIdx.x & 31) == 0) atomicOr(&flags[1], 1);
}

// Directed edge d of an edge list.  Plain list: d < n -> pairs[d].  symmetrize (make_directed, conv.py:19:
// cat([nbrs, nbrs.flip(1)])): d < n -> pairs[d]; n <= d < 2n -> pairs[d-n] flipped.  n comes from device memory when
// n_dev != nullptr (static-capacity lists replayed inside a CUDA graph), else from the host argument.
__device__ __forceinline__ bool directed_edge(const int64_t* __restrict__ pairs, int64_t d, int64_t n_host,
                                              const int64_t* __restrict__ n_dev, int symmetrize, int64_t& i, int64_t& j) {
  const int64_t n = n_dev ? *n_dev : n_host;
  if (d < n) { i = pairs[2 * d]; j = pairs[2 * d + 1]; return true; }
  if (symmetrize && d < 2 * n) { i = pairs[2 * (d - n) + 1]; j = pairs[2 * (d - n)]; return true; }
  return false;
}

__global__ void csr_count_kernel(const int64_t* __restrict__ pairs, int64_t E, const int64_t* __restrict__ n_dev, int symmetrize,
                                 int64_t n_recv, int64_t n_send, int32_t* __restrict__ deg_r, int32_t* __restrict__ deg_s,
                                 int32_t* __restrict__ err) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t i, j;
  if (!directed_edge(pairs, e, E, n_dev, symmetrize, i, j)) return;
  if (i < 0 || i >= n_recv || j < 0 || j >= n_send) { raise_flag(err, CGVAE_ERR_NODE_INDEX); return; }
  atomicAdd(&deg_r[i], 1);
  atomicAdd(&deg_s[j], 1);
}

// place edge ids into their receiver row / sender row (arbitrary order; rows are sorted afterwards)
__global__ void csr_place_kernel(const int64_t* __restrict__ pairs, int64_t E, const int64_t* __restrict__ n_dev, int symmetrize,
                                 const int32_t* __restrict__ rowptr_r, const int32_t* __restrict__ rowptr_s,
                                 int32_t* __restrict__ cursor_r, int32_t* __restrict__ cursor_s,
                                 int32_t* __restrict__ eid_r, int32_t* __restrict__ eid_s, int64_t n_recv, int64_t n_send) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t i, j;
  if (!directed_edge(pairs, e, E, n_dev, symmetrize, i, j)) return;
  if (i < 0 || i >= n_recv || j < 0 || j >= n_send) return;   // flagged by csr_count_kernel
  eid_r[rowptr_r[i] + atomicAdd(&cursor_r[i], 1)] = (int32_t)e;
  eid_s[rowptr_s[j] + atomicAdd(&cursor_s[j], 1)] = (int32_t)e;
}

// slots t < total (= rowptr[n_rows], read on the device) are live; the tail of a static-capacity graph is zeroed
__global__ void csr_finish_r_kernel(const int64_t* __restrict__ pairs, int64_t E, const int64_t* __restrict__ n_dev, int symmetrize,
                                    int64_t cap, const int32_t* __restrict__ total, const int32_t* __restrict__ eid_r,
                                    int32_t* __restrict__ col, int32_t* __restrict__ slot_of_edge) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= cap) return;
  if (t >= *total) { col[t] = 0; return; }
  const int e = eid_r[t];
  int64_t i, j;
  directed_edge(pairs, e, E, n_dev, symmetrize, i, j);
  col[t] = (int32_t)j;
  slot_of_edge[e] = (int32_t)t;
}
__global__ void csr_finish_s_kernel(const int64_t* __restrict__ pairs, int64_t E, const int64_t* __restrict__ n_dev, int symmetrize,
                                    int64_t cap, const int32_t* __restrict__ total, const int32_t* __restrict__ eid_s,
                                    const int32_t* __restrict__ slot_of_edge, int32_t* __restrict__ col_t, int32_t* __restrict__ perm_t) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= cap) return;
  if (t >= *total) { col_t[t] = 0; perm_t[t] = 0; return; }
  const int e = eid_s[t];
  int64_t i, j;
  directed_edge(pairs, e, E, n_dev, symmetrize, i, j);
  col_t[t] = (int32_t)i;
  perm_t[t] = slot_of_edge[e];
}

// ------------------------------------------------------------------------------------------
// segment ranks (CG2ChannelIdx)
// ------------------------------------------------------------------------------------------
__global__ void segment_count_kernel(const int64_t* __restrict__ mapping, int64_t n, int64_t n_beads, int32_t* __restrict__ deg,
                                     int32_t* __restrict__ err) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n) return;
  const int64_t b = mapping[a];
  if (b < 0 || b >= n_beads) { raise_flag(err, CGVAE_ERR_BEAD_INDEX); return; }
  atomicAdd(&deg[b], 1);
}
__global__ void segment_place_kernel(const int64_t* __restrict__ mapping, int64_t n, int64_t n_beads,
                                     const int32_t* __restrict__ rowptr_b, int32_t* __restrict__ cursor, int32_t* __restrict__ atoms) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n) return;
  const int64_t b = mapping[a];
  if (b < 0 || b >= n_beads) return;                           // flagged by segment_count_kernel
  atoms[rowptr_b[b] + atomicAdd(&cursor[b], 1)] = (int32_t)a;
}
__global__ void segment_rank_kernel(const int64_t* __restrict__ mapping, int64_t n, int64_t n_beads,
                                    const int32_t* __restrict__ rowptr_b, const int32_t* __restrict__ atoms,
                                    int32_t* __restrict__ slot_of_atom, int64_t* __restrict__ rank) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n || t >= rowptr_b[n_beads]) return;                 // fewer live slots only when indices were rejected
  const int a = atoms[t];
  slot_of_atom[a] = (int32_t)t;
  rank[a] = t - rowptr_b[mapping[a]];
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

int cgvae_abi_version(void) { return CGVAE_ABI_VERSION; }
const char* cgvae_last_error(void) { return g_err; }
unsigned long long cgvae_launch_count(void) { return g_launches.load(); }
int cgvae_set_pdl(int on) {
  const int prev = cgvae::pdl_enabled() ? 1 : 0;
  cgvae::g_pdl.store(on ? 1 : 0, std::memory_order_relaxed);
  return prev;
}

int cgvae_set_matmul_precision(int mode) {
  CGVAE_REQUIRE(mode == 0 || mode == 1, "set_matmul_precision: mode must be 0 (\"highest\", 3xTF32) or 1 (\"high\", 1xTF32), got %d",
                mode);
  return cgvae::g_matmul_precision.exchange(mode, std::memory_order_relaxed);
}
int cgvae_get_matmul_precision(void) { return cgvae::matmul_precision(); }

int cgvae_set_error_flags(int device, int32_t* flags) {
  CGVAE_REQUIRE(device >= 0 && device < kMaxDevices, "set_error_flags: bad device %d", device);
  g_err_flags[device].store(flags);
  return 0;
}

size_t cgvae_radius_graph_ws_bytes(int64_t n, int64_t n_frames) {
  return radius_ws_layout(n > 0 ? n : 1, n_frames > 0 ? n_frames : 1, nullptr, nullptr) + 256;
}

static int radius_prepare_cells(const float* xyz, int64_t n, const int64_t* frame_ptr, int64_t n_frames, float cutoff,
                                void* ws, size_t ws_bytes, RadiusWs* w, cudaStream_t st) {
  CGVAE_REQUIRE(ws && ws_bytes >= cgvae_radius_graph_ws_bytes(n, n_frames), "radius_graph: workspace too small");
  radius_ws_layout(n, n_frames, reinterpret_cast<char*>(ws), w);
  CGVAE_ZERO(w->cell_count, sizeof(int32_t) * (size_t)w->max_cells, st);
  launch_kernel(frame_bounds_kernel, dim3((unsigned)n_frames), dim3(256), 0, st, xyz, frame_ptr, cutoff, w->frames);
  if (int rc = launched("frame_bounds")) return rc;
  launch_kernel(frame_offsets_kernel, dim3(1), dim3(32), 0, st, w->frames, n_frames);
  if (int rc = launched("frame_offsets")) return rc;
  const unsigned gb = (unsigned)ceil_div(n, 256);
  launch_kernel(assign_cells_kernel, dim3(gb), dim3(256), 0, st, xyz, n, frame_ptr, n_frames, w->frames, w->frame_of_atom, w->cell_of_atom, w->cell_count);
  if (int rc = launched("assign_cells")) return rc;
  launch_kernel(scan_kernel<int32_t>, dim3(1), dim3(1024), 0, st, w->cell_count, w->max_cells, w->cell_start);
  if (int rc = launched("cell_scan")) return rc;
  CGVAE_ZERO(w->cell_count, sizeof(int32_t) * (size_t)w->max_cells, st);
  launch_kernel(fill_cells_kernel, dim3(gb), dim3(256), 0, st, n, w->cell_of_atom, w->cell_start, w->cell_count, w->cell_atoms);
  return launched("fill_cells");
}

int cgvae_radius_graph_count(const float* xyz, int64_t n, const int64_t* frame_ptr, int64_t n_frames, float cutoff,
                             int undirected, int use_cells, int32_t* deg, void* ws, size_t ws_bytes, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CGVAE_REQUIRE(n >= 0 && n_frames >= 1 && n < INT_MAX, "radius_graph: bad sizes n=%lld frames=%lld", (long long)n, (long long)n_frames);
  if (n == 0) return 0;
  CGVAE_REQUIRE(xyz && frame_ptr && deg, "radius_graph: null pointer");
  RadiusWs w{};
  if (use_cells) {
    if (int rc = radius_prepare_cells(xyz, n, frame_ptr, n_frames, cutoff, ws, ws_bytes, &w, st)) return rc;
    launch_kernel(radius_query_kernel<false, true>, dim3((unsigned)ceil_div(n, kRadWarps)), dim3(kRadWarps * 32), 0, st, 
        xyz, n, frame_ptr, n_frames, cutoff, undirected, w, deg, nullptr, nullptr);
  } else {
    launch_kernel(radius_query_kernel<false, false>, dim3((unsigned)ceil_div(n, kRadWarps)), dim3(kRadWarps * 32), 0, st, 
        xyz, n, frame_ptr, n_frames, cutoff, undirected, w, deg, nullptr, nullptr);
  }
  return launched("radius_count");
}

int cgvae_radius_graph_fill(const float* xyz, int64_t n, const int64_t* frame_ptr, int64_t n_frames, float cutoff,
                            int undirected, int use_cells, const int64_t* rowptr, int64_t* out_pairs, void* ws,
                            size_t ws_bytes, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return 0;
  CGVAE_REQUIRE(xyz && frame_ptr && rowptr && out_pairs, "radius_graph_fill: null pointer");
  RadiusWs w{};
  if (use_cells) {
    // the cell structure written by cgvae_radius_graph_count into `ws` is reused as is
    CGVAE_REQUIRE(ws && ws_bytes >= cgvae_radius_graph_ws_bytes(n, n_frames), "radius_graph_fill: workspace too small");
    radius_ws_layout(n, n_frames, reinterpret_cast<char*>(ws), &w);
    launch_kernel(radius_query_kernel<true, true>, dim3((unsigned)ceil_div(n, kRadWarps)), dim3(kRadWarps * 32), 0, st, 
        xyz, n, frame_ptr, n_frames, cutoff, undirected, w, nullptr, rowptr, out_pairs);
  } else {
    launch_kernel(radius_query_kernel<true, false>, dim3((unsigned)ceil_div(n, kRadWarps)), dim3(kRadWarps * 32), 0, st, 
        xyz, n, frame_ptr, n_frames, cutoff, undirected, w, nullptr, rowptr, out_pairs);
  }
  return launched("radius_fill");
}

int cgvae_exclusive_scan(const int32_t* counts, int64_t n, int64_t* out, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n >= 0 && out, "exclusive_scan: bad arguments");
  launch_kernel(scan_kernel<int64_t>, dim3(1), dim3(1024), 0, (cudaStream_t)stream, counts, n, out);
  return launched("scan_i64");
}
int cgvae_scan_i32(const int32_t* counts, int64_t n, int32_t* out, cgvae_stream_t stream) {
  CGVAE_REQUIRE(n >= 0 && out, "scan_i32: bad arguments");
  launch_kernel(scan_kernel<int32_t>, dim3(1), dim3(1024), 0, (cudaStream_t)stream, counts, n, out);
  return launched("scan_i32");
}

int cgvae_edge_orientation(const int64_t* pairs, int64_t n_edges, int32_t* flags, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CGVAE_REQUIRE(flags, "edge_orientation: null flags");
  CGVAE_ZERO(flags, 2 * sizeof(int32_t), st);
  if (n_edges == 0) return 0;
  launch_kernel(edge_orientation_kernel, dim3((unsigned)ceil_div(n_edges, 256)), dim3(256), 0, st, pairs, n_edges, flags);
  return launched("edge_orientation");
}

int cgvae_csr_count(const int64_t* pairs, int64_t n_edges, const int64_t* n_edges_dev, int symmetrize, int64_t n_recv,
                    int64_t n_send, int32_t* deg_r, int32_t* deg_s, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t cap = symmetrize ? 2 * n_edges : n_edges;
  CGVAE_REQUIRE(n_edges >= 0 && cap < INT_MAX && deg_r && deg_s, "csr_count: bad arguments");
  CGVAE_ZERO(deg_r, sizeof(int32_t) * (size_t)n_recv, st);
  CGVAE_ZERO(deg_s, sizeof(int32_t) * (size_t)n_send, st);
  if (cap == 0) return 0;
  launch_kernel(csr_count_kernel, dim3((unsigned)ceil_div(cap, 256)), dim3(256), 0, st, pairs, n_edges, n_edges_dev, symmetrize, n_recv, n_send, deg_r, deg_s,
                err_flags());
  return launched("csr_count");
}

int cgvae_csr_fill(const int64_t* pairs, int64_t n_edges_in, const int64_t* n_edges_dev, int symmetrize, int64_t n_recv,
                   int64_t n_send, const int32_t* rowptr_r, const int32_t* rowptr_s, int32_t* scratch, int32_t* col, int32_t* eid,
                   int32_t* col_t, int32_t* perm_t, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_edges = symmetrize ? 2 * n_edges_in : n_edges_in;   // capacity in directed edges
  if (n_edges == 0) return 0;
  CGVAE_REQUIRE(pairs && rowptr_r && rowptr_s && scratch && col && eid && col_t && perm_t, "csr_fill: null pointer");
  // scratch: cursor_r[n_recv] | cursor_s[n_send] | eid_s[E] | slot_of_edge[E]
  int32_t* cursor_r = scratch;
  int32_t* cursor_s = cursor_r + n_recv;
  int32_t* eid_s = cursor_s + n_send;
  int32_t* slot_of_edge = eid_s + n_edges;
  CGVAE_ZERO(cursor_r, sizeof(int32_t) * (size_t)(n_recv + n_send), st);
  const unsigned gb = (unsigned)ceil_div(n_edges, 256);
  launch_kernel(csr_place_kernel, dim3(gb), dim3(256), 0, st, pairs, n_edges_in, n_edges_dev, symmetrize, rowptr_r, rowptr_s, cursor_r, cursor_s, eid, eid_s,
                n_recv, n_send);
  if (int rc = launched("csr_place")) return rc;
  // rows were filled in atomic (arbitrary) order: sorting by edge id makes the layout deterministic and
  // keeps the reference's edge-list order inside every row
  launch_kernel(sort_rows_kernel, dim3((unsigned)ceil_div(n_recv, kSortWarps)), dim3(kSortWarps * 32), 0, st, rowptr_r, n_recv, eid);
  if (int rc = launched("csr_sort_r")) return rc;
  launch_kernel(sort_rows_kernel, dim3((unsigned)ceil_div(n_send, kSortWarps)), dim3(kSortWarps * 32), 0, st, rowptr_s, n_send, eid_s);
  if (int rc = launched("csr_sort_s")) return rc;
  launch_kernel(csr_finish_r_kernel, dim3(gb), dim3(256), 0, st, pairs, n_edges_in, n_edges_dev, symmetrize, n_edges, rowptr_r + n_recv, eid, col,
                                          slot_of_edge);
  if (int rc = launched("csr_finish_r")) return rc;
  launch_kernel(csr_finish_s_kernel, dim3(gb), dim3(256), 0, st, pairs, n_edges_in, n_edges_dev, symmetrize, n_edges, rowptr_s + n_send, eid_s,
                                          slot_of_edge, col_t, perm_t);
  return launched("csr_finish_s");
}

int cgvae_segment_count(const int64_t* mapping, int64_t n, int64_t n_beads, int32_t* deg, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CGVAE_REQUIRE(deg && n >= 0 && n < INT_MAX, "segment_count: bad arguments");
  CGVAE_ZERO(deg, sizeof(int32_t) * (size_t)n_beads, st);
  if (n == 0) return 0;
  launch_kernel(segment_count_kernel, dim3((unsigned)ceil_div(n, 256)), dim3(256), 0, st, mapping, n, n_beads, deg, err_flags());
  return launched("segment_count");
}

int cgvae_segment_rank(const int64_t* mapping, int64_t n, int64_t n_beads, const int32_t* rowptr_b, int32_t* scratch,
                       int32_t* atoms, int32_t* slot_of_atom, int64_t* rank, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return 0;
  CGVAE_REQUIRE(mapping && rowptr_b && scratch && atoms && slot_of_atom && rank, "segment_rank: null pointer");
  CGVAE_ZERO(scratch, sizeof(int32_t) * (size_t)n_beads, st);
  const unsigned gb = (unsigned)ceil_div(n, 256);
  launch_kernel(segment_place_kernel, dim3(gb), dim3(256), 0, st, mapping, n, n_beads, rowptr_b, scratch, atoms);
  if (int rc = launched("segment_place")) return rc;
  launch_kernel(sort_rows_kernel, dim3((unsigned)ceil_div(n_beads, kSortWarps)), dim3(kSortWarps * 32), 0, st, rowptr_b, n_beads, atoms);
  if (int rc = launched("segment_sort")) return rc;
  launch_kernel(segment_rank_kernel, dim3(gb), dim3(256), 0, st, mapping, n, n_beads, rowptr_b, atoms, slot_of_atom, rank);
  return launched("segment_rank");
}

}  // extern "C"
