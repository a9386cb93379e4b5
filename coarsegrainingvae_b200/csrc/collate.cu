// Ragged collation of an HBM-resident protein set into one batch (data.DeviceProteinDataset.collate).
//
// Every per-protein array of the set lives in one concatenated store per kind of row (atoms, residues, bonds, C-alpha
// edges, dihedrals, C-alpha indices) with a row-offset table item_ptr[kind][P+1].  A batch is a vector of item indices
// (-1 = empty slot).  Two launches, no host synchronisation, CUDA-graph capturable:
//   collate_scan_kernel   one CTA, one warp per kind: exclusive scan of the selected items' sizes into slot_off
//                         [kind][n_slots+1] and the live counts min(total, capacity); overflow or an item index outside
//                         [-1, n_items) raises CGVAE_ERR_COLLATE_BIT (the excess rows are dropped, nothing is written past a
//                         capacity).
//   collate_gather_kernel one thread per output row over the concatenated row space of all outputs.  A live row finds its
//                         slot by binary search in slot_off and copies the source row, adding the slot's running atom or
//                         residue count to index rows; a row past the live count gets the pad value (zero, or for the
//                         atom -> residue map the pad bead live_residues + k / atoms_per_bead of pad atom k).  Thread 0
//                         also writes the per-key count outputs and the loss denominators.
// The plan travels in the kernel parameters (__grid_constant__, like wgrad_grouped_kernel): no table memory, no copies.
#include "common.cuh"

namespace cgvae {

__global__ void __launch_bounds__(32 * CGVAE_COLLATE_KINDS) collate_scan_kernel(const __grid_constant__ cgvae_collate_plan plan,
                                                                                  int32_t* __restrict__ err) {
  CGVAE_KERNEL_PROLOGUE();
  const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_slots = plan.n_slots, n_items = plan.n_items;
  const int64_t* ptr = plan.item_ptr + (int64_t)k * (n_items + 1);
  int64_t* off = plan.slot_off + (int64_t)k * (n_slots + 1);
  int64_t carry = 0;
  bool bad = false;
  for (int64_t base = 0; base < n_slots; base += 32) {
    const int64_t s = base + lane;
    int64_t v = 0;
    if (s < n_slots) {
      const int64_t p = plan.idx[s];
      if (p >= 0 && p < n_items) v = ptr[p + 1] - ptr[p];
      else if (p != -1) bad = true;
    }
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (s < n_slots) off[s] = carry + x - v;
    carry += __shfl_sync(0xffffffffu, x, 31);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0 && k == 0) raise_flag(err, CGVAE_ERR_COLLATE_BIT);
  if (lane == 0) {
    off[n_slots] = carry;
    const int64_t cap = plan.live_cap[k];
    plan.counts[k] = carry < cap ? carry : cap;
    if (carry > cap) raise_flag(err, CGVAE_ERR_COLLATE_BIT);
  }
}

// largest slot s in [0, n_slots) with off[s] <= r: the (non-empty) slot that holds output row r < off[n_slots]
__device__ __forceinline__ int64_t slot_of_row(const int64_t* __restrict__ off, int64_t n_slots, int64_t r) {
  int64_t lo = 0, hi = n_slots;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (off[mid] <= r) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256) collate_gather_kernel(const __grid_constant__ cgvae_collate_plan plan) {
  CGVAE_KERNEL_PROLOGUE();
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0) {
    for (int k = 0; k < CGVAE_COLLATE_KINDS; ++k)
      if (plan.count_out[k] != nullptr) plan.count_out[k][0] = plan.counts[k];
    if (plan.norms != nullptr) {      // (atoms, residues, bonds) denominators of the loss means, as update_dp_norms forms them
      plan.norms[0] = fmaxf((float)plan.counts[CGVAE_COLLATE_ATOMS], 1.f);
      plan.norms[1] = fmaxf((float)plan.counts[CGVAE_COLLATE_RESIDUES], 1.f);
      plan.norms[2] = fmaxf((float)plan.counts[CGVAE_COLLATE_BONDS], 1.f);
    }
  }
  int64_t begin = 0;
  int i = 0;
  for (; i < plan.n_out; ++i) {
    if (g < begin + plan.out[i].rows) break;
    begin += plan.out[i].rows;
  }
  if (i >= plan.n_out) return;
  const cgvae_collate_out& o = plan.out[i];
  const int64_t r = g - begin;
  const int w = o.width;
  const int64_t live = plan.counts[o.kind];
  if (r < live) {
    const int64_t n_slots = plan.n_slots;
    const int64_t* off = plan.slot_off + (int64_t)o.kind * (n_slots + 1);
    const int64_t s = slot_of_row(off, n_slots, r);
    const int64_t p = plan.idx[s];
    const int64_t src_row = plan.item_ptr[(int64_t)o.kind * (plan.n_items + 1) + p] + (r - off[s]);
    if (o.elem_bytes == 8) {
      const int64_t add = o.add_kind >= 0 ? plan.slot_off[(int64_t)o.add_kind * (n_slots + 1) + s] : 0;
      const int64_t* src = static_cast<const int64_t*>(o.src) + src_row * w;
      int64_t* dst = static_cast<int64_t*>(o.dst) + r * w;
      for (int c = 0; c < w; ++c) dst[c] = src[c] + add;
    } else {
      const float* src = static_cast<const float*>(o.src) + src_row * w;
      float* dst = static_cast<float*>(o.dst) + r * w;
      for (int c = 0; c < w; ++c) dst[c] = src[c];
    }
  } else if (o.elem_bytes == 8) {
    int64_t v = 0;
    if (o.pad_beads) {
      // pad atom k -> pad bead live_res + k / A: no bead holds more than A atoms (the CG2ChannelIdx bound, cgvae.py:473)
      v = plan.counts[CGVAE_COLLATE_RESIDUES] + (r - live) / plan.atoms_per_bead;
      if (v >= plan.n_beads) v = plan.n_beads - 1;       // only after an overflow, which is flagged
    }
    int64_t* dst = static_cast<int64_t*>(o.dst) + r * w;
    for (int c = 0; c < w; ++c) dst[c] = v;
  } else {
    float* dst = static_cast<float*>(o.dst) + r * w;
    for (int c = 0; c < w; ++c) dst[c] = 0.f;
  }
}

}  // namespace cgvae

using namespace cgvae;

extern "C" {

size_t cgvae_collate_plan_bytes(void) { return sizeof(cgvae_collate_plan); }

int cgvae_collate(const cgvae_collate_plan* plan, cgvae_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CGVAE_REQUIRE(plan != nullptr, "collate: null plan");
  CGVAE_REQUIRE(plan->n_out >= 0 && plan->n_out <= CGVAE_COLLATE_MAX_OUT, "collate: n_out %d outside [0, %d]", plan->n_out,
                CGVAE_COLLATE_MAX_OUT);
  CGVAE_REQUIRE(plan->n_slots >= 0 && plan->n_items >= 0 && plan->atoms_per_bead >= 1, "collate: bad sizes");
  CGVAE_REQUIRE(plan->item_ptr && plan->slot_off && plan->counts && (plan->idx || plan->n_slots == 0), "collate: null pointer");
  int64_t rows = 0;
  for (int i = 0; i < plan->n_out; ++i) {
    const cgvae_collate_out& o = plan->out[i];
    CGVAE_REQUIRE(o.kind >= 0 && o.kind < CGVAE_COLLATE_KINDS && o.add_kind >= -1 && o.add_kind < CGVAE_COLLATE_KINDS,
                  "collate: output %d: bad kind", i);
    CGVAE_REQUIRE(o.elem_bytes == 4 || o.elem_bytes == 8, "collate: output %d: elem_bytes must be 4 or 8", i);
    CGVAE_REQUIRE(o.width >= 1 && o.rows >= 0 && (o.dst || o.rows == 0), "collate: output %d: bad shape", i);
    CGVAE_REQUIRE(o.elem_bytes == 8 || (o.add_kind < 0 && !o.pad_beads), "collate: output %d: offsets need int64 rows", i);
    CGVAE_REQUIRE(!o.pad_beads || plan->n_beads >= 1, "collate: output %d: pad beads need n_beads >= 1", i);
    rows += o.rows;
  }
  launch_kernel(collate_scan_kernel, dim3(1), dim3(32 * CGVAE_COLLATE_KINDS), 0, st, *plan, err_flags());
  if (int rc = launched("collate_scan")) return rc;
  launch_kernel(collate_gather_kernel, dim3((unsigned)std::max<int64_t>(1, ceil_div(rows, 256))), dim3(256), 0, st, *plan);
  return launched("collate_gather");
}

}  // extern "C"
