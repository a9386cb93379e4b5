/*
 * cgvae_b200.h -- C ABI of libcgvae_sm100.so: the B200 (sm_100a) implementation of the CGVAE
 * equivariant message-passing hot path.
 *
 * The reference (wwang2/CoarseGrainingVAE) has no FFI of its own: the path sits behind plain
 * nn.Module.forward calls that bottom out in ATen ops and torch_scatter (SURVEY.md section 8b).
 * Each entry point below therefore names the reference Python interface it replaces
 * (file:line under /root/reference/CoarseGrainingVAE).  The reference-side binding (ctypes) is
 * shown in INTEGRATION.md; coarsegrainingvae_b200/_lib.py is that binding.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller
 *    (PyTorch allocates), 16-byte aligned, contiguous.  Kernels never allocate, free or
 *    retain pointers; scratch is passed in (`ws`, size from the matching *_ws_bytes()).
 *  - all launches go on `stream`; no host synchronisation inside (CUDA-graph capturable);
 *    output sizes that depend on data (edge counts) are left in device memory for the caller
 *    to read (the last element of the scanned offsets).
 *  - return 0 on success, <0 argument error, >0 cudaError_t; text via cgvae_last_error()
 *    (thread-local).  All entry points are re-entrant (autograd calls backward from worker
 *    threads).
 *  - layouts: scalars s[N][F]; vectors v[N][3][F] ("planar": xyz major, channel minor);
 *    phi[N][K][F]; filter weights in the reference's native nn.Linear layout Wf[K*F][R],
 *    bf[K*F]; dense weights W[out][in].
 *  - graphs: receiver-major CSR (rowptr[n_recv+1], col[E] = sender) with per-edge data in CSR
 *    order (basis[E][RB], unit[E][4]); sender-major CSR (rowptr_t[n_send+1], col_t[E] =
 *    receiver, perm_t[E] = CSR slot of the same edge in receiver order) for the backward.
 *    Internal index arrays are int32; edge lists crossing the boundary are the reference's
 *    int64 [E][2] (column 0 receiver, column 1 sender).
 */
#ifndef CGVAE_B200_H_
#define CGVAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cgvae_stream_t; /* cudaStream_t */

#define CGVAE_ABI_VERSION 1

/* activation codes (reference modules.py:32-42 `layer_types`) */
enum { CGVAE_ACT_NONE = 0, CGVAE_ACT_SWISH = 1, CGVAE_ACT_RELU = 2, CGVAE_ACT_TANH = 3,
       /* the rest of the reference's layer_types registry (modules.py:32-42) */
       CGVAE_ACT_SIGMOID = 4, CGVAE_ACT_SHIFTED_SOFTPLUS = 5, CGVAE_ACT_LEAKY_RELU = 6, CGVAE_ACT_ELU = 7 };
/* GEMM operand forms */
enum { CGVAE_GEMM_NT = 0, /* C[M,N] = A[M,K] * B[N,K]^T   (y = x W^T, Dense.forward modules.py:101) */
       CGVAE_GEMM_NN = 1, /* C[M,N] = A[M,K] * B[K,N]     (grad_in = grad_out W)                    */
       CGVAE_GEMM_TN = 2  /* C[M,N] = A[K,M]^T * B[K,N]   (grad_W = grad_out^T x)                   */ };

int cgvae_abi_version(void);
const char* cgvae_last_error(void);
/* number of kernels launched by this library in the calling process (bench.py `gpu_launches`) */
unsigned long long cgvae_launch_count(void);
/* Index validation without host round trips: the kernels SKIP an out-of-range index (no out-of-bounds access) and
 * OR a bit into the caller-owned device word registered here for `device` (NULL unregisters); the host reads it when
 * it synchronises anyway and raises what the reference raises (IndexError at cgvae.py:473 / nn.Embedding). */
enum { CGVAE_ERR_LIFT_RANK_BIT = 1,   /* a bead holds more atoms than channels F (cgvae.py:473) */
       CGVAE_ERR_EMBED_INDEX_BIT = 2, /* embedding id outside the table (cgvae.py:273,380,591) */
       CGVAE_ERR_BEAD_INDEX_BIT = 4,  /* CG_mapping entry outside [0, n_beads) */
       CGVAE_ERR_NODE_INDEX_BIT = 8,  /* edge-list entry outside [0, n_nodes) */
       CGVAE_ERR_COLLATE_BIT = 16     /* a collated batch exceeds its capacities, or selects an item outside the set */ };
int cgvae_set_error_flags(int device, int32_t* flags);

/* ------------------------------------------------------------------ graph builders (integer) */

/* get_neighbor_list, data.py:65-82 -- all pairs with fp32 |x_i-x_j| <= cutoff, i != j, within the
 * same frame (frame_ptr[n_frames+1] atom offsets: the per-frame loop of
 * CGDataset.generate_neighbor_list data.py:207-225 plus the CG_collate offsets data.py:255-270).
 * undirected != 0 keeps j > i.  Two calls: count (fills deg[n], per-atom neighbour count) then,
 * after an exclusive scan into rowptr[n+1], fill (writes out[E][2] int64, sorted by (i, j)).
 * `use_cells` != 0: cell-list search (cells of edge >= cutoff per frame); 0: tiled brute force.
 * ws: cgvae_radius_graph_ws_bytes(n, n_frames).  Bit-exact vs the reference. */
size_t cgvae_radius_graph_ws_bytes(int64_t n, int64_t n_frames);
int cgvae_radius_graph_count(const float* xyz, int64_t n, const int64_t* frame_ptr, int64_t n_frames,
                             float cutoff, int undirected, int use_cells, int32_t* deg, void* ws,
                             size_t ws_bytes, cgvae_stream_t stream);
int cgvae_radius_graph_fill(const float* xyz, int64_t n, const int64_t* frame_ptr, int64_t n_frames,
                            float cutoff, int undirected, int use_cells, const int64_t* rowptr,
                            int64_t* out_pairs, void* ws, size_t ws_bytes, cgvae_stream_t stream);

/* exclusive scan of int32 counts into int64 offsets out[n+1] (out[n] = total). */
int cgvae_exclusive_scan(const int32_t* counts, int64_t n, int64_t* out, cgvae_stream_t stream);

/* make_directed, conv.py:10-20 -- flags[0] = any(col0 > col1), flags[1] = any(col1 > col0) (device
 * int32[2], zeroed by the call); the caller appends the flipped list when not both are set. */
int cgvae_edge_orientation(const int64_t* pairs, int64_t n_edges, int32_t* flags, cgvae_stream_t stream);

/* Receiver CSR + sender CSR of a directed edge list (replaces scatter_add(index=nbrs[:,0]) call
 * sites conv.py:223-240,392-400,553-561).  key_col = 0 builds rows over column 0.
 *   cgvae_csr_count : deg_r[n_recv], deg_s[n_send] (int32, zeroed by the call)
 *   cgvae_csr_fill  : rowptr_r/rowptr_s are int32 exclusive scans (n+1).  Writes, in the original
 *                     edge order within every row (deterministic): col[E] (sender), eid[E] (original
 *                     edge id of each CSR slot), col_t[E] (receiver), perm_t[E] (receiver-CSR slot).
 * symmetrize != 0: `pairs` is the one-directional list and the flipped copy of make_directed
 * (conv.py:19, cat([nbrs, nbrs.flip(1)])) is generated on the fly: directed edge d >= n is pairs[d-n]
 * flipped; all outputs then hold 2*n_edges slots.  n_edges_dev (nullable): the live edge count read
 * from DEVICE memory, with n_edges the static capacity of `pairs` -- this keeps every launch shape
 * fixed so a whole training step can be replayed as one CUDA graph while the edge count changes. */
int cgvae_csr_count(const int64_t* pairs, int64_t n_edges, const int64_t* n_edges_dev, int symmetrize,
                    int64_t n_recv, int64_t n_send, int32_t* deg_r, int32_t* deg_s, cgvae_stream_t stream);
int cgvae_scan_i32(const int32_t* counts, int64_t n, int32_t* out, cgvae_stream_t stream);
int cgvae_csr_fill(const int64_t* pairs, int64_t n_edges, const int64_t* n_edges_dev, int symmetrize,
                   int64_t n_recv, int64_t n_send,
                   const int32_t* rowptr_r, const int32_t* rowptr_s, int32_t* scratch /* n_recv+n_send+2E int32 */,
                   int32_t* col, int32_t* eid, int32_t* col_t, int32_t* perm_t, cgvae_stream_t stream);

/* CG2ChannelIdx, cgvae.py:451-460 -- rank[n] = #{m < n : mapping[m] == mapping[n]}; also the bead
 * CSR (rowptr_b[n_beads+1] given by the caller from cgvae_csr_count/scan; atoms[n] in ascending
 * order per bead).  Exact. */
int cgvae_segment_count(const int64_t* mapping, int64_t n, int64_t n_beads, int32_t* deg, cgvae_stream_t stream);
int cgvae_segment_rank(const int64_t* mapping, int64_t n, int64_t n_beads, const int32_t* rowptr_b,
                       int32_t* scratch /* n_beads int32 */, int32_t* atoms, int32_t* slot_of_atom, int64_t* rank,
                       cgvae_stream_t stream);

/* ------------------------------------------------------------------ edge geometry (fp32) */

/* preprocess_r conv.py:25-29 + PainnRadialBasis modules.py:148-172 + CosineEnvelope modules.py:52-58,
 * for the edges of a CSR: edge in slot e is (recv <- send).  r = xs[send] - xr[recv]
 * (cgvae.py:276,280,383; for the contraction graph xr = cg_xyz, send = atom).
 * basis[e][r] = rbf_r * env (r < R), basis[e][R] = env (bias column), zero padded to RB;
 * unit[e] = (ux, uy, uz, d).  coef[R] = n*pi/cutoff computed by the host exactly as the reference.
 * edge_wgt (nullable, indexed by ORIGINAL edge id through eid) is folded into the basis
 * (conv.py:528-533).  r_edge (nullable): per-edge displacement [E][3] in ORIGINAL edge order, used instead
 * of the coordinates when the caller passes r_ij directly (block-level forward signatures). */
int cgvae_edge_geometry(const float* xyz_send, const float* xyz_recv, const float* r_edge, const int32_t* rowptr,
                        const int32_t* col, int64_t n_recv, int64_t n_edges, const float* coef, int R, int RB, float cutoff,
                        const float* edge_wgt, const int32_t* eid, float* basis, float* unit,
                        cgvae_stream_t stream);

/* Backward of cgvae_edge_geometry (the reference's autograd of conv.py:25-29, modules.py:52-58,148-172): per-edge
 * displacement cotangent dr from the cotangents d_basis[E][RB] and d_unit[E][4] (either nullable = zero), same arguments
 * as the forward.  Without r_edge: dr[E][3] in receiver-CSR slot order; with r_edge: dr[eid[e]] in ORIGINAL edge order
 * (the gradient of r_edge).  Padded tail slots of a static-capacity graph give zero.  Deterministic. */
int cgvae_edge_geometry_bwd(const float* xyz_send, const float* xyz_recv, const float* r_edge, const int32_t* rowptr,
                            const int32_t* col, int64_t n_recv, int64_t n_edges, const float* coef, int R, int RB, float cutoff,
                            const float* edge_wgt, const int32_t* eid, const float* d_basis, const float* d_unit, float* dr,
                            cgvae_stream_t stream);
/* Coordinate gradients from dr[E][3] (receiver-CSR order, r_e = x_send[j] - x_recv[i]): g_send[n_send][3] = sum over the
 * sender CSR (rowptr_t, perm_t), g_recv[n_recv][3] = -sum over the receiver CSR, each in CSR order.  same != 0: sender and
 * receiver are one coordinate tensor, g_send = both terms, g_recv unused. */
int cgvae_edge_coord_reduce(const float* dr, const int32_t* rowptr, int64_t n_recv, const int32_t* rowptr_t,
                            const int32_t* perm_t, int64_t n_send, int same, float* g_send, float* g_recv,
                            cgvae_stream_t stream);

/* ------------------------------------------------------------------ dense contractions */

/* Dense / nn.Linear forward and backward contractions (modules.py:75-114, conv.py:41-49,568-586).
 * C = epilogue(op(A) op(B)) with epilogue, in order: + bias[N] (nullable); z_out = value (nullable,
 * pre-activation copy, ld = ldc); act; * dact(z_in) when z_in != NULL (activation backward with the
 * saved pre-activation, act code `dact`); + add[M,N] (nullable residual, ld = ldc).
 * ws (nullable): ws_bytes of scratch for deterministic split-K when the output grid cannot fill 148 SMs: the
 * K-slices are written there and a second kernel adds them in slice order, so the result does not depend on
 * scheduling.  Not shared between launches that may run concurrently.  counters / n_counters are ignored. */
int cgvae_gemm(int form, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
               int64_t M, int64_t N, int64_t K, const float* bias, int act, float* z_out,
               const float* z_in, int dact, const float* add, void* ws, size_t ws_bytes,
               int32_t* counters, int n_counters, cgvae_stream_t stream);
/* Two bias-free Dense layers on the SAME input whose weight matrices are adjacent in memory (W = [W1: N1 rows; W2: N2 rows],
 * row stride ldw): C1[M,N1] = x W1^T, C2[M,N2] = x W2^T (both contiguous) in ONE weight-streaming launch when M <= 48
 * (u_mat / v_mat of UpdateBlock.forward conv.py:592-598 on the planar [3N,F] view); otherwise two cgvae_gemm launches. */
int cgvae_dense_pair_fwd(const float* x, int64_t ldx, const float* W, int64_t ldw, int64_t M, int64_t N1, int64_t N2,
                         int64_t K, float* C1, float* C2, cgvae_stream_t stream);
/* out[N] = sum over rows of X[M][N] (bias gradients); deterministic. */
int cgvae_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, cgvae_stream_t stream);

/* Grouped parameter gradients of Dense layers on small node sets (autograd of modules.py:99-112 /
 * nn.Linear for the 12..96-row decoder graphs): for every problem
 *   dW[n_out][n_in] = gy[rows][n_out]^T x[rows][n_in]   (dW contiguous; skipped when dW == NULL)
 *   db[n_out]       = column sums of gy                 (skipped when db == NULL)
 * All problems of the table are produced by ONE launch per 48 problems (the cost is writing dW, and one
 * launch per layer cannot keep enough stores in flight).  `problems` is a HOST array (the table is
 * passed to the device in the kernel parameters; it may be freed when the call returns); the pointers
 * inside are device pointers.  Row sums run in row order: deterministic.
 * seg_rows > 0: the operands are row-wise concatenations of rows / seg_rows matrices of seg_rows rows each, lying
 * seg_stride_g / seg_stride_x ELEMENTS apart -- the all-gathered factors of data-parallel ranks: the sum over ranks
 * of the per-rank gradients gy_r^T x_r is one contraction over all rows, in rank order (no gradient all-reduce). */
typedef struct cgvae_wgrad_problem {
  const float* gy;   /* [rows][n_out], row stride ldg */
  const float* x;    /* [rows][n_in], row stride ldx; may be NULL when dW is NULL */
  float* dW;         /* [n_out][n_in] contiguous, or NULL */
  float* db;         /* [n_out], or NULL */
  int32_t rows, n_out, n_in, ldg, ldx, seg_rows;
  int64_t seg_stride_g, seg_stride_x;
} cgvae_wgrad_problem;
int cgvae_wgrad_grouped(const cgvae_wgrad_problem* problems, int n_problems, cgvae_stream_t stream);

/* ------------------------------------------------------------------ message blocks */

/* One fused message layer = gather phi/v at the sender, filter w = basis*[Wf;bf], channel mixing and
 * deterministic CSR segment reduction into receivers, residual add.
 *   n_split 3: EquiMessageBlock.forward conv.py:505-563 and ContractiveMessageBlock.forward
 *              conv.py:703-733 (bipartite graph atoms -> beads)
 *   n_split 4: EquiMessageCross.forward conv.py:358-402 (v_recv = v; also writes q[n_recv][3][F] =
 *              sum_e m3 * v_j, saved for the backward)
 * phi[n_send][K][F], v_send[n_send][3][F]; res_s/res_v nullable residuals (cgvae.py:287-288);
 * v_is_zero != 0 skips the v gathers (first layer of every stack: cgvae.py:274,90). */
int cgvae_message_fwd(int n_split, const float* phi, const float* v_send, const float* v_recv,
                      const int32_t* rowptr, const int32_t* col, const float* basis, const float* unit,
                      const float* Wf, const float* bf, int64_t n_recv, int64_t n_send, int F, int R, int RB,
                      const float* res_s, const float* res_v, int v_is_zero,
                      float* out_s, float* out_v, float* q, cgvae_stream_t stream);

/* Backward of the above, reduced by SENDER over the transposed CSR (deterministic):
 * g_phi[n_send][K][F], g_v_send[n_send][3][F] (+= g_out_v pass-through when `residual`),
 * dWf[K*F][R], dbf[K*F].  n_split 4 also adds the receiver-side term q x g_out_v.
 * ws: cgvae_message_bwd_ws_bytes(n_split, F, RB, n_send). */
size_t cgvae_message_bwd_ws_bytes(int n_split, int F, int RB, int64_t n_send);
int cgvae_message_bwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const float* q,
                      const int32_t* rowptr_t, const int32_t* col_t, const int32_t* perm_t,
                      const float* basis, const float* unit, const float* Wf, const float* bf,
                      int64_t n_recv, int64_t n_send, int F, int R, int RB,
                      const float* g_out_s, const float* g_out_v, int residual, int v_is_zero,
                      float* g_phi, float* g_v_send, float* dWf, float* dbf,
                      void* ws, size_t ws_bytes, cgvae_stream_t stream);

/* Geometry cotangents of a message layer (csrc/message_geom.cu), run only when a coordinate requires grad.  Receiver-CSR
 * slot order, one store per edge, fixed summation order; same operands as cgvae_message_fwd plus the layer's output
 * gradients g_out_s[n_recv][F], g_out_v[n_recv][3][F].
 *   n_split 3, 4: d_basis[E][RB] = sum_k,f gm_k phi_j[k] Wf'[kF+f][.] with gm = (<g_v,v_j>, g_s, <g_v,u>, <g_v,v_i x v_j>),
 *                 d_unit[E][4] = (sum_f phi_j[2] w[2] g_v[c], 0)
 *   n_split 9:    unit-only form: d_unit from split 1 (EquiMessagePsuedo); d_basis and g_out_s unused (the caller forms
 *                 d_basis = gw Wf' from cgvae_message9_bwd's gw with cgvae_gemm).
 * Padded tail slots get zero. */
int cgvae_message_geom_bwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const int32_t* rowptr,
                           const int32_t* col, int64_t n_recv, int64_t n_edges, const float* basis, const float* unit,
                           const float* Wf, const float* bf, int F, int R, int RB, const float* g_out_s, const float* g_out_v,
                           int v_is_zero, float* d_basis, float* d_unit, cgvae_stream_t stream);

/* ---- the same layers on the 5th-generation tensor cores (csrc/message_tc.cu) ----
 * Column tiles of a CSR: rows are taken RC (4, 8 or 16) at a time; the columns of a chunk are (sorted union of the partner
 * nodes of its rows) x (the RC rows), 32 columns per batch record (both tf32 halves of the basis tile in the tensor core's
 * canonical K-major layout, unit vectors, partner ids; non-edges keep an all-zero basis row).  Built once per graph and
 * shared by all layers on it: forward tiles from the receiver CSR (rowptr, col, slot_map = NULL), backward tiles from the
 * sender CSR (rowptr_t, col_t, slot_map = perm_t: CSR slot whose basis / unit row the edge uses).
 *   nbatch[n_chunks] scratch, bptr[n_chunks+1] batch offsets, ngroups[n_chunks], rec[n_batches_cap * rec_bytes]. */
int64_t cgvae_msg_tiles_batches_cap(int64_t n_rows, int64_t n_partners, int64_t n_edge_slots, int RC);
size_t cgvae_msg_tiles_rec_bytes(void);
int cgvae_msg_tiles_build(const int32_t* rowptr, const int32_t* col, const int32_t* slot_map, int64_t n_rows,
                          int64_t n_partners, int64_t n_edge_slots, const float* basis, const float* unit, int RB, int RC,
                          int32_t* nbatch, int32_t* bptr, int32_t* ngroups, void* rec, int64_t n_batches_cap,
                          cgvae_stream_t stream);
/* cgvae_message_fwd on forward tiles: the filter rbf @ W_filter (modules.py:192-197) is a 3xTF32 tcgen05.mma per batch
 * (accumulators in TMEM, channels on the TMEM lanes), the sender rows are gathered once per (chunk, sender) and re-used
 * from registers for the RC receivers of the chunk.  Same outputs, same arguments as cgvae_message_fwd. */
size_t cgvae_message_tc_ws_bytes(int n_split, int RC, int64_t n_rows, int F);
int cgvae_message_tc_fwd(int n_split, const float* phi, const float* v_send, const float* v_recv, const int32_t* bptr,
                         const int32_t* ngroups, const void* rec, int64_t n_batches_cap, int RC, const float* Wf,
                         const float* bf, int64_t n_recv, int F, int R, const float* res_s, const float* res_v,
                         int v_is_zero, float* out_s, float* out_v, float* q, void* ws, size_t ws_bytes,
                         cgvae_stream_t stream);

/* EquiMessagePsuedo.forward conv.py:180-242 (9 splits) and its backward.  State (s, sbar, v, vbar)
 * on one node set; residual adds fused (cgvae.py:108-111).  The backward also needs the receiver CSR
 * (receiver-side gradient terms) and writes gw[E][9][F] (per-edge filter gradient, original CSR slot
 * order) from which the caller forms dWf = basis^T gw with cgvae_gemm(TN). */
int cgvae_message9_fwd(const float* phi, const float* s, const float* sbar, const float* v, const float* vbar,
                       const int32_t* rowptr, const int32_t* col, const float* basis, const float* unit,
                       const float* Wf, const float* bf, int64_t n, int F, int R, int RB, int residual,
                       float* out_s, float* out_sbar, float* out_v, float* out_vbar, cgvae_stream_t stream);
int cgvae_message9_bwd(const float* phi, const float* s, const float* sbar, const float* v, const float* vbar,
                       const int32_t* rowptr, const int32_t* col,
                       const int32_t* rowptr_t, const int32_t* col_t, const int32_t* perm_t,
                       const float* basis, const float* unit, const float* Wf, const float* bf,
                       int64_t n, int64_t n_edge_slots, int F, int R, int RB, int residual,
                       const float* g_s, const float* g_sbar, const float* g_v, const float* g_vbar,
                       float* gi_s, float* gi_sbar, float* gi_v, float* gi_vbar, float* g_phi, float* gw,
                       cgvae_stream_t stream);

/* ------------------------------------------------------------------ update block (conv.py:588-616) */

/* x[N][2F] = [ s | sqrt(sum_c (Vv_c^2 + 1e-10)) ]   (conv.py:600-601) */
int cgvae_update_norm_fwd(const float* s, const float* Vv, int64_t N, int F, float* x, cgvae_stream_t stream);
/* v_out = v + Uv*a_vv ; s_out = s + <Uv,Vv>*a_sv + a_ss,  q[N][3][F] = (a_vv,a_sv,a_ss)  (conv.py:603-614);
 * residual == 0 returns the deltas only (the reference block API). */
int cgvae_update_combine_fwd(const float* s, const float* v, const float* Uv, const float* Vv, const float* q,
                             int64_t N, int F, int residual, float* s_out, float* v_out, cgvae_stream_t stream);
/* -> gq[N][3][F], gUv[N][3][F], gVv[N][3][F] (the part that does not pass through the norm) */
int cgvae_update_combine_bwd(const float* Uv, const float* Vv, const float* q, const float* g_s, const float* g_v,
                             int64_t N, int F, float* gq, float* gUv, float* gVv, cgvae_stream_t stream);
/* gs_in = g_s + gx[:, :F] ; gVv += gx[:, F:] * Vv / nrm  (nrm = x[:, F:]) */
int cgvae_update_norm_bwd(const float* x, const float* Vv, const float* gx, const float* g_s,
                          int64_t N, int F, int residual, float* gs_in, float* gVv, cgvae_stream_t stream);
/* The same two kernels with gUv / gVv as column halves of ONE matrix [3N][ldg] (ldg = 2F, gVv = gUv + F): the input gradient
 * through u_mat and v_mat (conv.py:592-598; weights adjacent in memory) is then a single contraction over 2F. */
int cgvae_update_combine_bwd_ld(const float* Uv, const float* Vv, const float* q, const float* g_s, const float* g_v, int64_t N, int F,
                                float* gq, float* gUv, float* gVv, int64_t ldg, cgvae_stream_t stream);
int cgvae_update_norm_bwd_ld(const float* x, const float* Vv, const float* gx, const float* g_s, int64_t N, int F, int residual,
                             float* gs_in, float* gVv, int64_t ldg, cgvae_stream_t stream);

/* ------------------------------------------------------------------ pooling and lifting */

/* scatter_mean / scatter_add over the bead CSR (torch_scatter call sites cgvae.py:297-298,479;
 * datasets.py:487).  X[N][W] -> out[n_beads][W]; mean divides by max(count,1).  Backward gathers. */
int cgvae_segment_reduce_fwd(const float* X, const int32_t* rowptr_b, const int32_t* atoms, int64_t n_beads,
                             int64_t W, int mean, float* out, cgvae_stream_t stream);
int cgvae_segment_reduce_bwd(const float* g_out, const int64_t* mapping, const int32_t* rowptr_b, int64_t N,
                             int64_t W, int mean, float* g_X, cgvae_stream_t stream);
/* Embedding gather (cgvae.py:273,380,591): out[n] = table[idx[n]] ; idx int64.  n_rows > 0: ids outside
 * [0, n_rows) give a NaN row and set CGVAE_ERR_EMBED_INDEX (nn.Embedding raises IndexError). */
int cgvae_gather_rows(const float* table, const int64_t* idx, int64_t N, int64_t W, int64_t n_rows, float* out,
                      cgvae_stream_t stream);

/* Bead -> atom lifting, CGequiVAE.decoder cgvae.py:466-482 / PCN.decoder cgvae.py:556-576:
 * rel[n] = V[mapping[n]][:, rank[n]] ; mode 1: rel -= bead mean (offset=True); mode 2: rel[n] = 0 where
 * pin[n] != 0 (PCN C-alpha re-anchoring cgvae.py:569-571); xyz_out = rel + cg_xyz[mapping].
 * Backward writes g_V[n_beads][3][F] (zero filled by the call). */
int cgvae_lift_fwd(const float* V, const float* cg_xyz, const int64_t* mapping, const int64_t* rank,
                   const int32_t* rowptr_b, const int32_t* atoms, const uint8_t* pin, int64_t N, int64_t n_beads,
                   int F, int mode, float* xyz_out, cgvae_stream_t stream);
int cgvae_lift_bwd(const float* g_xyz, const int64_t* mapping, const int64_t* rank, const int32_t* rowptr_b,
                   const int32_t* atoms, const uint8_t* pin, int64_t N, int64_t n_beads, int F, int mode,
                   float* g_V, cgvae_stream_t stream);

/* ------------------------------------------------------------------ optimiser step */

/* torch.nn.utils.clip_grad_norm_(params, max_norm) + torch.optim.Adam.step() (scripts/utils.py:151-157) fused over flat
 * buffers p / g / m / v of n floats (train.FlatGrads lays parameters and gradients out contiguously).  `step` is a device
 * float holding the number of steps taken so far (incremented by the call: graph-replay safe); norm_out (nullable)
 * receives the unclipped gradient norm.  The gradient buffer itself is left unscaled.  grad_scale: the gradients
 * are taken as grad_scale * g (1/world after a data-parallel all-reduce(sum): saves the separate scaling pass; 1.0f
 * otherwise).  ws: cgvae_adam_ws_bytes().
 * Skip guard of the reference loop (scripts/utils.py:145-148: `if loss.item() >= gamma*200 or isnan(loss): continue`),
 * decided on the device: with loss != NULL the step is a no-op (p / m / v / step untouched, skipped[0] += 1 when
 * skipped != NULL) if loss[0]*loss_scale is NaN or >= loss_limit; a non-finite gradient norm is skipped too (it would
 * otherwise be written into the moments and parameters).  loss_scale = 1/world when loss[0] is an all-reduced sum. */
size_t cgvae_adam_ws_bytes(void);
int cgvae_adam_clip_step(float* p, const float* g, float* m, float* v, int64_t n, float max_norm, float grad_scale,
                         float lr, float beta1, float beta2, float eps, float* step, float* norm_out,
                         const float* loss, float loss_scale, float loss_limit, float* skipped, void* ws,
                         size_t ws_bytes, cgvae_stream_t stream);
/* The same update for a data-parallel run that shards the optimiser (reduce-scatter of the gradients, Adam on this rank's
 * 1/world slice, all-gather of the parameters): cgvae_grad_sumsq leaves the 1024 partial sums of squares of the local slice
 * in ws[0..1024) and a copy of loss[0] in ws[1024]; the caller all-reduces (SUM) the 1025 floats; cgvae_adam_apply then clips
 * with the GLOBAL norm, applies the skip guard on ws[1024] * loss_scale (use_ws_loss != 0) and updates the slice. */
int cgvae_grad_sumsq(const float* g, int64_t n, const float* loss, void* ws, size_t ws_bytes, cgvae_stream_t stream);
int cgvae_adam_apply(float* p, const float* g, float* m, float* v, int64_t n, float max_norm, float grad_scale, float lr, float beta1,
                     float beta2, float eps, float* step, float* norm_out, int use_ws_loss, float loss_scale, float loss_limit,
                     float* skipped, void* ws, size_t ws_bytes, cgvae_stream_t stream);

/* ------------------------------------------------------------------ losses and the VAE latent

 * sigma = 1e-12 + exp(logvar / 2), z = eps * sigma + mu (cgvae.py:445-449,500-507; z == NULL: sigma only) and its
 * backward g_mu = g_z, g_logvar = (g_sigma + g_z * eps) * 0.5 * (sigma - 1e-12) (g_z / g_sigma / eps / g_mu nullable). */
int cgvae_vae_latent_fwd(const float* mu, const float* logvar, const float* eps, int64_t n, float* sigma, float* z,
                         cgvae_stream_t stream);
int cgvae_vae_latent_bwd(const float* g_z, const float* g_sigma, const float* eps, const float* sigma, int64_t n, float* g_mu,
                         float* g_logvar, cgvae_stream_t stream);
/* y = c + exp(x / 2) (prior std, cgvae.py:401: c = 1e-9) ; gx = gy * 0.5 * (y - c) */
int cgvae_std_logvar_fwd(const float* x, int64_t n, float c, float* y, cgvae_stream_t stream);
int cgvae_std_logvar_bwd(const float* gy, const float* y, int64_t n, float c, float* gx, cgvae_stream_t stream);
/* Loss of the training loop, scripts/utils.py:81-141: out4 = (loss, recon, kl, graph) with
 *   loss = mean((xyz_rec - xyz)^2) + beta * KL(mu, sigma || pmu, pstd) + gamma * mean over bonds of (|rec_a - rec_b|_e - |x_a - x_b|_e)^2,
 * |.|_e = sqrt(sum^2 + 1e-6); KL keeps the reference's division by pstd (not pstd^2, utils.py:85); pmu == NULL: KL against
 * the standard normal (utils.py:82-83); mu == NULL: no KL term (PCN).  The bonds come as the receiver CSR of the
 * SYMMETRISED bond list (cgvae_csr_count / cgvae_csr_fill with symmetrize = 1): every list entry is seen from both atoms,
 * the forward halves the doubled sum and the backward is a per-atom gather (deterministic; no index_put).  norms
 * (nullable device float[3]): denominators (atoms, beads, bonds) for data-parallel training (global count / world).
 * Two launches each way; reductions in a fixed order.  ws: cgvae_loss_ws_bytes(). */
size_t cgvae_loss_ws_bytes(void);
int cgvae_loss_fwd(const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr, const int32_t* bond_col,
                   const float* mu, const float* sigma, const float* pmu, const float* pstd, int64_t n_beads, int F,
                   const float* norms, float beta, float gamma, float* out4, void* ws, size_t ws_bytes,
                   cgvae_stream_t stream);
int cgvae_loss_bwd(const float* g_loss, const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr,
                   const int32_t* bond_col, const float* mu, const float* sigma, const float* pmu, const float* pstd,
                   int64_t n_beads, int F, const float* norms, float beta, float gamma, float* g_xyz_rec, float* g_mu,
                   float* g_sigma, float* g_pmu, float* g_pstd, cgvae_stream_t stream);
/* Gradient of the same loss to the TARGET coordinates xyz (needed when xyz is also differentiated as the encoder input):
 * minus the reconstruction term's gradient plus the bond term's gradient to the target distances |x_a - x_b|_e, gathered
 * over the same symmetrised bond CSR with the same norms.  g_xyz[n_atoms][3].  One launch, deterministic. */
int cgvae_loss_bwd_target(const float* g_loss, const float* xyz, const float* xyz_rec, int64_t n_atoms, const int32_t* bond_rowptr,
                          const int32_t* bond_col, const float* norms, float gamma, float* g_xyz, cgvae_stream_t stream);
/* Dihedral loss of the PCN loop (scripts/pcn_utils.py:114-132 compute_dihe, :178-180):
 *   out[0] = mean_d (theta(xyz_rec; idx[d]) - theta(xyz; idx[d]))^2,  theta = atan(p1 / (p2 + 1e-6)) exactly as the reference
 * forms it (b1..b3, c1 = b2 x b3, c2 = b1 x b2, p1 = (b1.c1) sqrt(b2.b2 + 1e-6), p2 = c1.c2).  idx int64 [n_dihe][4];
 * n_live (nullable device int64): live rows of a zero-padded static list; norm (nullable device float): denominator for
 * data-parallel training.  contrib float [n_dihe][4][3]: per-(dihedral, slot) gradients kept for the backward, which is a
 * per-atom gather over the receiver CSR of the flattened list (cgvae_csr_* on pairs (idx[d][s], 4 d + s)): deterministic.
 * ws: 256 floats. */
int cgvae_dihedral_loss_fwd(const float* xyz, const float* xyz_rec, const int64_t* idx, int64_t n_dihe, const int64_t* n_live,
                            const float* norm, float* contrib, float* out, void* ws, size_t ws_bytes, cgvae_stream_t stream);
int cgvae_dihedral_loss_bwd(const float* g_loss, const float* contrib, const int32_t* rowptr, const int32_t* col, int64_t n_atoms,
                            int64_t n_dihe, const int64_t* n_live, const float* norm, float* g_xyz_rec, cgvae_stream_t stream);
/* PCN C-alpha pin mask with the predicate of cgvae.py:569-571 evaluated on the device: pin[0..n_atoms) = 0, then
 * pin[idx[i]] = 1 for the live entries iff idx[last] < n_atoms.  pin_bytes >= n_atoms, a multiple of 4. */
int cgvae_pin_mask(const int64_t* idx, int64_t n_idx, const int64_t* n_live, int64_t n_atoms, uint8_t* pin, size_t pin_bytes,
                   cgvae_stream_t stream);
/* ------------------------------------------------------------------ ragged batch collation

 * SCNCGDataset.__getitem__ + SCNCG_collate (data.py:292-398) for a protein set resident in device memory
 * (data.DeviceProteinDataset).  Each kind of row has one concatenated store (rows of item p: item_ptr[kind][p] ..
 * item_ptr[kind][p+1]); idx[n_slots] selects the items of a batch, -1 = empty slot.  One output per stored array:
 * rows [0, live) = the selected items' rows concatenated in slot order, each int64 row plus the running count of kind
 * add_kind of the slots before it (the collate offsets); rows [live, rows) = pad: zero, or with pad_beads the pad bead
 * counts[RESIDUES] + k / atoms_per_bead of pad row k (clamped to n_beads - 1).  counts[kind] = min(total, live_cap[kind]);
 * a larger total, or an idx entry outside [-1, n_items), sets CGVAE_ERR_COLLATE_BIT and writes nothing past any `rows`.
 * count_out[kind] (each nullable) receive copies of counts; norms (nullable float[3]) = max(1, counts) of (atoms,
 * residues, bonds): the loss denominators.  slot_off: workspace [KINDS][n_slots+1] (the per-slot output offsets).
 * `plan` is a HOST struct (it travels in the kernel parameters); the pointers inside are device pointers.  Two
 * launches, no host synchronisation, CUDA-graph capturable; integer rows are exact copies. */
enum { CGVAE_COLLATE_ATOMS = 0, CGVAE_COLLATE_RESIDUES = 1, CGVAE_COLLATE_BONDS = 2, CGVAE_COLLATE_EDGES = 3,
       CGVAE_COLLATE_DIHEDRALS = 4, CGVAE_COLLATE_CA = 5, CGVAE_COLLATE_KINDS = 6, CGVAE_COLLATE_MAX_OUT = 8 };
typedef struct cgvae_collate_out {
  void* dst;                /* [rows][width] */
  const void* src;          /* store of the output's kind, [item_ptr[kind][n_items]][width] */
  int64_t rows;             /* capacity rows of dst */
  int32_t width, elem_bytes; /* elements per row; 4 (float32) or 8 (int64) */
  int32_t kind, add_kind;   /* count kind of the rows; kind whose running count is added (-1: none) */
  int32_t pad_beads, reserved;
} cgvae_collate_out;
typedef struct cgvae_collate_plan {
  const int64_t* idx;       /* [n_slots] */
  const int64_t* item_ptr;  /* [KINDS][n_items+1] */
  int64_t* slot_off;        /* [KINDS][n_slots+1] workspace */
  int64_t* counts;          /* [KINDS] */
  int64_t* count_out[CGVAE_COLLATE_KINDS];
  float* norms;
  int64_t n_slots, n_items, atoms_per_bead, n_beads;
  int64_t live_cap[CGVAE_COLLATE_KINDS];
  int32_t n_out, reserved;
  cgvae_collate_out out[CGVAE_COLLATE_MAX_OUT];
} cgvae_collate_plan;
size_t cgvae_collate_plan_bytes(void);
int cgvae_collate(const cgvae_collate_plan* plan, cgvae_stream_t stream);
/* Sample-quality metrics of the ensemble-sampling loop (scripts/sampling.py:120-194,220-239,324-333).
 * cgvae_bond_graph: bond[i][j] = (i != j) && sqrt(((dx^2+dy^2)+dz^2)) < (radius[i] + radius[j]) * scale, in fp32 and in the
 * reference's operation order (bit-exact adjacency); radius = covalent cutoff radius per atom (COVCUTOFFTABLE, sampling.py:12-118).
 * cgvae_sample_quality: for every sample s of samples[n_samples][n][3] against the reference conformation:
 *   counts[s] = { #(gen != ref), sum(ref - gen), sum(ref) } over all ordered atom pairs, then the same three over pairs of heavy
 *   atoms (heavy[i] != 0) -- compare_graph / graph_diff_ratio of count_valid_graphs with heavy_only False / True;
 *   rmsd[s] = { all-atom, heavy-atom } root-mean-square deviation without alignment (compute_rmsd). */
int cgvae_bond_graph(const float* xyz, const float* radius, int64_t n, float scale, uint8_t* bond, cgvae_stream_t stream);
int cgvae_sample_quality(const float* ref_xyz, const float* samples, const float* radius, const uint8_t* heavy, int64_t n,
                         int64_t n_samples, float scale, int32_t* counts, float* rmsd, cgvae_stream_t stream);
/* Programmatic dependent launch for every launch of the library from now on (default on; CGVAE_PDL=0); returns the previous
 * setting.  Launches already captured in a CUDA graph keep the edges they were captured with. */
int cgvae_set_pdl(int on);
/* Precision of the tensor-core contractions for every launch from now on; returns the previous mode.
 *   0 = 3xTF32, fp32 parity (1e-5 relative); the default, like torch.set_float32_matmul_precision("highest");
 *   1 = 1xTF32, operands rounded to nearest TF32 (10-bit mantissa), fp32 accumulation, like torch's "high": stated bound
 *       4 * 2^-11 scale-relative per contraction with zero-mean operands.
 * It covers the tcgen05 GEMMs (>= 64 rows) and the filter of cgvae_message_tc_fwd; everything else stays fp32 in both
 * modes (SIMT GEMM tiles, weight-streaming GEMMs, cgvae_wgrad_grouped, cgvae_colsum, the message backward, the 9-split
 * kernels).  The dispatch (tiles, split-K, grid) is the same in both modes.  Launches already captured in a CUDA graph keep
 * the kernels they were captured with.  Any other mode: argument error, mode unchanged. */
int cgvae_set_matmul_precision(int mode);
/* the current mode of cgvae_set_matmul_precision (0 or 1) */
int cgvae_get_matmul_precision(void);
/* Declare [p, p + bytes) a parameter range: memory no kernel writes between two optimiser steps (the flat parameter buffer of
 * a training step).  With programmatic dependent launch enabled (CGVAE_PDL, default on) the weight-streaming GEMMs fetch a
 * weight matrix inside such a range BEFORE their dependency wait, overlapping the copy with the preceding kernel.  Ranges that
 * touch are merged; p == NULL clears the table. */
int cgvae_register_const_range(const void* p, size_t bytes);
/* p[0..n) = value (initial decoder state cgvae.py:90-95 without a library fill) */
int cgvae_fill(float* p, int64_t n, float value, cgvae_stream_t stream);

/* layout conversion at the module boundary: reference v[N][F][3] <-> planar v[N][3][F] */
int cgvae_vec_to_planar(const float* v_nf3, int64_t N, int F, float* v_n3f, cgvae_stream_t stream);
int cgvae_vec_from_planar(const float* v_n3f, int64_t N, int F, float* v_nf3, cgvae_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CGVAE_B200_H_ */
