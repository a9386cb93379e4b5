"""Autograd nodes of the hot path: every forward and every backward is a short sequence of C-ABI
kernel launches (ops.py); PyTorch only owns memory and the tape.  Gradients flow to features and
parameters, and to atom / bead coordinates (or the r_ij of the block API) when one of them requires
grad: the edge geometry then becomes an EdgeGeometry node and the message layers also return the
cotangents of its basis / unit records (DESIGN.md section 4).

Backward formulas: SURVEY.md Appendix A (checked against the oracle's autograd in tests/).
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import ops

SWISH = 1


def _phi_forward(s, W1, b1, W2, b2, act=SWISH):
    a1, z1 = ops.linear_fwd(s, W1, b1, act, save_pre=True)
    phi = ops.linear_fwd(a1, W2, b2, 0)
    return a1, z1, phi


def _phi_backward(g_phi2d, s, a1, z1, W1, b1, W2, b2, add_to_gs, act=SWISH):
    """backward of phi = Dense2(act(Dense1(s))) given g_phi [N, K*F]; returns gs (+add), gW1, gb1, gW2, gb2."""
    fork = ops.Fork(g_phi2d.device, enabled=not ops.deferring(g_phi2d.shape[0]))   # deferred: nothing to overlap
    gz1 = ops.linear_bwd_input(g_phi2d, W2, z_in=z1, dact=act)            # (g_phi W2) * act'(z1)
    with fork.branch():                                                   # parameter gradients: off the critical path
        gW2 = ops.linear_bwd_weight(g_phi2d, a1, W2)
        gb2 = ops.colsum(g_phi2d, b2)
    fork.sync()
    gs = ops.linear_bwd_input(gz1, W1, add=add_to_gs)
    with fork.branch():
        gW1 = ops.linear_bwd_weight(gz1, s, W1)
        gb1 = ops.colsum(gz1, b1)
    fork.join()
    return gs, gW1, gb1, gW2, gb2


class MLP2(Function):
    """y = Dense2(act(Dense1(x))): the phi-MLP of InvariantMessage (conv.py:41-49) and the Linear-act-Linear heads
    (atom_munet / atom_sigmanet scripts/run_ala.py:184-185, CGprior.mu / .sigma cgvae.py:368-369)."""

    @staticmethod
    def forward(ctx, act, x, W1, b1, W2, b2):
        x = x.contiguous()
        a1, z1, y = _phi_forward(x, W1, b1, W2, b2, act)
        ctx.act = act
        ctx.save_for_backward(x, a1, z1, W1, b1, W2, b2)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, a1, z1, W1, b1, W2, b2 = ctx.saved_tensors
        gx, gW1, gb1, gW2, gb2 = _phi_backward(gy.contiguous(), x, a1, z1, W1, b1, W2, b2, None, ctx.act)
        return None, gx, gW1, gb1, gW2, gb2


class LinearFn(Function):
    """y = x W^T + b (nn.Linear): the non-equivariant decoder head cgvae.py:469-471."""

    @staticmethod
    def forward(ctx, x, W, b):
        x = x.contiguous()
        ctx.save_for_backward(x, W, b)
        return ops.linear_fwd(x, W, b, 0)

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, W, b = ctx.saved_tensors
        gy = gy.contiguous()
        fork = ops.Fork(gy.device, enabled=not ops.deferring(gy.shape[0]))
        gx = ops.linear_bwd_input(gy, W)
        with fork.branch():
            gW = ops.linear_bwd_weight(gy, x, W)
            gb = ops.colsum(gy, b) if b is not None else None
        fork.join()
        return gx, gW, gb


def _requires_grad(*tensors):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


class EdgeGeometry(Function):
    """ops.edge_geometry as an autograd node (same launch, same bits); backward = the geometry backward plus the node
    reductions to the sender / receiver coordinates, or the gradient of r_edge.  xyz_recv None: one coordinate tensor
    for both ends of every edge (atom graph, CG graph)."""

    @staticmethod
    def forward(ctx, graph, n_rbf, cutoff, xyz_send, xyz_recv, r_edge, edge_wgt):
        same = xyz_send is not None and xyz_recv is None
        geom = ops.edge_geometry(graph, xyz_send, xyz_send if same else xyz_recv, n_rbf, cutoff, edge_wgt=edge_wgt, r_edge=r_edge)
        ctx.graph, ctx.n_rbf, ctx.cutoff, ctx.same = graph, n_rbf, cutoff, same     # not geom: it holds the outputs
        ctx.save_for_backward(xyz_send, xyz_recv, r_edge, edge_wgt)
        return geom.basis, geom.unit

    @staticmethod
    @once_differentiable
    def backward(ctx, d_basis, d_unit):
        xyz_send, xyz_recv, r_edge, edge_wgt = ctx.saved_tensors
        if ctx.needs_input_grad[6]:
            raise NotImplementedError("coordinate gradients: the gradient to edge_wgt is not implemented")
        dr = ops.edge_geometry_bwd(ctx.graph, ctx.n_rbf, ctx.cutoff, xyz_send, xyz_send if ctx.same else xyz_recv, d_basis, d_unit,
                                   edge_wgt, r_edge)
        if r_edge is not None:
            return None, None, None, None, None, dr, None
        g_send, g_recv = ops.edge_coord_reduce(ctx.graph, dr, ctx.same)
        return None, None, None, g_send, g_recv, None, None


def edge_geometry(graph, xyz_send, xyz_recv, n_rbf, cutoff, edge_wgt=None, r_edge=None):
    """ops.edge_geometry, differentiable when grad mode is on and a coordinate, r_edge or edge_wgt requires grad (the
    only case in which the geometry backward kernels run); otherwise the plain launch."""
    if not _requires_grad(xyz_send, xyz_recv, r_edge, edge_wgt):
        return ops.edge_geometry(graph, xyz_send, xyz_recv, n_rbf, cutoff, edge_wgt=edge_wgt, r_edge=r_edge)
    same = xyz_send is xyz_recv
    basis, unit = EdgeGeometry.apply(graph, n_rbf, cutoff, xyz_send, None if same else xyz_recv, r_edge, edge_wgt)
    return ops.Geometry(graph, basis, unit, n_rbf, ops.rb_for(n_rbf), cutoff)


class MessageBlock(Function):
    """InvariantMessage + EquiMessageBlock (n_split 3, conv.py:505-563) / EquiMessageCross (4, conv.py:358-402) /
    ContractiveMessageBlock (3 on the atoms->beads graph, conv.py:703-733).

    mode 'self'  : out = (s, v) + message   (stack use, residual of cgvae.py:287-288 fused)
    mode 'delta' : out = message            (the reference block API)
    mode 'other' : out = (res_s, res_v) + message, residual state on the receiver set (contraction)
    v None means v == 0 (first layer of every stack) and skips the vector gathers.
    basis / unit are geom.basis / geom.unit, inputs so that their cotangents reach an EdgeGeometry node.
    """

    @staticmethod
    def forward(ctx, geom, n_split, mode, act, s, v, res_s, res_v, W1, b1, W2, b2, Wf, bf, basis, unit):
        s = s.contiguous()
        a1, z1, phi = _phi_forward(s, W1, b1, W2, b2, act)
        N, F = s.shape
        phi3 = phi.view(N, n_split, F)
        if mode == "self":
            rs, rv = s, v
        elif mode == "other":
            rs, rv = res_s, res_v
        else:
            rs, rv = None, None
        out_s, out_v, q = ops.message_fwd(n_split, phi3, v, v if n_split == 4 else None, geom, Wf, bf, rs, rv,
                                          want_q=(n_split == 4 and v is not None))
        ctx.geom, ctx.n_split, ctx.mode, ctx.act = geom, n_split, mode, act
        ctx.v_none = v is None
        ctx.res_v_none = res_v is None
        ctx.save_for_backward(s, v, a1, z1, phi3, q, W1, b1, W2, b2, Wf, bf)
        return out_s, out_v

    @staticmethod
    @once_differentiable
    def backward(ctx, g_s, g_v):
        s, v, a1, z1, phi3, q, W1, b1, W2, b2, Wf, bf = ctx.saved_tensors
        g_s, g_v = g_s.contiguous(), g_v.contiguous()
        n_split, mode = ctx.n_split, ctx.mode
        residual = mode == "self"
        # with v == 0 and a fused residual the sender-side pass-through still applies (v_out = 0 + dv):
        g_phi, g_v_send, dWf, dbf = ops.message_bwd(n_split, phi3, v, v if n_split == 4 else None, q, ctx.geom, Wf, bf,
                                                    g_s, g_v, residual and not ctx.v_none)
        N, F = s.shape
        gs, gW1, gb1, gW2, gb2 = _phi_backward(g_phi.view(N, n_split * F), s, a1, z1, W1, b1, W2, b2,
                                               g_s if residual else None, ctx.act)
        gv = None if ctx.v_none else g_v_send
        g_res_s = g_s if mode == "other" else None
        g_res_v = g_v if (mode == "other" and not ctx.res_v_none) else None
        d_basis = d_unit = None
        if ctx.needs_input_grad[14] or ctx.needs_input_grad[15]:
            d_basis, d_unit = ops.message_geom_bwd(n_split, phi3, v, v if n_split == 4 else None, ctx.geom, Wf, bf, g_s, g_v)
        return None, None, None, None, gs, gv, g_res_s, g_res_v, gW1, gb1, gW2, gb2, dWf, dbf, d_basis, d_unit


class Message9Block(Function):
    """InvariantMessage (9 splits) + EquiMessagePsuedo, conv.py:180-242; residual adds of cgvae.py:108-111 fused."""

    @staticmethod
    def forward(ctx, geom, residual, act, s, sbar, v, vbar, W1, b1, W2, b2, Wf, bf, basis, unit):
        s, sbar, v, vbar = s.contiguous(), sbar.contiguous(), v.contiguous(), vbar.contiguous()
        a1, z1, phi = _phi_forward(s, W1, b1, W2, b2, act)
        N, F = s.shape
        phi3 = phi.view(N, 9, F)
        outs = ops.message9_fwd(phi3, s, sbar, v, vbar, geom, Wf, bf, residual)
        ctx.geom, ctx.residual, ctx.act = geom, residual, act
        ctx.save_for_backward(s, sbar, v, vbar, a1, z1, phi3, W1, b1, W2, b2, Wf, bf)
        return tuple(outs)

    @staticmethod
    @once_differentiable
    def backward(ctx, g_s, g_sbar, g_v, g_vbar):
        s, sbar, v, vbar, a1, z1, phi3, W1, b1, W2, b2, Wf, bf = ctx.saved_tensors
        geom_grad = ctx.needs_input_grad[13] or ctx.needs_input_grad[14]
        g_v = g_v.contiguous()
        args = (phi3, s, sbar, v, vbar, ctx.geom, Wf, bf, ctx.residual, g_s.contiguous(), g_sbar.contiguous(), g_v,
                g_vbar.contiguous())
        outs = ops.message9_bwd(*args, keep_gw=True) if geom_grad else ops.message9_bwd(*args)
        gi_s, gi_sbar, gi_v, gi_vbar, g_phi, dWf, dbf = outs[:7]
        d_basis = d_unit = None
        if geom_grad:
            d_basis, d_unit = ops.message9_geom_bwd(phi3, ctx.geom, Wf, bf, outs[7], g_v)
        N, F = s.shape
        gs, gW1, gb1, gW2, gb2 = _phi_backward(g_phi.view(N, 9 * F), s, a1, z1, W1, b1, W2, b2, gi_s, ctx.act)
        return None, None, None, gs, gi_sbar, gi_v, gi_vbar, gW1, gb1, gW2, gb2, dWf, dbf, d_basis, d_unit


class UpdateBlockFn(Function):
    """UpdateBlock.forward conv.py:588-616 on planar vectors; residual of cgvae.py:122-123 optionally fused."""

    @staticmethod
    def forward(ctx, residual, act, s, v, U, V, A0, c0, A1, c1):
        s, v = s.contiguous(), v.contiguous()
        N, F = s.shape
        v2 = v.view(3 * N, F)
        Uv, Vv = ops.linear_pair_fwd(v2, U, V)          # one launch when U and V are adjacent in the flat parameter buffer
        Uv, Vv = Uv.view(N, 3, F), Vv.view(N, 3, F)
        x = ops.update_norm_fwd(s, Vv)
        h, z = ops.linear_fwd(x, A0, c0, act, save_pre=True)
        q = ops.linear_fwd(h, A1, c1, 0).view(N, 3, F)
        s_out, v_out = ops.update_combine_fwd(s, v, Uv, Vv, q, residual)
        ctx.residual, ctx.act = residual, act
        ctx.save_for_backward(v, Uv, Vv, x, h, z, q, U, V, A0, c0, A1, c1)
        return s_out, v_out

    @staticmethod
    @once_differentiable
    def backward(ctx, g_s, g_v):
        v, Uv, Vv, x, h, z, q, U, V, A0, c0, A1, c1 = ctx.saved_tensors
        g_s, g_v = g_s.contiguous(), g_v.contiguous()
        N, _, F = v.shape
        # u_mat and v_mat adjacent in memory (the flat parameter buffer of a training step): their two input-gradient mixes
        # share the output, so gUv / gVv are produced as the column halves of one [3N, 2F] matrix and contracted once with
        # [U; V] ([2F, F]) -- one launch and one pass over the [3N, F] output instead of two
        pair = (U.is_cuda and U.is_contiguous() and V.is_contiguous() and U.shape == V.shape
                and V.data_ptr() == U.data_ptr() + 4 * U.numel()
                and U.untyped_storage().data_ptr() == V.untyped_storage().data_ptr())     # views of ONE buffer ([U; V] view below)
        gq, gUv, gVv = ops.update_combine_bwd(Uv, Vv, q, g_s, g_v, cat=pair)
        gq2 = gq.view(N, 3 * F)
        v2 = v.view(3 * N, F)
        if pair:
            gUV2 = gUv.as_strided((3 * N, 2 * F), (2 * F, 1))
            gUv2, gVv2 = gUV2[:, :F], gUV2[:, F:]
        else:
            gUv2, gVv2 = gUv.view(3 * N, F), gVv.view(3 * N, F)
        fork = ops.Fork(g_s.device, enabled=not ops.deferring(3 * N))
        gz = ops.linear_bwd_input(gq2, A1, z_in=z, dact=ctx.act)
        with fork.branch():                                                 # parameter gradients: off the critical path
            gA1 = ops.linear_bwd_weight(gq2, h, A1)
            gc1 = ops.colsum(gq2, c1)
            if not pair:
                gU = ops.linear_bwd_weight(gUv2, v2, U)
        fork.sync()
        gx = ops.linear_bwd_input(gz, A0)
        with fork.branch():
            gA0 = ops.linear_bwd_weight(gz, x, A0)
            gc0 = ops.colsum(gz, c0)
        gs_in = ops.update_norm_bwd(x, Vv, gx, g_s, gVv, ctx.residual)      # adds the norm path into gVv in place
        fork.sync()
        if pair:
            UV = U.as_strided((2 * F, U.shape[1]), (U.shape[1], 1))
            gv_in = ops.linear_bwd_input(gUV2, UV, add=g_v.view(3 * N, F) if ctx.residual else None).view(N, 3, F)
        else:
            gv_in = ops.linear_bwd_input(gUv2, U, add=g_v.view(3 * N, F) if ctx.residual else None)
            gv_in = ops.linear_bwd_input(gVv2, V, add=gv_in).view(N, 3, F)
        with fork.branch():
            if pair:
                # [gU; gV] = [gUv | gVv]^T v: one contraction into the adjacent gradient regions of u_mat and v_mat
                gUVw = ops.linear_bwd_weight(gUV2, v2, U, shape=(2 * F, U.shape[1]))
                gU, gV = gUVw[:F], gUVw[F:]
            else:
                gV = ops.linear_bwd_weight(gVv2, v2, V)
        fork.join()
        return None, None, gs_in, gv_in, gU, gV, gA0, gc0, gA1, gc1


class SegmentReduce(Function):
    """scatter_mean / scatter_add over beads (cgvae.py:297-298): X [N,...] -> [n_beads,...]."""

    @staticmethod
    def forward(ctx, seg, mean, X):
        ctx.seg, ctx.mean = seg, mean
        return ops.segment_reduce_fwd(X.contiguous(), seg, mean)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        return None, None, ops.segment_reduce_bwd(g.contiguous(), ctx.seg, ctx.mean)


class EmbeddingLookup(Function):
    """nn.Embedding(100, F, padding_idx=0) lookup (cgvae.py:273,380,591); deterministic gradient."""

    @staticmethod
    def forward(ctx, table, idx, padding_idx):
        idx = idx.to(torch.int64).contiguous()
        ctx.padding_idx = padding_idx
        ctx.n_rows = table.shape[0]
        ctx.save_for_backward(idx, table)
        return ops.gather_rows(table, idx)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        idx, table = ctx.saved_tensors
        n = idx.numel()
        if ctx.padding_idx is not None and n > 2048:
            # the padding row's gradient is discarded: its entries go to spare rows of <= 1024 each, past the table, so that
            # no row outgrows the 2048-entry shared-memory sort of graph.cu (a capacity-padded protein batch holds
            # thousands of pad residues); the other rows keep their entries in the same order
            spare = -(-n // 1024)
            pos = torch.arange(n, dtype=torch.int64, device=idx.device).remainder_(spare).add_(ctx.n_rows)
            seg = ops.build_segments(torch.where(idx == ctx.padding_idx, pos, idx), ctx.n_rows + spare)
            seg = ops.Segments(ctx.n_rows, seg.mapping, seg.rowptr, seg.atoms, seg.slot, seg.rank)
        else:
            seg = ops.build_segments(idx, ctx.n_rows)
        gt = ops.segment_reduce_fwd(g.contiguous(), seg, False, param=table)
        if ctx.padding_idx is not None:
            gt[ctx.padding_idx].zero_()
        return gt, None, None


class Lift(Function):
    """bead -> atom lifting (cgvae.py:466-482; PCN cgvae.py:556-576): V [Nc,3,F] -> xyz [N,3].  Every atom is its bead's
    position plus an offset, in all three modes, so the gradient to cg_xyz is the per-bead sum of the atom gradients."""

    @staticmethod
    def forward(ctx, seg, mode, pin, V, cg_xyz):
        ctx.seg, ctx.mode, ctx.pin, ctx.F = seg, mode, pin, V.shape[-1]
        return ops.lift_fwd(V.contiguous(), cg_xyz, seg, mode, pin)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        g = g.contiguous()
        g_cg = ops.segment_reduce_fwd(g, ctx.seg, False) if ctx.needs_input_grad[4] else None
        return None, None, None, ops.lift_bwd(g, ctx.seg, ctx.F, ctx.mode, ctx.pin), g_cg


class VAELatent(Function):
    """(z, sigma) = (eps * sigma + mu, 1e-12 + exp(logvar / 2)): the posterior scale and the reparametrisation of
    cgvae.py:445-449,500-507 in one launch (three element-wise launches + their backward in the reference)."""

    @staticmethod
    def forward(ctx, mu, logvar, eps):
        z, sigma = ops.vae_latent_fwd(mu, logvar, eps)
        ctx.save_for_backward(eps, sigma)
        return z, sigma

    @staticmethod
    @once_differentiable
    def backward(ctx, g_z, g_sigma):
        eps, sigma = ctx.saved_tensors
        g_mu, g_logvar = ops.vae_latent_bwd(g_z.contiguous() if g_z is not None else None,
                                            g_sigma.contiguous() if g_sigma is not None else None, eps, sigma)
        return g_mu, g_logvar, None


class StdLogvar(Function):
    """y = c + exp(x / 2): the prior std (cgvae.py:401, c = 1e-9) and the posterior std when no sample is drawn."""

    @staticmethod
    def forward(ctx, x, c):
        y = ops.std_logvar_fwd(x, c)
        ctx.c = c
        ctx.save_for_backward(y)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        (y,) = ctx.saved_tensors
        return ops.std_logvar_bwd(gy.contiguous(), y, ctx.c), None


class TrainingLoss(Function):
    """scripts/utils.py:117-141 as one node: returns (loss [1], components [4] = loss, recon, kl, graph; not differentiable).
    Gradients flow to xyz_recon, mu, sigma and the prior mean / std, and to the target xyz when it requires grad (the
    encoder input of a CGequiVAE batch whose coordinates are differentiated); the bond term uses the CSR of the symmetrised
    bond list."""

    @staticmethod
    def forward(ctx, bond_graph, beta, gamma, norms, xyz, xyz_rec, mu, sigma, pmu, pstd):
        xyz, xyz_rec = xyz.contiguous(), xyz_rec.contiguous()
        if mu is not None:
            mu, sigma = mu.contiguous(), sigma.contiguous()
        if pmu is not None:
            pmu, pstd = pmu.contiguous(), pstd.contiguous()
        out4 = ops.loss_fwd(xyz, xyz_rec, bond_graph, mu, sigma, pmu, pstd, norms, beta, gamma)
        ctx.bond_graph, ctx.beta, ctx.gamma, ctx.norms = bond_graph, beta, gamma, norms
        ctx.has = (mu is not None, pmu is not None)
        ctx.save_for_backward(xyz, xyz_rec, *([mu, sigma] if mu is not None else []), *([pmu, pstd] if pmu is not None else []))
        comps = out4.detach()
        ctx.mark_non_differentiable(comps)
        return out4.narrow(0, 0, 1).reshape(()), comps

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, _g_comps):
        saved = list(ctx.saved_tensors)
        xyz, xyz_rec = saved[0], saved[1]
        mu = sigma = pmu = pstd = None
        k = 2
        if ctx.has[0]:
            mu, sigma = saved[k], saved[k + 1]
            k += 2
        if ctx.has[1]:
            pmu, pstd = saved[k], saved[k + 1]
        g = g_loss.reshape(1).contiguous()
        g_rec, g_mu, g_sigma, g_pmu, g_pstd = ops.loss_bwd(g, xyz, xyz_rec, ctx.bond_graph, mu, sigma, pmu, pstd, ctx.norms,
                                                           ctx.beta, ctx.gamma)
        g_xyz = ops.loss_bwd_target(g, xyz, xyz_rec, ctx.bond_graph, ctx.norms, ctx.gamma) if ctx.needs_input_grad[4] else None
        return None, None, None, None, g_xyz, g_rec, g_mu, g_sigma, g_pmu, g_pstd


class DihedralLoss(Function):
    """mean_d (theta(xyz_rec; idx_d) - theta(xyz; idx_d))^2, the dihedral term of the PCN loop (scripts/pcn_utils.py:114-132,
    178-180).  Gradient to xyz_rec only (the reference moves the target to the CPU, detached); backward = per-atom gather
    over the CSR of the flattened index list: no atomics."""

    @staticmethod
    def forward(ctx, xyz, xyz_rec, idx, count, norm):
        n_atoms = xyz_rec.shape[0]
        idx = idx.to(torch.int64).contiguous()
        out, contrib = ops.dihedral_loss_fwd(xyz.contiguous(), xyz_rec.contiguous(), idx, count, norm)
        D = idx.shape[0]
        pairs = torch.stack([idx.reshape(-1), torch.arange(4 * D, dtype=torch.int64, device=idx.device)], 1)
        # a padded list's (0, 0, 0, 0) rows stay out of the CSR: they would pile 4 entries per pad row onto atom 0, and rows
        # that long fall back to the slow in-place sort of graph.cu (seconds per step at protein-batch capacities)
        live = None if count is None else (count.reshape(1).to(torch.int64) * 4).clamp_(max=4 * D)
        ctx.graph = ops.build_graph(pairs, n_atoms, n_send=max(4 * D, 1), n_edges_dev=live)
        ctx.n_atoms, ctx.count, ctx.norm = n_atoms, count, norm
        ctx.save_for_backward(contrib)
        return out.reshape(())

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        if ctx.needs_input_grad[0]:
            raise NotImplementedError("coordinate gradients: the gradient of the dihedral loss to its target xyz is not implemented")
        (contrib,) = ctx.saved_tensors
        g_rec = ops.dihedral_loss_bwd(g.reshape(1).contiguous(), contrib, ctx.graph, ctx.n_atoms, ctx.count, ctx.norm)
        return None, g_rec, None, None, None
