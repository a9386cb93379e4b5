"""Equivariant message / update / contraction blocks with the reference's class names, constructor
signatures, forward signatures and state_dict keys (conv.py of the reference), running on the
sm_100a kernels.

Two call levels:
  * ``forward(...)``  -- the reference block API: vectors in the reference layout [N,F,3], explicit
    ``r_ij`` / ``nbrs``, returns DELTAS (conv.py:505-563 etc.).  Builds the CSR + edge geometry per call.
  * ``fused(...)``    -- what the stacks in cgvae.py use: planar vectors [N,3,F], a prepared
    ``ops.Geometry``, residual add fused into the kernel, v=None meaning "still zero".
"""
import torch
from torch import nn

from . import functions as fn
from . import ops
from .modules import Dense, DistanceEmbed, Swish, shifted_softplus, activation_code, make_directed  # noqa: F401 (re-export)


def to_module(activation):
    """marker module of the reference's layer_types registry (modules.py:32-42)"""
    activation_code(activation)                 # raises for unknown names
    if activation == "swish":
        return Swish()
    if activation == "shifted_softplus":
        return shifted_softplus()
    if activation == "sigmoid":
        return nn.Sigmoid()
    if activation == "linear":
        return nn.Identity()
    return getattr(nn, activation)()


def _geometry_from_edges(nbrs, r_ij, n_nodes, n_rbf, cutoff, edge_wgt=None):
    graph = ops.build_graph(nbrs, n_nodes)
    return fn.edge_geometry(graph, None, None, n_rbf, cutoff, edge_wgt=edge_wgt, r_edge=r_ij)


class InvariantMessage(nn.Module):
    """phi-MLP + distance filter parameters (conv.py:31-75).  ``dist_filter`` / ``offset`` are unused by the
    reference forward and kept only for state_dict compatibility."""

    def __init__(self, in_feat_dim, out_feat_dim, activation, n_rbf, cutoff, dropout):
        super().__init__()
        self.inv_dense = nn.Sequential(
            Dense(in_features=in_feat_dim, out_features=in_feat_dim, bias=True, dropout_rate=dropout,
                  activation=to_module(activation)),
            Dense(in_features=in_feat_dim, out_features=out_feat_dim, bias=True, dropout_rate=dropout))
        self.dist_embed = DistanceEmbed(n_rbf=n_rbf, cutoff=cutoff, feat_dim=out_feat_dim, dropout=dropout)
        self.dist_filter = Dense(in_features=in_feat_dim, out_features=out_feat_dim, bias=True, dropout_rate=0.0)
        self.offset = torch.linspace(0.0, cutoff, in_feat_dim)
        self.act = activation_code(activation)
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def params(self):
        d0, d1 = self.inv_dense[0], self.inv_dense[1]
        return (d0.weight, d0.bias, d1.weight, d1.bias, self.dist_embed.filter_weight, self.dist_embed.filter_bias)


class _MessageBase(nn.Module):
    n_split = 3

    def _build(self, feat_dim, activation, n_rbf, cutoff, dropout):
        self.inv_message = InvariantMessage(in_feat_dim=feat_dim, out_feat_dim=feat_dim * self.n_split,
                                            activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=dropout)
        self.feat_dim = feat_dim

    def fused(self, s, v, geom):
        """(s, v) + message, planar layout; v may be None (all zero)."""
        return fn.MessageBlock.apply(geom, self.n_split, "self", self.inv_message.act, s, v, None, None,
                                     *self.inv_message.params(), geom.basis, geom.unit)

    def forward(self, s_j, v_j, r_ij, nbrs, edge_wgt=None):
        geom = _geometry_from_edges(nbrs, r_ij, s_j.shape[0], self.inv_message.n_rbf, self.inv_message.cutoff, edge_wgt)
        # the layout conversions [N,F,3] <-> [N,3,F] are autograd nodes of their own
        ds, dv = fn.MessageBlock.apply(geom, self.n_split, "delta", self.inv_message.act, s_j, _Planar.apply(v_j), None, None,
                                       *self.inv_message.params(), geom.basis, geom.unit)
        return ds, _Unplanar.apply(dv)


class _Planar(torch.autograd.Function):
    """[N,F,3] -> [N,3,F] with its transpose as backward."""

    @staticmethod
    def forward(ctx, v):
        return ops.vec_to_planar(v)

    @staticmethod
    def backward(ctx, g):
        return ops.vec_from_planar(g.contiguous())


class _Unplanar(torch.autograd.Function):
    @staticmethod
    def forward(ctx, v):
        return ops.vec_from_planar(v)

    @staticmethod
    def backward(ctx, g):
        return ops.vec_to_planar(g.contiguous())


class EquiMessageBlock(_MessageBase):
    """conv.py:487-563.  ``h_att`` / ``v_att`` exist only as (unused) parameters, as in the reference."""
    n_split = 3

    def __init__(self, feat_dim, activation, n_rbf, cutoff, dropout):
        super().__init__()
        self._build(feat_dim, activation, n_rbf, cutoff, dropout)
        self.h_att = nn.Sequential(nn.Linear(feat_dim, feat_dim), nn.ReLU(), nn.Linear(feat_dim, feat_dim))
        self.v_att = nn.Sequential(nn.Linear(feat_dim, feat_dim), nn.ReLU(), nn.Linear(feat_dim, feat_dim))


class EquiMessageCross(_MessageBase):
    """conv.py:343-402: adds the m3 * (v_i x v_j) term."""
    n_split = 4

    def __init__(self, feat_dim, activation, n_rbf, cutoff, dropout):
        super().__init__()
        self._build(feat_dim, activation, n_rbf, cutoff, dropout)


class EquiMessagePsuedo(nn.Module):
    """conv.py:165-242: 9 filter splits over (s, sbar, v, vbar)."""

    def __init__(self, feat_dim, activation, n_rbf, cutoff, dropout):
        super().__init__()
        self.inv_message = InvariantMessage(in_feat_dim=feat_dim, out_feat_dim=feat_dim * 9, activation=activation,
                                            n_rbf=n_rbf, cutoff=cutoff, dropout=dropout)

    def fused(self, s, sbar, v, vbar, geom):
        return fn.Message9Block.apply(geom, True, self.inv_message.act, s, sbar, v, vbar, *self.inv_message.params(),
                                      geom.basis, geom.unit)

    def forward(self, s_j, sbar_j, v_j, vbar_j, r_ij, nbrs, edge_wgt=None):
        # edge_wgt is accepted and ignored, exactly like the reference (conv.py:180-187 never reads it)
        geom = _geometry_from_edges(nbrs, r_ij, s_j.shape[0], self.inv_message.n_rbf, self.inv_message.cutoff)
        ds, dsbar, dv, dvbar = fn.Message9Block.apply(geom, False, self.inv_message.act, s_j, sbar_j, _Planar.apply(v_j), _Planar.apply(vbar_j),
                                                      *self.inv_message.params(), geom.basis, geom.unit)
        return ds, dsbar, _Unplanar.apply(dv), _Unplanar.apply(dvbar)


class UpdateBlock(nn.Module):
    """conv.py:566-616."""

    def __init__(self, feat_dim, activation, dropout):
        super().__init__()
        self.u_mat = Dense(in_features=feat_dim, out_features=feat_dim, bias=False)
        self.v_mat = Dense(in_features=feat_dim, out_features=feat_dim, bias=False)
        self.s_dense = nn.Sequential(
            Dense(in_features=2 * feat_dim, out_features=feat_dim, bias=True, dropout_rate=dropout,
                  activation=to_module(activation)),
            Dense(in_features=feat_dim, out_features=3 * feat_dim, bias=True, dropout_rate=dropout))
        self.act = activation_code(activation)

    def params(self):
        return (self.u_mat.weight, self.v_mat.weight, self.s_dense[0].weight, self.s_dense[0].bias,
                self.s_dense[1].weight, self.s_dense[1].bias)

    def fused(self, s, v):
        return fn.UpdateBlockFn.apply(True, self.act, s, v, *self.params())

    def forward(self, s_i, v_i):
        ds, dv = fn.UpdateBlockFn.apply(False, self.act, s_i, _Planar.apply(v_i), *self.params())
        return ds, _Unplanar.apply(dv)


class PseudoUpdateBlock(nn.Module):
    """conv.py:619-672: constructed by EquivariantPsuedoDecoder but never called (cgvae.py:115-119); parameters
    only, for state_dict compatibility."""

    def __init__(self, feat_dim, activation, dropout):
        super().__init__()
        self.u_mat = Dense(in_features=feat_dim, out_features=feat_dim, bias=False)
        self.v_mat = Dense(in_features=feat_dim, out_features=feat_dim, bias=False)
        self.s_dense = nn.Sequential(
            Dense(in_features=2 * feat_dim, out_features=feat_dim, bias=True, dropout_rate=dropout,
                  activation=to_module(activation)),
            Dense(in_features=feat_dim, out_features=3 * feat_dim, bias=True, dropout_rate=dropout))

    def forward(self, s_i, v_i):
        raise NotImplementedError("PseudoUpdateBlock.forward is dead code in the reference (never called)")


class ContractiveMessageBlock(nn.Module):
    """conv.py:677-733: atoms -> beads message with its own phi-MLP / filter (cutoff 20.0 at the call site)."""

    def __init__(self, feat_dim, activation, n_rbf, cutoff, dropout):
        super().__init__()
        self.inv_dense = nn.Sequential(
            Dense(in_features=feat_dim, out_features=feat_dim, bias=True, dropout_rate=dropout,
                  activation=to_module(activation)),
            Dense(in_features=feat_dim, out_features=3 * feat_dim, bias=True, dropout_rate=dropout))
        self.dist_embed = DistanceEmbed(n_rbf=n_rbf, cutoff=cutoff, feat_dim=3 * feat_dim, dropout=dropout)
        self.act = activation_code(activation)
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def params(self):
        d0, d1 = self.inv_dense[0], self.inv_dense[1]
        return (d0.weight, d0.bias, d1.weight, d1.bias, self.dist_embed.filter_weight, self.dist_embed.filter_bias)

    def fused(self, s, v, H, V, geom):
        """(H, V) + contraction of atom state (s, v) over the atoms->beads graph."""
        return fn.MessageBlock.apply(geom, 3, "other", self.act, s, v, H, V, *self.params(), geom.basis, geom.unit)

    def forward(self, s_i, v_i, r_iI, mapping):
        # scatter_add without dim_size (conv.py:725-731): the output has max(mapping)+1 rows -- one host read,
        # as in torch_scatter
        n_beads = int(mapping.max().item()) + 1
        seg = ops.build_segments(mapping, n_beads)
        graph = ops.contraction_graph(seg)
        geom = fn.edge_geometry(graph, None, None, self.n_rbf, self.cutoff, r_edge=r_iI)
        dS, dV = fn.MessageBlock.apply(geom, 3, "delta", self.act, s_i, _Planar.apply(v_i), None, None, *self.params(),
                                       geom.basis, geom.unit)
        return dS, _Unplanar.apply(dV)
