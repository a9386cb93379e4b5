"""Model assembly with the reference's class names, constructor signatures, attribute names and
state_dict keys (cgvae.py of the reference): EquiEncoder, CGprior, EquivariantDecoder,
EquivariantPsuedoDecoder, CGequiVAE, PCN.  Every stack runs on planar vectors, computes the edge
geometry once per graph (the reference recomputes it in every layer) and calls one fused message
kernel per layer.
"""
import torch
from torch import nn

from . import functions as fn
from . import ops
from .conv import (ContractiveMessageBlock, EquiMessageBlock, EquiMessageCross, EquiMessagePsuedo, PseudoUpdateBlock,
                   UpdateBlock, _Unplanar, to_module)
from .modules import Dense, DistanceEmbed, make_directed


class BatchGraphs(object):
    """CSR graphs and segment tables of one batch, built once and shared by encoder / prior / decoder
    (the reference re-runs make_directed in each of them: cgvae.py:270-271,378,87,165)."""

    def __init__(self, nbr_count=None, cg_nbr_count=None, nbr_symmetrize=True, cg_nbr_symmetrize=True):
        self.atom = None      # ops.Graph over atoms (directed)
        self.cg = None        # ops.Graph over beads (directed)
        self.seg = None       # ops.Segments (mapping)
        self.contract = None  # ops.Graph atoms -> beads
        self._geom = {}
        # static-shape mode (CUDA-graph replay): nbr_list / CG_nbr_list are one-directional lists padded to a fixed
        # capacity and these int64 device scalars hold the live row counts; the flipped half of make_directed is
        # generated inside the CSR kernels and no host read happens.
        self.counts = {"atom": nbr_count, "cg": cg_nbr_count}
        # make_directed (conv.py:10-20) appends the flipped list only when the list is one-directional; its two
        # ``.any().item()`` reads are taken on the host when the static batch is prepared (train.to_static_batch) and
        # arrive here as plain bools: a bidirectional list (dir_mp=True, or the bond-derived CG graph of
        # cg_cutoff=None) must NOT be doubled.
        self.symmetrize = {"atom": bool(nbr_symmetrize), "cg": bool(cg_nbr_symmetrize)}

    @classmethod
    def for_batch(cls, batch):
        return cls(batch.get('nbr_count'), batch.get('CG_nbr_count'), batch.get('nbr_symmetrize', True),
                   batch.get('CG_nbr_symmetrize', True))

    def directed_graph(self, which, nbr_list, n_nodes, already_directed=False):
        count = self.counts.get(which)
        if count is not None:
            sym = self.symmetrize.get(which, True) and not already_directed
            return ops.build_graph(nbr_list, n_nodes, symmetrize=sym, n_edges_dev=count)
        pairs = nbr_list if already_directed else make_directed(nbr_list)[0]
        return ops.build_graph(pairs, n_nodes)

    def geometry(self, which, xyz_send, xyz_recv, n_rbf, cutoff):
        key = (which, int(n_rbf), float(cutoff))
        if key not in self._geom:
            self._geom[key] = fn.edge_geometry(getattr(self, which), xyz_send, xyz_recv, n_rbf, cutoff)
        return self._geom[key]


def _num_beads(mapping, hint=None):
    if hint is not None:
        return int(hint)
    return int(mapping.max().item()) + 1


def _embed(table_module, idx):
    return fn.EmbeddingLookup.apply(table_module.weight, idx, table_module.padding_idx)


def _mlp(seq, act_code, x):
    return fn.MLP2.apply(act_code, x, seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias)


class EquivariantPsuedoDecoder(nn.Module):
    """cgvae.py:52-125."""

    def __init__(self, n_atom_basis, n_rbf, cutoff, num_conv, activation, breaksym=False):
        nn.Module.__init__(self)
        self.message_blocks = nn.ModuleList(
            [EquiMessagePsuedo(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=0.0)
             for _ in range(num_conv)])
        self.update_blocks = nn.ModuleList(
            [UpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(num_conv)])
        self.pseudo_update_blocks = nn.ModuleList(
            [PseudoUpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(num_conv)])
        self.breaksym = breaksym
        self.n_atom_basis = n_atom_basis
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def forward(self, cg_xyz, CG_nbr_list, mapping, S, graphs=None, planar=False):
        g = graphs if graphs is not None else BatchGraphs()
        if g.cg is None:
            g.cg = g.directed_graph("cg", CG_nbr_list, S.shape[0])
        geom = g.geometry("cg", cg_xyz, cg_xyz, self.n_rbf, self.cutoff)
        n, f = S.shape
        # initial decoder state (cgvae.py:90-95): V = Vbar = 0, Sbar = 1 (breaksym) or 0 -- two fills of our own
        zeros = ops.fill((6 * n * f,), 0.0, S)
        V, Vbar = zeros[:3 * n * f].view(n, 3, f), zeros[3 * n * f:].view(n, 3, f)
        Sbar = ops.fill((n, f), 1.0 if self.breaksym else 0.0, S)
        for i, message_block in enumerate(self.message_blocks):
            S, Sbar, V, Vbar = message_block.fused(S, Sbar, V, Vbar, geom)
            S, V = self.update_blocks[i].fused(S, V)
        return S, (V if planar else _Unplanar.apply(V))


class EquivariantDecoder(nn.Module):
    """cgvae.py:129-191 (``deg_inv_sqrt`` at :171 is computed and never used by the reference)."""

    def __init__(self, n_atom_basis, n_rbf, cutoff, num_conv, activation, cross_flag=True):
        nn.Module.__init__(self)
        block = EquiMessageCross if cross_flag else EquiMessageBlock
        self.message_blocks = nn.ModuleList(
            [block(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=0.0)
             for _ in range(num_conv)])
        self.update_blocks = nn.ModuleList(
            [UpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(num_conv)])
        self.n_atom_basis = n_atom_basis
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def forward(self, cg_xyz, CG_nbr_list, mapping, H, graphs=None, planar=False):
        g = graphs if graphs is not None else BatchGraphs()
        if g.cg is None:
            g.cg = g.directed_graph("cg", CG_nbr_list, H.shape[0])
        geom = g.geometry("cg", cg_xyz, cg_xyz, self.n_rbf, self.cutoff)
        V = None  # zero until the first message layer has run
        for i, message_block in enumerate(self.message_blocks):
            H, V = message_block.fused(H, V, geom)
            H, V = self.update_blocks[i].fused(H, V)
        if V is None:                               # num_conv = 0: the reference returns its zero-initialised vectors
            n, f = H.shape
            V = ops.fill((n, 3, f), 0.0, H)
        return H, (V if planar else _Unplanar.apply(V))


class EquiEncoder(nn.Module):
    """cgvae.py:194-331.  update_blocks / cg_message_blocks / cg_update_blocks / atom2CGcouplings / dist_embed are
    parameters the reference constructs and never calls; they are kept for state_dict compatibility."""

    def __init__(self, n_conv, n_atom_basis, n_rbf, activation, cutoff, dir_mp=False, cg_mp=False):
        super().__init__()
        self.atom_embed = nn.Embedding(100, n_atom_basis, padding_idx=0)
        self.dist_embed = DistanceEmbed(n_rbf=n_rbf, cutoff=cutoff, feat_dim=n_atom_basis, dropout=0.0)
        self.message_blocks = nn.ModuleList(
            [EquiMessageBlock(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=0.0)
             for _ in range(n_conv)])
        self.update_blocks = nn.ModuleList(
            [UpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(n_conv)])
        self.cg_message_blocks = nn.ModuleList(
            [EquiMessageBlock(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=0.0)
             for _ in range(n_conv)])
        self.cg_update_blocks = nn.ModuleList(
            [UpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(n_conv)])
        self.cgmessage_layers = nn.ModuleList(
            [ContractiveMessageBlock(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=20.0, dropout=0.0)
             for _ in range(n_conv)])
        self.atom2CGcouplings = nn.ModuleList(
            [nn.Sequential(Dense(in_features=n_atom_basis, out_features=n_atom_basis, bias=True,
                                 activation=to_module(activation)),
                           Dense(in_features=n_atom_basis, out_features=n_atom_basis, bias=True))
             for _ in range(n_conv)])
        self.n_conv = n_conv
        self.dir_mp = dir_mp
        self.cg_mp = cg_mp
        self.n_atom_basis = n_atom_basis
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def forward(self, z, xyz, cg_xyz, mapping, nbr_list, cg_nbr_list, graphs=None, num_beads=None):
        g = graphs if graphs is not None else BatchGraphs()
        if g.atom is None:
            g.atom = g.directed_graph("atom", nbr_list, xyz.shape[0], already_directed=self.dir_mp)
        if g.seg is None:
            g.seg = ops.build_segments(mapping, _num_beads(mapping, num_beads))
        if g.contract is None:
            g.contract = ops.contraction_graph(g.seg)
        geom_atom = g.geometry("atom", xyz, xyz, self.n_rbf, self.cutoff)
        geom_con = g.geometry("contract", xyz, cg_xyz, self.n_rbf, 20.0)    # cutoff fixed at 20.0: cgvae.py:249

        h = _embed(self.atom_embed, z)
        v = None
        H = V = None
        for i in range(self.n_conv):
            h, v = self.message_blocks[i].fused(h, v, geom_atom)
            if i == 0:                                                       # cgvae.py:296-298
                H = fn.SegmentReduce.apply(g.seg, True, h)
                V = fn.SegmentReduce.apply(g.seg, True, v)
            H, V = self.cgmessage_layers[i].fused(h, v, H, V, geom_con)
        return H, h


class CGprior(nn.Module):
    """cgvae.py:334-403."""

    def __init__(self, n_conv, n_atom_basis, n_rbf, activation, cutoff, dir_mp=False):
        super().__init__()
        self.atom_embed = nn.Embedding(100, n_atom_basis, padding_idx=0)
        self.dist_embed = DistanceEmbed(n_rbf=n_rbf, cutoff=cutoff, feat_dim=n_atom_basis, dropout=0.0)
        self.message_blocks = nn.ModuleList(
            [EquiMessageBlock(feat_dim=n_atom_basis, activation=activation, n_rbf=n_rbf, cutoff=cutoff, dropout=0.0)
             for _ in range(n_conv)])
        self.update_blocks = nn.ModuleList(
            [UpdateBlock(feat_dim=n_atom_basis, activation=activation, dropout=0.0) for _ in range(n_conv)])
        self.mu = nn.Sequential(nn.Linear(n_atom_basis, n_atom_basis), nn.Tanh(), nn.Linear(n_atom_basis, n_atom_basis))
        self.sigma = nn.Sequential(nn.Linear(n_atom_basis, n_atom_basis), nn.Tanh(), nn.Linear(n_atom_basis, n_atom_basis))
        self.n_conv = n_conv
        self.dir_mp = dir_mp
        self.n_rbf, self.cutoff = n_rbf, cutoff

    def forward(self, cg_z, cg_xyz, cg_nbr_list, graphs=None):
        g = graphs if graphs is not None else BatchGraphs()
        if g.cg is None:
            g.cg = g.directed_graph("cg", cg_nbr_list, cg_xyz.shape[0])
        geom = g.geometry("cg", cg_xyz, cg_xyz, self.n_rbf, self.cutoff)
        h = _embed(self.atom_embed, cg_z)
        v = None
        for i in range(self.n_conv):
            h, v = self.message_blocks[i].fused(h, v, geom)
        H_mu = _mlp(self.mu, 3, h)
        H_sigma = _mlp(self.sigma, 3, h)
        H_std = fn.StdLogvar.apply(H_sigma, 1e-9)
        return H_mu, H_std


def _act_code_of(module):
    from .modules import module_activation_code
    return module_activation_code(module)


class CGequiVAE(nn.Module):
    """cgvae.py:406-513."""

    def __init__(self, encoder, equivaraintconv, atom_munet, atom_sigmanet, n_cgs, feature_dim, prior_net=None,
                 det=False, equivariant=True, offset=True):
        nn.Module.__init__(self)
        self.encoder = encoder
        self.equivaraintconv = equivaraintconv
        self.atom_munet = atom_munet
        self.atom_sigmanet = atom_sigmanet
        self.n_cgs = n_cgs
        self.prior_net = prior_net
        self.det = det
        self.offset = offset
        self.equivariant = equivariant
        if equivariant is False:
            self.euclidean = nn.Linear(self.encoder.n_atom_basis, self.encoder.n_atom_basis * 3)

    def get_inputs(self, batch):
        xyz = batch['nxyz'][:, 1:]
        cg_xyz = batch['CG_nxyz'][:, 1:]
        cg_z = batch['CG_nxyz'][:, 0]
        z = batch['nxyz'][:, 0]
        mapping = batch['CG_mapping']
        nbr_list = batch['nbr_list']
        CG_nbr_list = batch['CG_nbr_list']
        num_CGs = batch['num_CGs']
        return z, cg_z, xyz, cg_xyz, nbr_list, CG_nbr_list, mapping, num_CGs

    def reparametrize(self, mu, sigma, eps=None):
        if eps is None:
            eps = torch.randn_like(sigma)
        return eps.mul(sigma).add_(mu)

    def CG2ChannelIdx(self, CG_mapping):
        """rank of each atom inside its bead (cgvae.py:451-460), computed on the device, exact."""
        n_beads = int(CG_mapping.max().item()) + 1 if CG_mapping.numel() else 0
        return ops.build_segments(CG_mapping, n_beads).rank

    def decoder(self, cg_xyz, CG_nbr_list, S_I, s_i, mapping, num_CGs, graphs=None):
        g = graphs if graphs is not None else BatchGraphs()
        if g.seg is None:
            g.seg = ops.build_segments(mapping, cg_xyz.shape[0])
        cg_s, cg_v = self.equivaraintconv(cg_xyz, CG_nbr_list, mapping, S_I, graphs=g, planar=True)
        if self.equivariant is False:
            # cgvae.py:469-471: dv = euclidean(cg_s).reshape(Nc, F, 3) replaces the equivariant vectors; [Nc,F,3] -> planar
            from .conv import _Planar
            n_b, F = cg_s.shape
            cg_v = _Planar.apply(fn.LinearFn.apply(cg_s, self.euclidean.weight, self.euclidean.bias).view(n_b, F, 3))
        return fn.Lift.apply(g.seg, 1 if self.offset else 0, None, cg_v, cg_xyz.contiguous())

    def forward(self, batch, eps=None):
        atomic_nums, cg_z, xyz, cg_xyz, nbr_list, CG_nbr_list, mapping, num_CGs = self.get_inputs(batch)
        xyz, cg_xyz = xyz.contiguous(), cg_xyz.contiguous()
        g = batch.get('_graphs') or BatchGraphs.for_batch(batch)
        S_I, s_i = self.encoder(atomic_nums, xyz, cg_xyz, mapping, nbr_list, CG_nbr_list, graphs=g,
                                num_beads=cg_xyz.shape[0])
        if self.prior_net:
            H_prior_mu, H_prior_sigma = self.prior_net(cg_z, cg_xyz, CG_nbr_list, graphs=g)
        else:
            H_prior_mu, H_prior_sigma = None, None
        z = S_I
        mu = _mlp(self.atom_munet, _act_code_of(self.atom_munet[1]), z)
        logvar = _mlp(self.atom_sigmanet, _act_code_of(self.atom_sigmanet[1]), z)
        if self.det:
            sigma, z_sample = fn.StdLogvar.apply(logvar, 1e-12), z
        else:
            # sigma = 1e-12 + exp(logvar / 2) and z = eps * sigma + mu in one launch (cgvae.py:445-449,500-507)
            if eps is None:
                eps = torch.randn_like(logvar)
            z_sample, sigma = fn.VAELatent.apply(mu, logvar, eps)
        hook = getattr(self, "_latent_grad_hook", None)
        if hook is not None and z_sample.requires_grad:
            # fires when the backward pass has left the decoder (train.TrainStep: data-parallel overlap)
            z_sample.register_hook(hook)
        xyz_recon = self.decoder(cg_xyz, CG_nbr_list, z_sample, s_i, mapping, num_CGs, graphs=g)
        ops.check_device_errors(xyz_recon.device)      # IndexError where the reference raises one (cgvae.py:473)
        return mu, sigma, H_prior_mu, H_prior_sigma, xyz, xyz_recon


class PCN(nn.Module):
    """Protein completion network, cgvae.py:516-594."""

    def __init__(self, equivaraintconv, feature_dim, offset=True):
        nn.Module.__init__(self)
        self.equivaraintconv = equivaraintconv
        self.offset = offset
        self.embedding = nn.Embedding(100, feature_dim, padding_idx=0)

    def get_inputs(self, batch):
        xyz = batch['xyz']
        cg_xyz = batch['ca_xyz']
        cg_z = batch['res']
        mapping = batch['cg_map']
        nbr_list = batch['bond_edge_list']
        CG_nbr_list = batch['CG_nbr_list']
        num_CGs = [len(seq) for seq in batch['seq']] if 'seq' in batch else None     # unused by the decoder
        return cg_z, xyz, cg_xyz, nbr_list, CG_nbr_list, mapping, num_CGs

    def CG2ChannelIdx(self, CG_mapping):
        n_beads = int(CG_mapping.max().item()) + 1 if CG_mapping.numel() else 0
        return ops.build_segments(CG_mapping, n_beads).rank

    def decoder(self, cg_xyz, CG_nbr_list, S_I, ca_idx, mapping, num_CGs, graphs=None, ca_count=None):
        g = graphs if graphs is not None else BatchGraphs()
        if g.seg is None:
            g.seg = ops.build_segments(mapping, cg_xyz.shape[0])
        cg_s, cg_v = self.equivaraintconv(cg_xyz, CG_nbr_list, mapping, S_I, graphs=g, planar=True)
        n_atoms = mapping.shape[0]
        pin = None
        # cgvae.py:569-571: C-alpha atoms are pinned to their bead unless the index list overruns the atoms.  The
        # predicate (ca_idx[-1] < n_atoms) is evaluated on the device: an all-zero mask == no re-anchoring, and no host
        # read stands between the step and a CUDA-graph capture.  ca_count: live entries of a zero-padded static list.
        if ca_idx.numel():
            pin = ops.pin_mask(ca_idx, n_atoms, ca_count)
        return fn.Lift.apply(g.seg, 2 if pin is not None else 0, pin, cg_v, cg_xyz.contiguous())

    def forward(self, batch):
        cg_z, xyz, cg_xyz, nbr_list, CG_nbr_list, mapping, num_CGs = self.get_inputs(batch)
        S_I = _embed(self.embedding, cg_z)
        xyz_recon = self.decoder(cg_xyz.contiguous(), CG_nbr_list, S_I, batch['ca_idx'], mapping, num_CGs,
                                 graphs=batch.get('_graphs') or BatchGraphs(None, batch.get('CG_nbr_count'), True,
                                                                            batch.get('CG_nbr_symmetrize', True)),
                                 ca_count=batch.get('ca_count'))
        ops.check_device_errors(xyz_recon.device)
        return None, None, None, None, xyz, xyz_recon
