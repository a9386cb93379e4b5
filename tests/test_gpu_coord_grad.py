"""GPU (B200): gradients to atom / bead coordinates and to the r_ij / r_iI of the block API through the sm_100a kernels
(csrc/message_geom.cu, the geometry backward and node reduction of csrc/geom.cu, loss_bwd_target in csrc/loss.cu).

  * parity with the float64 oracle (tests/coord_cases.check, fp32 rule: per tensor within max(1e-5, 10 x the fp32
    oracle's own error), all coordinate gradients together within 1e-5 relative L2), small goldens and config-sized
    batches;
  * properties at full size: translation invariance, rotation equivariance, bitwise repeatability;
  * nothing else changes: outputs and parameter gradients are bitwise those of a run without coordinate gradients;
  * which kernels ran (torch.profiler), padded static-capacity graphs, the cases that raise."""
import numpy as np
import pytest
import torch

import coarsegrainingvae_b200 as cg
from coarsegrainingvae_b200 import functions as fn, ops, synthetic
from tests import coord_cases as cc, parity_cases as pc
from tests.test_gpu_dense_paths import _probe

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
GEOM_KERNELS = {"message_geom_bwd_kernel", "edge_geometry_bwd_kernel", "edge_coord_reduce_kernel"}


def _gpu_radius(xyz, cutoff):
    return ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=DEV), cutoff).cpu().numpy()


def _to(batch, dev, dtype=None):
    out = {}
    for k, v in batch.items():
        if torch.is_tensor(v):
            v = v.to(dtype) if (dtype is not None and v.dtype.is_floating_point) else v
            v = v.to(dev)
        out[k] = v
    return out


# ------------------------------------------------------------------------------------------ parity with float64

@pytest.mark.parametrize("tag", ["k3", "k4", "k9", "k3w"])
def test_block_api_r_ij(tag):
    print(tag, cc.check(*cc.block_r(DEV, tag, torch.float32), TOL, fp32_rule=True))


def test_contraction_r_iI():
    print(cc.check(*cc.contraction_r(DEV, torch.float32), TOL, fp32_rule=True))


@pytest.mark.parametrize("tag", ["vae_sym", "vae_noneq"])
def test_cgvae_loss_coordinates(tag):
    """through train.training_loss (functions.TrainingLoss: the target-coordinate gradient kernel)"""
    print(tag, cc.check(*cc.cgvae_coords(DEV, tag, torch.float32, fused_loss=True), TOL, fp32_rule=True))


@pytest.mark.parametrize("tag,ca_pin", [("pcn_cross", True), ("pcn_plain", True), ("pcn_cross", False)])
def test_pcn_ca_xyz(tag, ca_pin):
    print(tag, ca_pin, cc.check(*cc.pcn_coords(DEV, tag, torch.float32, ca_pin), TOL, fp32_rule=True))


def _c2_setup():
    cfg = dict(synthetic.CONFIGS["c2_chignolin"])
    n_conf = cfg["batch"] = 2
    batch = synthetic.cgvae_batch(cfg, 0, _gpu_radius, cg.CG_collate)
    torch.manual_seed(123)
    model = pc.build_vae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"],
                         cfg["cg_cutoff"], cfg["n_cgs"] == 3, cfg["n_cgs"]).to(DEV)
    eps = torch.randn(n_conf * cfg["n_cgs"], cfg["n_basis"], generator=torch.Generator().manual_seed(7))
    spec = dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], enc_nconv=cfg["enc_nconv"], dec_nconv=cfg["dec_nconv"],
                atom_cutoff=cfg["atom_cutoff"], cg_cutoff=cfg["cg_cutoff"], decoder="pseudo", breaksym=cfg["n_cgs"] == 3,
                activation="swish")
    return cfg, batch, model, eps, spec


def _c2_run(cfg, batch, model, eps, coords):
    from coarsegrainingvae_b200 import train
    model.zero_grad(set_to_none=True)
    b = _to(batch, DEV)
    if coords:
        b["nxyz"], b["CG_nxyz"] = b["nxyz"].clone().requires_grad_(), b["CG_nxyz"].clone().requires_grad_()
    out = model(b, eps=eps.to(DEV))
    loss = train.training_loss(out, out[4], b["bond_edge_list"], cfg["beta"], cfg["gamma"])[0]
    loss.backward()
    grads = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    return out, grads, ((b["nxyz"].grad, b["CG_nxyz"].grad) if coords else None)


def test_c2_chignolin_full_width():
    """c2 (F = 600, 2 x 175 atoms, 9-split decoder): d loss / d nxyz, d CG_nxyz vs the float64 oracle"""
    from oracle import cgvae_oracle as orc
    cfg, batch, model, eps, spec = _c2_setup()
    _, _, (gx, gc) = _c2_run(cfg, batch, model, eps, True)

    def oracle(dt):
        P = {k: v.detach().cpu().to(dt) for k, v in model.state_dict().items()}
        b = _to(batch, "cpu", dt)
        b["nxyz"], b["CG_nxyz"] = b["nxyz"].clone().requires_grad_(), b["CG_nxyz"].clone().requires_grad_()
        orc.training_loss(orc.cgvae_forward(P, spec, b, eps=eps.to(dt)), b, cfg["beta"], cfg["gamma"])[0].backward()
        return {"nxyz": b["nxyz"].grad, "CG_nxyz": b["CG_nxyz"].grad}

    print(cc.check({"nxyz": gx, "CG_nxyz": gc}, oracle, TOL, fp32_rule=True))


def _pcn_reduced():
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    cfg["n_res"] = 60
    batch = synthetic.pcn_batch(cfg, 0, _gpu_radius, n_proteins=2)
    torch.manual_seed(123)
    net = cg.EquivariantDecoder(n_atom_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], cutoff=cfg["cg_cutoff"],
                                num_conv=cfg["dec_nconv"], activation="swish", cross_flag=True)
    model = cg.PCN(net, feature_dim=cfg["n_basis"], offset=False).to(DEV)
    spec = dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], dec_nconv=cfg["dec_nconv"], atom_cutoff=cfg["cg_cutoff"],
                decoder="cross", activation="swish")
    return cfg, batch, model, spec


def _pcn_run(model, batch, coords):
    model.zero_grad(set_to_none=True)
    b = _to(batch, DEV)
    if coords:
        b["ca_xyz"], b["xyz"] = b["ca_xyz"].clone().requires_grad_(), b["xyz"].clone().requires_grad_()
    out = model(b)
    (out[5] - out[4]).pow(2).mean().backward()
    grads = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    return out, grads, ((b["xyz"].grad, b["ca_xyz"].grad) if coords else None)


def test_pcn_reduced_protein_batch():
    """the batch of test_gpu_parity.test_pcn_step_reduced_protein_batch (F = 512, 9 cross layers, 2 x 60 residues)"""
    from oracle import cgvae_oracle as orc
    cfg, batch, model, spec = _pcn_reduced()
    _, _, (gx, gc) = _pcn_run(model, batch, True)

    def oracle(dt):
        P = {k: v.detach().cpu().to(dt) for k, v in model.state_dict().items()}
        b = _to(batch, "cpu", dt)
        b["ca_xyz"], b["xyz"] = b["ca_xyz"].clone().requires_grad_(), b["xyz"].clone().requires_grad_()
        o = orc.pcn_forward(P, spec, b)
        (o[5] - o[4]).pow(2).mean().backward()
        return {"xyz": b["xyz"].grad, "ca_xyz": b["ca_xyz"].grad}

    print(cc.check({"xyz": gx, "ca_xyz": gc}, oracle, TOL, fp32_rule=True))


# ------------------------------------------------------------------------------------------ nothing else changes

def test_outputs_and_parameter_gradients_unchanged():
    cfg, batch, model, eps, _ = _c2_setup()
    o0, g0, _ = _c2_run(cfg, batch, model, eps, False)
    o1, g1, _ = _c2_run(cfg, batch, model, eps, True)
    for a, b in zip(o0, o1):
        assert (a is None and b is None) or torch.equal(a, b)
    assert g0.keys() == g1.keys() and all(torch.equal(g0[k], g1[k]) for k in g0)
    _, batch, model, _ = _pcn_reduced()
    o0, g0, _ = _pcn_run(model, batch, False)
    o1, g1, _ = _pcn_run(model, batch, True)
    assert torch.equal(o0[5], o1[5])
    assert g0.keys() == g1.keys() and all(torch.equal(g0[k], g1[k]) for k in g0)


# ------------------------------------------------------------------------------------------ properties at full size

def _rotation():
    return torch.as_tensor(synthetic.random_rotation(np.random.default_rng(5)), dtype=torch.float32, device=DEV)


def _layer_20k(graph, xyz, v, Q=None):
    """one EquiMessageBlock (F = 128, R = 7) on the 6 A graph of 20 000 atoms; loss = <out_s, gs> + <out_v, gv>"""
    torch.manual_seed(11)
    blk = cg.EquiMessageBlock(feat_dim=128, activation="swish", n_rbf=7, cutoff=6.0, dropout=0.0).to(DEV)
    x = xyz.clone().requires_grad_()
    geom = fn.edge_geometry(graph, x, x, 7, 6.0)
    s = torch.randn(xyz.shape[0], 128, generator=torch.Generator().manual_seed(3)).to(DEV)
    gs = torch.randn(xyz.shape[0], 128, generator=torch.Generator().manual_seed(4)).to(DEV)
    gv = torch.randn(xyz.shape[0], 3, 128, generator=torch.Generator().manual_seed(6)).to(DEV)
    if Q is not None:
        gv = torch.einsum("ab,nbf->naf", Q, gv)
    out_s, out_v = blk.fused(s, v.contiguous(), geom)           # the fused API reads planar v as a contiguous array
    ((out_s * gs).sum() + (out_v * gv).sum()).backward()
    return x.grad, graph.n_edges


def test_layer_20k_atoms_properties():
    xyz = torch.as_tensor(synthetic.lattice_points(20000, 2.2, np.random.default_rng(1)), dtype=torch.float32, device=DEV)
    v = torch.randn(20000, 3, 128, generator=torch.Generator().manual_seed(2)).to(DEV)
    graph = ops.build_graph(ops.radius_graph(xyz, 6.0, undirected=False), xyz.shape[0])     # kept for the rotated inputs
    g, n_edges = _layer_20k(graph, xyz, v)
    assert n_edges > 1_000_000
    g2, _ = _layer_20k(graph, xyz, v)
    assert torch.equal(g, g2)                                        # bitwise repeatable
    scale = float(g.abs().max())
    assert float(g.double().sum(0).abs().max()) < 1e-4 * scale * g.shape[0] ** 0.5      # translation invariance
    Q = _rotation()
    gr, _ = _layer_20k(graph, xyz @ Q.t(), torch.einsum("ab,nbf->naf", Q, v), Q)
    assert float((gr - g @ Q.t()).abs().max()) < 1e-4 * scale       # rotating the inputs rotates the gradient


def _pcn_full(rot=None):
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    batch = synthetic.pcn_batch(cfg, 0, _gpu_radius, n_proteins=cfg["batch"])
    torch.manual_seed(123)
    from coarsegrainingvae_b200.factory import build_pcn
    model = build_pcn(cfg["n_basis"], cfg["n_rbf"], cfg["cg_cutoff"], cfg["dec_nconv"]).to(DEV)
    b = _to(batch, DEV)
    if rot is not None:
        b["xyz"], b["ca_xyz"] = b["xyz"] @ rot.t(), b["ca_xyz"] @ rot.t()
    b["ca_xyz"], b["xyz"] = b["ca_xyz"].clone().requires_grad_(), b["xyz"].clone().requires_grad_()
    out = model(b)
    (out[5] - out[4]).pow(2).mean().backward()
    return b["xyz"].grad, b["ca_xyz"].grad


def test_pcn_c4_full_batch_properties():
    """c4 PCN, 64 proteins x ~2 000 atoms: translation invariance of xyz + ca_xyz gradients, rotation, repeatability"""
    gx, gc = _pcn_full()
    gx2, gc2 = _pcn_full()
    assert torch.equal(gx, gx2) and torch.equal(gc, gc2)
    scale = max(float(gx.abs().max()), float(gc.abs().max()))
    total = gx.double().sum(0) + gc.double().sum(0)
    assert float(total.abs().max()) < 1e-4 * scale * (gx.shape[0] + gc.shape[0]) ** 0.5
    Q = _rotation()
    rx, rc = _pcn_full(Q)
    assert float((rc - gc @ Q.t()).abs().max()) < 1e-3 * scale
    assert float((rx - gx @ Q.t()).abs().max()) < 1e-3 * scale


# ------------------------------------------------------------------------------------------ which kernels ran

def test_geometry_kernels_run_only_for_coordinate_gradients():
    cfg, batch, model, eps, _ = _c2_setup()
    _, launched = _probe(lambda: _c2_run(cfg, batch, model, eps, True))
    names = {k for k, _, _ in launched}
    assert GEOM_KERNELS <= names, names
    from coarsegrainingvae_b200.train import TrainStep
    trainer = TrainStep(model, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01)
    b = _to(batch, DEV)
    trainer.prepare(b, eps.to(DEV))
    try:
        trainer.step(b, eps.to(DEV))
        _, launched = _probe(lambda: trainer.step(b, eps.to(DEV)))
    finally:
        trainer.flat.release()                       # unregisters the gradient sink (ops.GRAD_SINK) for later tests
    names = {k for k, _, _ in launched}
    assert names and not (names & (GEOM_KERNELS | {"loss_bwd_target_kernel"})), names


# ------------------------------------------------------------------------------------------ edge cases

def test_static_capacity_tail_gives_zero():
    """a padded static-capacity graph gives the gradient of the unpadded one, bitwise"""
    xyz = torch.as_tensor(synthetic.lattice_points(300, 2.2, np.random.default_rng(9)), dtype=torch.float32, device=DEV)
    pairs = ops.radius_graph(xyz, 3.0)         # mean degree below the tensor-core forward's threshold: SIMT path
    E = pairs.shape[0]
    padded = torch.zeros((E + 77, 2), dtype=torch.int64, device=DEV)
    padded[:E] = pairs
    count = torch.tensor([E], dtype=torch.int64, device=DEV)
    torch.manual_seed(2)
    blk = cg.EquiMessageBlock(feat_dim=64, activation="swish", n_rbf=7, cutoff=3.0, dropout=0.0).to(DEV)
    s = torch.randn(300, 64, generator=torch.Generator().manual_seed(3)).to(DEV)

    def run(graph):
        x = xyz.clone().requires_grad_()
        geom = fn.edge_geometry(graph, x, x, 7, 3.0)
        h, v = blk.fused(s, None, geom)
        h, v = blk.fused(h, v, geom)
        (h.pow(2).sum() + v.pow(2).sum()).backward()
        return x.grad

    g_plain = run(ops.build_graph(pairs, 300, symmetrize=True))
    g_pad = run(ops.build_graph(padded, 300, symmetrize=True, n_edges_dev=count))
    assert float(g_plain.abs().max()) > 0 and torch.equal(g_plain, g_pad)


def test_unsupported_cases_raise():
    z = pc.load("blocks_small.npz")
    sec = pc.section(z, "k3w")
    blk = cg.EquiMessageBlock(feat_dim=int(z["meta/F"]), activation="swish", n_rbf=int(z["meta/R"]),
                              cutoff=float(z["meta/cutoff"]), dropout=0.0).to(DEV)
    r = torch.from_numpy(z["in/r"]).to(DEV)
    nbrs = torch.from_numpy(z["in/nbrs"]).to(DEV)
    w = sec["w"].to(DEV).requires_grad_()
    ds, dv = blk(sec["s"].to(DEV), sec["v"].to(DEV), r, nbrs, edge_wgt=w)
    with pytest.raises(NotImplementedError, match="edge_wgt"):
        (ds.sum() + dv.sum()).backward()
    # the dihedral loss's target
    xyz = torch.randn(8, 3, device=DEV, requires_grad=True)
    rec = torch.randn(8, 3, device=DEV, requires_grad=True)
    idx = torch.tensor([[0, 1, 2, 3], [4, 5, 6, 7]], device=DEV)
    loss = fn.DihedralLoss.apply(xyz, rec, idx, None, None)
    with pytest.raises(NotImplementedError, match="dihedral"):
        loss.backward()
    # double backward through the geometry
    rr = r.clone().requires_grad_()
    ds, dv = blk(sec["s"].to(DEV), sec["v"].to(DEV), rr, nbrs)
    (g,) = torch.autograd.grad(ds.sum() + dv.sum(), rr, create_graph=True)
    with pytest.raises(RuntimeError):
        g.sum().backward()
