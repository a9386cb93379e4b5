"""CPU: gradients to atom / bead coordinates and to the r_ij / r_iI of the block API, through the real autograd nodes
running on the kernel emulator (tests/emulator.py + tests/coord_emulator.py) in float64, against the oracle's autograd
at 1e-10.  This pins the derivations the geometry-backward kernels implement; the kernels are checked on the GPU
(test_gpu_coord_grad.py)."""
import pytest
import torch

import coarsegrainingvae_b200 as cg
from tests import coord_cases as cc, coord_emulator
from tests.golden_util import load, section

TOL = 1e-10


@pytest.fixture(autouse=True)
def _emulated(monkeypatch):
    coord_emulator.install(monkeypatch)


@pytest.mark.parametrize("tag", ["k3", "k4", "k9", "k3w"])
def test_block_api_r_ij(tag):
    cc.check(*cc.block_r("cpu", tag, torch.float64), TOL)


def test_contraction_r_iI():
    cc.check(*cc.contraction_r("cpu", torch.float64), TOL)


@pytest.mark.parametrize("tag", ["vae_sym", "vae_noneq"])
def test_cgvae_loss_coordinates(tag):
    cc.check(*cc.cgvae_coords("cpu", tag, torch.float64), TOL)


@pytest.mark.parametrize("tag,ca_pin", [("pcn_cross", True), ("pcn_plain", True), ("pcn_cross", False)])
def test_pcn_ca_xyz(tag, ca_pin):
    cc.check(*cc.pcn_coords("cpu", tag, torch.float64, ca_pin), TOL)


def test_edge_weight_gradient_raises():
    z = load("blocks_small.npz")
    sec = section(z, "k3w")
    blk = cg.EquiMessageBlock(feat_dim=int(z["meta/F"]), activation="swish", n_rbf=int(z["meta/R"]),
                              cutoff=float(z["meta/cutoff"]), dropout=0.0).double()
    w = sec["w"].double().requires_grad_()
    ds, dv = blk(sec["s"].double(), sec["v"].double(), torch.from_numpy(z["in/r"]).double(), torch.from_numpy(z["in/nbrs"]),
                 edge_wgt=w)
    with pytest.raises(NotImplementedError, match="edge_wgt"):
        (ds.sum() + dv.sum()).backward()


def test_no_geometry_node_without_coordinate_grad():
    """coordinates that do not require grad (or no grad mode) keep the plain geometry: no EdgeGeometry node"""
    z = load("blocks_small.npz")
    graph = cg.ops.build_graph(torch.from_numpy(z["in/nbrs"]), int(section(z, "k3")["s"].shape[0]))
    r = torch.from_numpy(z["in/r"]).double()
    assert cg.functions.edge_geometry(graph, None, None, 4, 5.0, r_edge=r).basis.grad_fn is None
    with torch.no_grad():
        assert cg.functions.edge_geometry(graph, None, None, 4, 5.0, r_edge=r.requires_grad_()).basis.grad_fn is None
    assert cg.functions.edge_geometry(graph, None, None, 4, 5.0, r_edge=r).basis.grad_fn is not None
