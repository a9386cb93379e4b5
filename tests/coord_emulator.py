"""TEST-ONLY stand-ins for the coordinate-gradient kernels (csrc/message_geom.cu, the geometry backward and node
reduction of csrc/geom.cu), installed on top of tests/emulator.py.  Each restates, in plain torch, the hand-derived
formula the kernel implements (not torch autograd of the forward), so that the real autograd nodes run on it in float64
against the oracle's autograd pin the derivations."""
import numpy as np
import torch

from coarsegrainingvae_b200 import ops
from tests import emulator as em


def edge_geometry_bwd(graph, n_rbf, cutoff, xyz_send, xyz_recv, d_basis, d_unit, edge_wgt=None, r_edge=None):
    r = r_edge[graph.eid] if r_edge is not None else xyz_send[graph.col] - xyz_recv[em._recv_of_slot(graph)]
    dt = r.dtype
    d = ((r ** 2 + 1e-8).sum(-1)) ** 0.5
    u = r / d[:, None]
    gd = torch.zeros_like(d)
    gu = torch.zeros_like(r)
    if d_unit is not None:
        gu, gd = d_unit[:, :3], d_unit[:, 3].clone()
    if d_basis is not None:
        R = n_rbf
        a = np.pi / cutoff
        coef = torch.arange(1, R + 1).to(dt) * np.pi / cutoff
        env = 0.5 * (torch.cos(a * d) + 1)
        denv = -0.5 * a * torch.sin(a * d)
        rbf = torch.sin(coef[None, :] * d[:, None]) / d[:, None]
        drbf = (coef[None, :] * torch.cos(coef[None, :] * d[:, None]) - rbf) / d[:, None]
        dbd = (d_basis[:, :R] * (drbf * env[:, None] + rbf * denv[:, None])).sum(1) + d_basis[:, R] * denv
        if edge_wgt is not None:
            dbd = dbd * edge_wgt[graph.eid]
        gd = gd + dbd * (d < cutoff).to(dt)
    dr = gd[:, None] * u + (gu - (u * gu).sum(1, keepdim=True) * u) / d[:, None]
    if r_edge is not None:
        out = torch.zeros_like(r_edge)
        out[graph.eid] = dr
        return out
    return dr


def edge_coord_reduce(graph, dr, same):
    g_send = torch.zeros(graph.n_send, 3, dtype=dr.dtype).index_add_(0, graph.col, dr)
    g_recv = -torch.zeros(graph.n_recv, 3, dtype=dr.dtype).index_add_(0, em._recv_of_slot(graph), dr)
    if same:
        return g_send + g_recv, None
    return g_send, g_recv


def message_geom_bwd(n_split, phi, v_send, v_recv, geom, Wf, bf, g_out_s, g_out_v):
    g = geom.graph
    F = phi.shape[-1]
    W = em._filter_matrix(Wf, bf, n_split, F, geom.rb)          # [K, RB, F]
    i, j = em._recv_of_slot(g), g.col
    b, u = geom.basis, geom.unit[:, :3]
    gv = g_out_v[i]
    ku = 1 if n_split == 9 else 2
    d_unit = torch.zeros(g.n_edges, 4, dtype=phi.dtype)
    d_unit[:, :3] = ((phi[j, ku] * (b @ W[ku]))[:, None, :] * gv).sum(2)
    if n_split == 9:
        return None, d_unit
    a = torch.zeros(g.n_edges, n_split, F, dtype=phi.dtype)
    a[:, 1] = g_out_s[i] * phi[j, 1]
    a[:, 2] = (gv * u[:, :, None]).sum(1) * phi[j, 2]
    if v_send is not None:
        vj = v_send[j]
        a[:, 0] = (gv * vj).sum(1) * phi[j, 0]
        if n_split == 4:
            a[:, 3] = (gv * em._cross(v_recv[i], vj)).sum(1) * phi[j, 3]
    return torch.einsum("ekf,krf->er", a, W), d_unit


def message9_bwd(phi, s, sbar, v, vbar, geom, Wf, bf, residual, g_s, g_sbar, g_v, g_vbar, keep_gw=False):
    outs = em.message9_bwd(phi, s, sbar, v, vbar, geom, Wf, bf, residual, g_s, g_sbar, g_v, g_vbar)
    if not keep_gw:
        return outs
    # gw[e] = gm[e] * phi[j] per receiver-CSR slot (the same gm terms as emulator.message9_bwd)
    g = geom.graph
    n, F = s.shape
    i, j = em._recv_of_slot(g), g.col
    u = geom.unit[:, :3]
    dot = lambda a, b: (a * b).sum(1)
    gm = torch.stack([
        g_s[i] * s[i],
        dot(g_v[i], u[:, :, None].expand(-1, -1, F)),
        dot(g_v[i], v[j]),
        dot(g_v[i], em._cross(v[i], vbar[j])),
        sbar[i] * dot(g_v[i], vbar[j]),
        dot(g_vbar[i], vbar[j]),
        sbar[i] * dot(g_vbar[i], v[j]),
        dot(g_vbar[i], em._cross(v[i], v[j])),
        dot(g_vbar[i], em._cross(vbar[i], vbar[j])),
    ], 1)
    return tuple(outs) + ((gm * phi[j]).reshape(g.n_edges, 9 * F),)


def message9_geom_bwd(phi, geom, Wf, bf, gw, g_v):
    R = geom.n_rbf
    d_basis = torch.zeros(geom.graph.n_edges, geom.rb, dtype=phi.dtype)
    d_basis[:, :R] = gw @ Wf
    d_basis[:, R] = gw @ bf
    _, d_unit = message_geom_bwd(9, phi, None, None, geom, Wf, bf, None, g_v)
    return d_basis, d_unit


_NAMES = ["edge_geometry_bwd", "edge_coord_reduce", "message_geom_bwd", "message9_bwd", "message9_geom_bwd"]


def install(monkeypatch):
    """tests/emulator.py plus the coordinate-gradient ops, for the duration of one test."""
    em.install(monkeypatch)
    for name in _NAMES:
        monkeypatch.setattr(ops, name, globals()[name])
