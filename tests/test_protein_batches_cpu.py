"""CPU: the capacity arithmetic of data.DeviceProteinDataset, the host-side layout of the collate plan, and the data-parallel
denominators of capacity-padded PCN batches (gloo, world size 2).  No kernels run."""
import ctypes
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch import nn

from coarsegrainingvae_b200.data import PROTEIN_KINDS, protein_capacities

# columns: atoms, residues, bonds, C-alpha edges, dihedrals, C-alpha indices
SIZES = np.array([[100, 12, 150, 40, 22, 12],
                  [310, 40, 600, 120, 78, 40],
                  [55, 7, 80, 9, 12, 7],
                  [220, 30, 390, 95, 58, 30],
                  [8, 1, 7, 0, 0, 1]], dtype=np.int64)


def test_capacities_from_batch_size():
    assert PROTEIN_KINDS == ("atoms", "residues", "bonds", "ca_edges", "dihedrals", "ca_idx")
    caps = protein_capacities(SIZES, 14, batch_size=2)
    # the two largest entries of every column, whichever proteins they belong to; 530 atoms -> ceil(530 / 14) = 38 pad beads
    assert caps == {"xyz": 530, "ca_xyz": 70 + 38, "bond_edge_list": 990, "CG_nbr_list": 215, "dihe_idxs": 136,
                    "ca_idx": 70}
    caps = protein_capacities(SIZES, 4, batch_size=1)
    assert caps == {"xyz": 310, "ca_xyz": 40 + 78, "bond_edge_list": 600, "CG_nbr_list": 120, "dihe_idxs": 78, "ca_idx": 40}
    everything = protein_capacities(SIZES, 3, batch_size=99)        # more slots than proteins: all of them
    tot = SIZES.sum(0)
    assert everything["xyz"] == tot[0] and everything["ca_xyz"] == tot[1] + -(-tot[0] // 3)


def test_capacities_from_planned_batches():
    batches = [[0, 2, -1], [4, 4, 4], [1, -1, -1], [3, 2, 0]]
    caps = protein_capacities(SIZES, 5, batches=batches)
    per_batch = np.stack([SIZES[[0, 2]].sum(0), SIZES[[4, 4, 4]].sum(0), SIZES[[1]].sum(0), SIZES[[3, 2, 0]].sum(0)])
    want = per_batch.max(0)                                          # the worst planned batch per kind
    assert caps["xyz"] == want[0] == 375 and caps["ca_xyz"] == want[1] + 75
    assert [caps[k] for k in ("bond_edge_list", "CG_nbr_list", "dihe_idxs", "ca_idx")] == list(want[2:])
    empty = protein_capacities(SIZES, 5, batches=[[-1, -1]])
    assert all(v == 0 for v in empty.values())


def test_collate_plan_layout_matches_library():
    """ops.CollatePlan is passed by pointer to cgvae_collate: its size must be the library's sizeof(cgvae_collate_plan)."""
    from coarsegrainingvae_b200 import _lib, ops
    if not os.path.exists(_lib.LIB_PATH):
        from coarsegrainingvae_b200.build import build
        build()
    lib = _lib.load()
    assert ctypes.sizeof(ops.CollatePlan) == lib.cgvae_collate_plan_bytes()
    assert ctypes.sizeof(ops._CollateOut) == 48


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


# live (atoms, residues, bonds, dihedrals) of the two ranks' shards, and the padded capacities both ranks share
LIVE = [(1210, 151, 2380, 290), (845, 104, 1650, 198)]
CAPS = (1400, 260, 2600, 320)


def _dp_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from coarsegrainingvae_b200.train import PCNTrainStep
    tr = PCNTrainStep(nn.Linear(1, 1), gamma=2.0, kappa=0.5, optimizer="torch")
    a, r, b, d = LIVE[rank]
    one = lambda v: torch.tensor([v], dtype=torch.int64)
    batch = {"xyz": torch.zeros(CAPS[0], 3), "ca_xyz": torch.zeros(CAPS[1], 3), "bond_edge_list": torch.zeros(CAPS[2], 2,
             dtype=torch.int64), "dihe_idxs": torch.zeros(CAPS[3], 4, dtype=torch.int64), "atom_count": one(a),
             "res_count": one(r), "bond_count": one(b), "dihe_count": one(d), "loss_norms": torch.ones(3)}
    first = tr.update_dp_norms(dict(batch))
    # a second call writes into the existing tensors (what a captured graph reads)
    keep = first["dp_norms"], first["dihe_norm"]
    first["dihe_count"].fill_(d + 10 * (rank + 1))
    second = tr.update_dp_norms(first)
    assert second["dp_norms"] is keep[0] and second["dihe_norm"] is keep[1]
    out.put((rank, first["dp_norms"].tolist(), second["dihe_norm"].tolist()))
    dist.barrier()
    dist.destroy_process_group()


def test_update_dp_norms_uses_live_counts_on_ragged_shards():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=300) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    glob = np.array(LIVE, dtype=np.float64).sum(0) / world
    dihe_after = (LIVE[0][3] + 10 + LIVE[1][3] + 20) / world
    for rank, norms, dihe in results:
        # global LIVE counts / world -- not the padded shapes (1400, 260, 2600), and the dihedral norm is filled
        assert norms[0] == glob[0] and norms[1] == glob[1] and norms[2] == glob[2], (rank, norms)
        assert dihe == [dihe_after], (rank, dihe)
    assert results[0][1:] == results[1][1:]


def _protein(n_res=5, per=3):
    n_at = n_res * per
    return {"xyz": np.zeros((n_at, 3), np.float32), "ca_xyz": np.zeros((n_res, 3), np.float32),
            "res": np.ones(n_res, np.int64), "cg_map": np.repeat(np.arange(n_res), per),
            "bond_edge_list": np.stack([np.arange(n_at - 1), np.arange(1, n_at)], 1),
            "dihe_idxs": np.stack([np.arange(n_at - 3) + k for k in range(4)], 1), "ca_idx": np.arange(n_res) * per + 1}


def test_construction_rejects_indices_outside_their_protein():
    """IndexError before anything reaches the device: every index must lie inside its own protein (a ca_idx entry past
    the protein's atoms would make the C-alpha pin predicate depend on which proteins share a batch)."""
    import pytest
    from coarsegrainingvae_b200.data import DeviceProteinDataset
    bad = []
    for key, val in (("cg_map", 5), ("bond_edge_list", 15), ("dihe_idxs", -1), ("ca_idx", 15)):
        p = _protein()
        arr = np.array(p[key])
        arr.reshape(-1)[-1] = val
        p[key] = arr
        bad.append((key, p))
    for key, p in bad:
        with pytest.raises(IndexError, match=key):
            DeviceProteinDataset([_protein(), p], cg_cutoff=8.0)
    with pytest.raises(ValueError):
        DeviceProteinDataset([dict(_protein(), cg_map=np.zeros(4, np.int64))], cg_cutoff=8.0)
    with pytest.raises(RuntimeError):
        DeviceProteinDataset([_protein()], cg_cutoff=8.0, device="cpu")
