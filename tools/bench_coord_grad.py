"""Cost of coordinate gradients: forward + backward with and without ``requires_grad`` on the coordinates.

    python tools/bench_coord_grad.py [--repeats 5] [--iters 5]

Workloads: the c2 model (CGequiVAE, F = 600, 2 x 175 atoms, training loss), the c4 PCN model (64 proteins x ~2 000
atoms, MSE loss, as bench.py's other_workloads builds it) and one EquiMessageBlock (F = 128, R = 7) on the 6 A graph
of 20 000 atoms (~1.5 M directed edges).  Each repeat times both variants with CUDA events over ``iters`` iterations
(after a warm-up), in alternating order; the median over repeats is printed with the card name and power limit as one
JSON line per workload.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import coarsegrainingvae_b200 as cg                      # noqa: E402
from coarsegrainingvae_b200 import functions as fn, ops, synthetic, train     # noqa: E402
from coarsegrainingvae_b200.factory import build_cgvae, build_pcn       # noqa: E402

DEV = "cuda"


def _card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def _radius(xyz, cutoff):
    return ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=DEV), cutoff).cpu().numpy()


def _to(batch):
    return {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in batch.items()}


def c2_workload():
    cfg = dict(synthetic.CONFIGS["c2_chignolin"])
    cfg["batch"] = 2
    batch = _to(synthetic.cgvae_batch(cfg, 0, _radius, cg.CG_collate))
    torch.manual_seed(123)
    model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"], cfg["cg_cutoff"],
                        cfg["n_cgs"]).to(DEV)
    eps = torch.randn(2 * cfg["n_cgs"], cfg["n_basis"], device=DEV)

    def run(coords):
        b = dict(batch)
        if coords:
            b["nxyz"], b["CG_nxyz"] = b["nxyz"].clone().requires_grad_(), b["CG_nxyz"].clone().requires_grad_()
        out = model(b, eps=eps)
        train.training_loss(out, out[4], b["bond_edge_list"], cfg["beta"], cfg["gamma"])[0].backward()
    return "c2 CGequiVAE fwd+bwd (F=600, 2 x 175 atoms)", model, run


def c4_workload():
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    batch = _to(synthetic.pcn_batch(cfg, 0, _radius, n_proteins=cfg["batch"]))
    torch.manual_seed(123)
    model = build_pcn(cfg["n_basis"], cfg["n_rbf"], cfg["cg_cutoff"], cfg["dec_nconv"]).to(DEV)

    def run(coords):
        b = dict(batch)
        if coords:
            b["ca_xyz"] = b["ca_xyz"].clone().requires_grad_()
        out = model(b)
        (out[5] - out[4]).pow(2).mean().backward()
    return "c4 PCN fwd+bwd (F=512, 9 cross layers, %d proteins)" % cfg["batch"], model, run


def layer_workload():
    xyz = torch.as_tensor(synthetic.lattice_points(20000, 2.2, np.random.default_rng(1)), dtype=torch.float32, device=DEV)
    graph = ops.build_graph(ops.radius_graph(xyz, 6.0, undirected=False), 20000)
    torch.manual_seed(11)
    blk = cg.EquiMessageBlock(feat_dim=128, activation="swish", n_rbf=7, cutoff=6.0, dropout=0.0).to(DEV)
    s = torch.randn(20000, 128, device=DEV)
    v = torch.randn(20000, 3, 128, device=DEV)

    def run(coords):
        x = xyz.clone().requires_grad_(coords)
        geom = fn.edge_geometry(graph, x, x, 7, 6.0)
        out_s, out_v = blk.fused(s, v, geom)
        (out_s.sum() + out_v.sum()).backward()
    return "EquiMessageBlock fwd+bwd (F=128, R=7, 20 000 atoms, 6 A, %d edges)" % graph.n_edges, blk, run


def _time(run, model, coords, iters):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        model.zero_grad(set_to_none=True)
        run(coords)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    card = _card()
    for make in (c2_workload, c4_workload, layer_workload):
        name, model, run = make()
        for coords in (False, True):
            _time(run, model, coords, 2)                      # warm-up: module loads, tiles, allocator
        t = {False: [], True: []}
        for r in range(args.repeats):
            for coords in ((False, True) if r % 2 == 0 else (True, False)):
                t[coords].append(_time(run, model, coords, args.iters))
        base, grad = float(np.median(t[False])), float(np.median(t[True]))
        print(json.dumps({"workload": name, "card": card, "ms_without_coord_grad": round(base, 3),
                          "ms_with_coord_grad": round(grad, 3), "ratio": round(grad / base, 3),
                          "spread_without": [round(min(t[False]), 3), round(max(t[False]), 3)],
                          "spread_with": [round(min(t[True]), 3), round(max(t[True]), 3)]}), flush=True)
        model, run = None, None
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
