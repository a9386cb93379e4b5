"""On-device collation of variable-length proteins (data.DeviceProteinDataset) and the PCN step it feeds.

    python tools/bench_protein_batches.py [--proteins 256] [--batch 64] [--steps 8] [--calls 200] [--out DIR]

Dataset: a seeded ragged set like the c4 workload -- residues drawn in 120..400, 6..14 atoms per residue, C-alpha graph at
15.5 A; PCN with F = 512, 9 cross layers; batches of 64 proteins.  Reports, as JSON lines with the card name, power limit
and SM clock read in the same run:
  * collate: the static collate (two launches) per call, eager and replayed from a CUDA graph, CUDA events over ``calls``
    calls; against the host path (per-protein concatenation + train.to_static_pcn_batch + H2D), host clock to a synchronise;
  * steps: one GraphedTrainStep captured at worst-case capacities replaying ragged batches (collate into its static buffers
    + replay) against eager PCNTrainStep steps on the unpadded batches, CUDA events over ``steps`` steps;
  * padding: one batch of a length-bucketed epoch replayed by graphs captured at worst-case capacities, at the capacities of
    the whole bucket plan, at those of its own bucket and at the batch's exact size (train.to_static_pcn_batch, no pad
    rows), in alternating rounds.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from coarsegrainingvae_b200 import data, synthetic, train     # noqa: E402
from coarsegrainingvae_b200.factory import build_pcn     # noqa: E402

DEV = "cuda"
CUTOFF, F, N_RBF, LAYERS = 15.5, 512, 8, 9
GAMMA, KAPPA = 1.0, 1.0


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def protein(rng, n_res):
    per = rng.integers(6, 15, size=n_res)
    start = np.concatenate([[0], np.cumsum(per)[:-1]])
    n_at = int(per.sum())
    ca = synthetic.lattice_points(n_res, 5.2, rng)
    cg_map = np.repeat(np.arange(n_res), per)
    xyz = (ca[cg_map] + rng.normal(scale=1.5, size=(n_at, 3))).astype(np.float32)
    ca_idx = start + 1
    xyz[ca_idx] = ca
    chain = np.arange(n_at - 2)
    bonds = np.concatenate([np.stack([chain, chain + 1], 1), np.stack([chain, chain + 2], 1)], 0)
    r = start[:-1]
    dihe = np.concatenate([np.stack([r, r + 1, r + 2, start[1:]], 1), np.stack([r + 1, r + 2, start[1:], start[1:] + 1], 1)], 0)
    return {"xyz": xyz, "ca_xyz": ca, "res": rng.integers(1, 21, size=n_res), "cg_map": cg_map, "bond_edge_list": bonds,
            "dihe_idxs": dihe, "ca_idx": ca_idx, "seq": "A" * n_res}


T0 = time.perf_counter()


def log(msg):
    print("[%7.1f s] %s" % (time.perf_counter() - T0, msg), file=sys.stderr, flush=True)


def events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def host_collate(items, idx, caps):
    """the host pipeline: per-protein concatenation with offsets, to_static_pcn_batch, H2D of every tensor"""
    cols = {k: [] for k in ("xyz", "ca_xyz", "res", "cg_map", "bond_edge_list", "CG_nbr_list", "ca_idx", "dihe_idxs")}
    a_off = r_off = 0
    for i in idx:
        p = items[i]
        for k in ("xyz", "ca_xyz", "res"):
            cols[k].append(p[k])
        cols["cg_map"].append(p["cg_map"] + r_off)
        cols["CG_nbr_list"].append(p["CG_nbr_list"] + r_off)
        for k in ("bond_edge_list", "ca_idx", "dihe_idxs"):
            cols[k].append(p[k] + a_off)
        a_off += p["xyz"].shape[0]
        r_off += p["ca_xyz"].shape[0]
    batch = train.to_static_pcn_batch({k: torch.cat(v, 0) for k, v in cols.items()}, caps)
    return {k: v.to(DEV) for k, v in batch.items() if torch.is_tensor(v)}


def make_step(batch, capturable=True):
    torch.manual_seed(3)
    model = build_pcn(F, N_RBF, CUTOFF, LAYERS).to(DEV)
    tr = train.PCNTrainStep(model, GAMMA, KAPPA, capturable=capturable)
    tr.prepare(batch, None)
    return tr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proteins", type=int, default=256)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = []

    def emit(rec):
        rec["device"] = card()
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    rng = np.random.default_rng(2024)
    log("building %d proteins" % a.proteins)
    prots = [protein(rng, int(rng.integers(120, 401))) for _ in range(a.proteins)]
    t0 = time.perf_counter()
    ds = data.DeviceProteinDataset(prots, CUTOFF)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    B, P = a.batch, a.proteins
    batches = [rng.permutation(P)[:B].tolist() for _ in range(max(a.steps, 8))]
    worst = ds.capacities(batch_size=B)
    order = np.argsort(ds.sizes[:, 0], kind="stable")
    buckets = [order[i:i + B].tolist() for i in range(0, P - B + 1, B)]
    bucketed = ds.capacities(batches=buckets)

    log("dataset on the device in %.1f s" % build_s)
    # ---- collate
    idx_d = [torch.tensor(b, device=DEV) for b in batches]
    out = ds.collate(idx_d[0], static=True, capacities=worst)
    moved = sum(int(t.numel() * t.element_size()) for k, t in out.items() if torch.is_tensor(t))
    for i in range(10):
        ds.collate(idx_d[i % len(idx_d)], static=True, out=out)
    eager_ms = events_ms(lambda i: ds.collate(idx_d[i % len(idx_d)], static=True, out=out), a.calls)
    static_idx = idx_d[0].clone()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ds.collate(static_idx, static=True, out=out)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        ds.collate(static_idx, static=True, out=out)
    for _ in range(10):
        g.replay()
    graph_ms = events_ms(lambda i: g.replay(), a.calls)
    ptr = ds.item_ptr.cpu().numpy()
    host_items = []
    for i in range(P):
        item = {k: ds.store[k][ptr[kind][i]:ptr[kind][i + 1]].cpu() for k, kind, *_ in data._PROTEIN_KEYS}
        host_items.append(item)
    lists_caps = {k: worst[k] for k in ("CG_nbr_list", "bond_edge_list", "dihe_idxs", "ca_idx")}
    host_collate(host_items, batches[0], lists_caps)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_host = 10
    for i in range(n_host):
        host_collate(host_items, batches[i % len(batches)], lists_caps)
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - t0) * 1e3 / n_host
    emit({"what": "collate", "proteins": P, "batch": B, "dataset_build_s": round(build_s, 2), "capacities": worst,
          "atoms_per_bead": ds.atoms_per_bead, "bytes_written": moved, "eager_us": round(eager_ms * 1e3, 1),
          "graph_replay_us": round(graph_ms * 1e3, 1), "host_path_us": round(host_ms * 1e3, 1),
          "written_GBps_graph": round(moved / (graph_ms * 1e-3) / 1e9, 1)})

    # ---- graphed steps over ragged batches vs eager unpadded steps
    log("capturing the step at worst-case capacities")
    trg = make_step(out)
    step = train.GraphedTrainStep(trg, out, None)
    raws = [ds.collate(b) for b in batches]
    log("eager step")
    tre = make_step(raws[0], capturable=False)
    log("timing steps")
    for i in range(2):
        ds.collate(idx_d[i], static=True, out=step.static)
        step.step({})
        tre.step(raws[i], None)
    torch.cuda.synchronize()

    def graphed(i):
        ds.collate(idx_d[i % len(idx_d)], static=True, out=step.static)
        step.step({})
    res = {"graphed_ms": [], "eager_ms": []}
    for _ in range(a.rounds):
        res["graphed_ms"].append(events_ms(graphed, a.steps))
        res["eager_ms"].append(events_ms(lambda i: tre.step(raws[i % len(raws)], None), a.steps))
    gm, em = float(np.median(res["graphed_ms"])), float(np.median(res["eager_ms"]))
    emit({"what": "steps", "batch": B, "steps": a.steps, "rounds": a.rounds, "graphed_padded_ms": round(gm, 2),
          "eager_unpadded_ms": round(em, 2), "graphed_steps_per_s": round(1e3 / gm, 2), "eager_steps_per_s": round(1e3 / em, 2),
          "all_ms": res})
    del step, trg, tre
    torch.cuda.empty_cache()

    # ---- padding overhead on one batch of the bucketed epoch
    b = buckets[len(buckets) // 2]
    raw = ds.collate(b)
    exact_lists = {k: int(raw[k].shape[0]) for k in ("CG_nbr_list", "bond_edge_list", "dihe_idxs", "ca_idx")}
    own = ds.capacities(batches=[b])
    variants = {"worst": ds.collate(b, static=True, capacities=worst),
                "bucket_plan": ds.collate(b, static=True, capacities=bucketed),
                "own_bucket": ds.collate(b, static=True, capacities=own),
                "exact": {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in train.to_static_pcn_batch({k: v.cpu() for k, v in raw.items()
                                                                               if torch.is_tensor(v)}, exact_lists).items()}}
    graphs = {}
    for name, batch in variants.items():
        log("capturing the %s graph" % name)
        graphs[name] = train.GraphedTrainStep(make_step(batch), batch, None)
    times = {name: [] for name in graphs}
    for _ in range(a.rounds):
        for name, gs in graphs.items():
            gs.step({})
            times[name].append(events_ms(lambda i: gs.step({}), a.steps))
    med = {name: float(np.median(v)) for name, v in times.items()}
    emit({"what": "padding", "batch_atoms": int(raw["xyz"].shape[0]), "batch_residues": int(raw["ca_xyz"].shape[0]),
          "rows": {k: [int(v["xyz"].shape[0]), int(v["ca_xyz"].shape[0]), int(v["CG_nbr_list"].shape[0])] for k, v in variants.items()},
          "ms": {k: round(v, 2) for k, v in med.items()},
          "overhead_vs_exact": {k: round(med[k] / med["exact"] - 1.0, 3) for k in med if k != "exact"}, "all_ms": times})
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_protein_batches.jsonl"), "w") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
