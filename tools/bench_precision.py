"""Times the two matmul precision modes ("highest" = 3xTF32, "high" = 1xTF32, ops.set_matmul_precision) side by side.

    python tools/bench_precision.py --out DIR [--rounds 5] [--only gemm,message,steps]

Measured in one run, with the two modes alternating round by round (CUDA events around CUDA-graph replays, median over
the rounds):
  * the tcgen05 GEMMs of the c2 (chignolin, F = 600) and c4 (protein, F = 512) steps, each with its scale-relative error
    against float64 (tests.golden_util.rel_err) in both modes;
  * the tensor-core message forward on the c2 atom graph (K = 3) and on the c4 cross block (16 000 beads, K = 4);
  * the whole c2 graphed train step and the whole c4 graphed PCN step (one CUDA graph captured per mode).
The device name, power limit and SM clock are read with nvidia-smi (query only) in the same run.  One JSON object per
measurement goes to DIR/bench_precision.jsonl and to stdout.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODES = ("highest", "high")
GEMMS = [  # (config, form, M, N, K): the shapes of the steps' node-level contractions
    ("c2", "NT", 350, 1800, 600), ("c2", "NN", 350, 600, 1800), ("c2", "TN", 1800, 600, 350),
    ("c4", "NT", 16000, 2048, 512), ("c4", "NN", 16000, 512, 2048), ("c4", "TN", 2048, 512, 16000),
    ("c4", "NN", 48000, 512, 512), ("c4", "TN", 512, 512, 48000),
]


def _device_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "nvidia-smi unavailable: %s" % e
    return {"what": "device", "query": q, "nvidia_smi": out}


def _time(fn, iters):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _alternate(fns, rounds, iters, warm=3):
    """fns: {mode: callable}; both warmed, then `rounds` rounds of `iters` calls each, modes alternating -> per mode the
    median and the spread (min, max) of the per-call times in ms"""
    import torch
    for m in MODES:
        for _ in range(warm):
            fns[m]()
    torch.cuda.synchronize()
    t = {m: [] for m in MODES}
    for r in range(rounds):
        order = MODES if r % 2 == 0 else MODES[::-1]
        for m in order:
            t[m].append(_time(fns[m], iters))
    return {m: {"ms": statistics.median(v), "min": min(v), "max": max(v)} for m, v in t.items()}


def _iters_for(fn, target_ms=200.0):
    import torch
    fn()
    torch.cuda.synchronize()
    one = _time(fn, 3)
    return max(3, min(2000, int(target_ms / max(one, 1e-3))))


def _graphed(fn, reps):
    """`reps` calls of fn captured as one CUDA graph (kernel time, not the host cost of the Python wrappers); returns the
    replay and keeps the graph alive through it"""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for _ in range(reps):
            fn()
    torch.cuda.synchronize()
    return g.replay


def _per_call(times, reps):
    return {m: {k: v / reps for k, v in t.items()} for m, t in times.items()}


def _result(row, times):
    row.update({"ms_" + m: times[m]["ms"] for m in MODES})
    row.update({"spread_ms_" + m: [times[m]["min"], times[m]["max"]] for m in MODES})
    row["speedup_high"] = times["highest"]["ms"] / times["high"]["ms"]
    return row


def bench_gemms(dev, rounds, emit):
    import torch
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops
    forms = {"NT": ops.GEMM_NT, "NN": ops.GEMM_NN, "TN": ops.GEMM_TN}
    for cfg, fname, M, N, K in GEMMS:
        form = forms[fname]
        gen = torch.Generator(device=dev).manual_seed(M + N + K)
        sa, sb = {"NT": ((M, K), (N, K)), "NN": ((M, K), (K, N)), "TN": ((K, M), (K, N))}[fname]
        A = torch.randn(*sa, device=dev, generator=gen)
        B = torch.randn(*sb, device=dev, generator=gen) / math.sqrt(K)
        C = torch.empty(M, N, device=dev)
        A64, B64 = A.double(), B.double()
        ref = {"NT": lambda: A64 @ B64.t(), "NN": lambda: A64 @ B64, "TN": lambda: A64.t() @ B64}[fname]()
        errs = {}
        fns = {}
        reps = 20
        for m in MODES:
            with cg.matmul_precision(m):            # the mode is fixed at capture
                ops.gemm(form, A, B, M, N, K, out=C)
                torch.cuda.synchronize()
                errs[m] = float((C.double() - ref).abs().max() / ref.abs().max())
                fns[m] = _graphed(lambda: ops.gemm(form, A, B, M, N, K, out=C), reps)
        del ref, A64, B64
        iters = _iters_for(fns["highest"])
        times = _per_call(_alternate(fns, rounds, iters), reps)
        flops = 2.0 * M * N * K
        row = {"what": "gemm", "config": cfg, "form": fname, "M": M, "N": N, "K": K, "iters_per_round": iters,
               "rel_err_highest": errs["highest"], "rel_err_high": errs["high"],
               "tflops_highest": flops / times["highest"]["ms"] * 1e-9, "tflops_high": flops / times["high"]["ms"] * 1e-9,
               "operand_mb": 4.0 * (A.numel() + B.numel() + C.numel()) / 2 ** 20}
        row["iters_per_round"] = iters * reps
        emit(_result(row, times))
        fns = None
        torch.cuda.empty_cache()


def bench_message(dev, rounds, emit):
    import numpy as np
    import torch
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops, synthetic
    cases = [("c2 atom graph (2 x 175 atoms, cutoff 12)", 3, 350, 2.2, 12.0, 600, 10),
             ("c4 cross block (16 000 beads, cutoff 15.5)", 4, 16000, 5.2, 15.5, 512, 8)]
    old = ops.MSG_TC
    ops.MSG_TC = "1"             # the tensor-core forward on both graphs (the modes differ only there)
    try:
        for label, K, n, spacing, cutoff, F, R in cases:
            g = torch.Generator().manual_seed(n)
            xyz = synthetic.lattice_points(n, spacing, np.random.default_rng(n), rotate=False)
            half = ops.radius_graph(torch.as_tensor(xyz, device=dev), cutoff, True)
            graph = ops.build_graph(torch.cat([half, half.flip(1)], 0), n)
            x = torch.as_tensor(xyz, device=dev)
            geom = ops.edge_geometry(graph, x, x, R, cutoff)
            phi = torch.randn(n, K, F, generator=g).to(dev)
            v = torch.randn(n, 3, F, generator=g).to(dev)
            Wf = (torch.randn(K * F, R, generator=g) * 0.5).to(dev)
            bf = (torch.randn(K * F, generator=g) * 0.5).to(dev)
            vr = v if K == 4 else None
            fns = {}
            reps = 10
            for m in MODES:
                with cg.matmul_precision(m):
                    fns[m] = _graphed(lambda: ops.message_fwd(K, phi, v, vr, geom, Wf, bf, None, None, want_q=K == 4), reps)
            iters = _iters_for(fns["highest"])
            times = _per_call(_alternate(fns, rounds, iters), reps)
            emit(_result({"what": "message_fwd", "graph": label, "K": K, "F": F, "edges": int(graph.n_edges),
                          "iters_per_round": iters * reps}, times))
            fns = None
    finally:
        ops.MSG_TC = old
    torch.cuda.empty_cache()


def bench_steps(dev, rounds, emit):
    import torch
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops, synthetic
    from coarsegrainingvae_b200.factory import build_cgvae, build_pcn
    from coarsegrainingvae_b200.train import GraphedTrainStep, PCNTrainStep, TrainStep, to_static_batch, to_static_pcn_batch

    def rad(xyz, c):
        return ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=dev), c).cpu().numpy()

    # c2: the bench.py workload (chignolin, batch 2), one graph per mode, the same seeded weights
    cfg = dict(synthetic.CONFIGS["c2_chignolin"])
    raw = synthetic.cgvae_batch(cfg, 0, rad, cg.CG_collate)
    B, n, ncg = cfg["batch"], cfg["n_atoms"], cfg["n_cgs"]
    caps = {"nbr_list": B * n * (n - 1) // 2, "CG_nbr_list": max(B * ncg * (ncg - 1) // 2, 1),
            "bond_edge_list": raw["bond_edge_list"].shape[0] + 64}
    batch = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in to_static_batch(raw, caps).items()}
    steps, keep = {}, []
    for m in MODES:
        torch.manual_seed(123)
        model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"],
                            cfg["cg_cutoff"], cfg["n_cgs"]).to(dev)
        tr = TrainStep(model, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01, capturable=True)
        tr.prepare(batch, None)
        with cg.matmul_precision(m):
            g = GraphedTrainStep(tr, batch, None)
        keep.append((tr, g))
        steps[m] = (lambda g=g: g.step(batch))
    times = _alternate(steps, rounds, 50)
    emit(_result({"what": "step", "config": "c2 chignolin train step, batch 2, one CUDA graph", "iters_per_round": 50}, times))
    for tr, _ in keep:
        tr.flat.release()
    keep, steps = [], {}
    torch.cuda.empty_cache()

    # c4: the PCN step of bench.py's secondary workloads (64 proteins x 2 000 atoms)
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    raw = synthetic.pcn_batch(cfg, 0, rad, n_proteins=cfg["batch"])
    caps = {k: int(raw[k].shape[0]) + 64 for k in ("CG_nbr_list", "bond_edge_list", "dihe_idxs", "ca_idx")}
    batch = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in to_static_pcn_batch(raw, caps).items()}
    for m in MODES:
        torch.manual_seed(123)
        model = build_pcn(cfg["n_basis"], cfg["n_rbf"], cfg["cg_cutoff"], cfg["dec_nconv"]).to(dev)
        tr = PCNTrainStep(model, 1.0, 0.1, lr=1e-4, capturable=True)
        tr.prepare(batch, None)
        with cg.matmul_precision(m):
            g = GraphedTrainStep(tr, batch, None)
        keep.append((tr, g))
        steps[m] = (lambda g=g: g.step(batch))
    times = _alternate(steps, rounds, 5, warm=2)
    emit(_result({"what": "step", "config": "c4 PCN train step, 64 proteins x 2 000 atoms, one CUDA graph",
                  "iters_per_round": 5, "max_memory_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30}, times))
    for tr, _ in keep:
        tr.flat.release()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_precision.jsonl")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds per measurement (odd: median of the rounds)")
    ap.add_argument("--only", default="gemm,message,steps")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("bench_precision.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_precision.jsonl")
    with open(path, "w") as fh:
        def emit(row):
            line = json.dumps(row)
            print(line, flush=True)
            fh.write(line + "\n")
            fh.flush()
        emit(_device_info())
        only = set(args.only.split(","))
        if "gemm" in only:
            bench_gemms(dev, args.rounds, emit)
        if "message" in only:
            bench_message(dev, args.rounds, emit)
        if "steps" in only:
            bench_steps(dev, args.rounds, emit)
        emit(_device_info())          # clocks after the run


if __name__ == "__main__":
    main()
