#!/usr/bin/env python
"""bench.py -- headline benchmark of the CGVAE equivariant message-passing hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cuda|reference] [--workload c2_chignolin|c1_dipeptide]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): chignolin all-atom CGVAE,
175 atoms, n_cgs 6, batch 2, enc_nconv 2 / dec_nconv 9, n_basis 600, n_rbf 10, cutoffs 12 / 25 A, synthetic
jittered-lattice conformations, random-init weights.  One "step" = one optimisation step of the reference's
training loop (scripts/utils.py:112-157): make_directed + CSR build + edge geometry + forward + loss + backward
(+ gradient all-reduce over NCCL when N > 1) + clip_grad_norm_(0.01) + Adam.

Prints ONE JSON line (rank 0).  `value` = conformations/s with the batch resident in HBM; `e2e` = the same through
the public API from pinned HOST buffers with the H2D copy and the D2H loss read inside the timed region;
`kernel_family_shares` = CUPTI timeline of graph replays grouped into kernel families; `roofline` = the modelled family
with the largest share of the step (algorithmic bytes or flops of one step / its kernel time, against MEASURED_PEAKS.json),
all modelled families in `roofline_kernels`; `hbm_floor` = the step's compulsory HBM traffic / measured bandwidth;
`other_workloads` = BASELINE configs 3 / 4 / 5 (ensemble sampling, PCN protein step, one layer at 20 000 atoms);
`cpu_baseline` = the UNMODIFIED reference (baseline/_ref, tools/install_reference.sh) on this box's host cores, bounded
sample (the oracle port only if the reference install is missing).

--impl reference: times the unmodified reference's own training step (its CPU PyTorch path, all host threads) for the
same metric / config; under torchrun only rank 0 runs and prints.

--dump-outputs DIR (--impl cuda): after the K timed steps, rank 0 writes what the last of them computed as float32 .npy
files: `loss` (the value the step returns), `parameters` (the used parameters after its Adam update) and `gradients` (the
gradients it formed), the two buffers in flat-buffer order and, above 4 Mi floats, sampled at the same seeded positions on
every run.  Inputs, weights and noise are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# DRAM traffic of ONE launch (dram__bytes_read.sum + dram__bytes_write.sum) at the chignolin shapes, from the committed
# ncu --set full captures of tools/profile_kernels.py: profiles/r2_ncu_message_tc_fwd_raw.csv (message forward on the atom
# graph) and profiles/r2_ncu_full_hot_kernels_raw.csv (message backward; the 5400 x 600 weight matrix streamed by the NT
# kernel: 12.96 MB algorithmic; the 350 x 1800 x 600 NT problem of the tcgen05 GEMM: 5.6 MB of operands + output)
NCU_DRAM_BYTES = {"message_atom_fwd": 17.5e6, "message_atom_bwd": 12.5e6, "gemm_stream": 13.06e6, "gemm_tcgen05": 5.24e6}
NCU_TRAFFIC_NOTE = {"gemm_stream": "one NT launch streaming the 5400 x 600 matrix (12.96 MB algorithmic; the NN launch reads 13.25 MB): "
                                   "the matrix is read exactly once",
                    "gemm_tcgen05": "one NT launch 350 x 1800 x 600 (reads only: the 2.5 MB output had not been written back yet)"}
NCU_SOURCE = ("profiles/r2_ncu_message_tc_fwd_raw.csv (forward, tensor-core kernel) / profiles/r2_ncu_full_hot_kernels_raw.csv "
              "(backward): same shapes")

METRIC = "conformations/s (fwd+bwd train step)"
UNIT = "conformations/s"


def _args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="c2_chignolin", choices=["c2_chignolin", "c1_dipeptide"])
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic batches cycled through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of one CUDA graph per step")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads (c3 sampling, c4 protein, c5 layer)")
    ap.add_argument("--fixed-eps", action="store_true", help="pass a fixed noise tensor instead of drawing it inside the step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to --impl cuda")
    return args


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm_gbs=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback")


def _spec(cfg):
    return dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], enc_nconv=cfg["enc_nconv"], dec_nconv=cfg["dec_nconv"],
                atom_cutoff=cfg["atom_cutoff"], cg_cutoff=cfg["cg_cutoff"], decoder="pseudo", breaksym=cfg["n_cgs"] == 3,
                activation="swish")


def _config_json(name, cfg, n_gpus, extra=None):
    out = {"workload": "%s: CGVAE train step, %d atoms x batch %d per GPU, n_cgs %d, enc_nconv %d / dec_nconv %d, n_basis %d, "
                       "n_rbf %d, cutoffs %g/%g A" % (name, cfg["n_atoms"], cfg["batch"], cfg["n_cgs"], cfg["enc_nconv"],
                                                      cfg["dec_nconv"], cfg["n_basis"], cfg["n_rbf"], cfg["atom_cutoff"],
                                                      cfg["cg_cutoff"]),
           "batch_per_gpu": cfg["batch"], "global_batch": cfg["batch"] * n_gpus,
           "parallelism": "dp%d (conformations sharded by rank, one NCCL all-reduce of the used-gradient bucket)" % n_gpus,
           "step": "make_directed + CSR + geometry + fwd + loss + bwd + clip_grad_norm_ + Adam",
           "l2": "no explicit flush: parameters + gradients + Adam state streamed every step are >1 GB, far above the 126 MB L2"}
    if extra:
        out.update(extra)
    return out


class ClockSampler(object):
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md recipe)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- CPU reference arm

def _oracle_step_fn(cfg, pool_size, threads):
    """the reference algorithm on CPU (oracle port): returns (step(i) -> loss, description)."""
    import torch
    from coarsegrainingvae_b200 import synthetic
    from oracle import cgvae_oracle as orc
    from oracle import graph_oracle as gorc
    from coarsegrainingvae_b200.factory import build_cgvae

    torch.set_num_threads(threads)
    torch.manual_seed(123)
    model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"], cfg["cg_cutoff"],
                        cfg["n_cgs"])                                      # parameter container only (CPU tensors)
    P = dict(model.named_parameters())
    spec = _spec(cfg)
    batches = [gorc.collate([{k: v.numpy() for k, v in synthetic.cgvae_sample(cfg, 1234 + 100 + i * cfg["batch"] + k,
                                                                               gorc.radius_graph).items()}
                             for k in range(cfg["batch"])]) for i in range(pool_size)]
    batches = [{k: torch.from_numpy(v) for k, v in b.items()} for b in batches]
    gen = torch.Generator().manual_seed(7)
    eps = torch.randn(cfg["batch"] * cfg["n_cgs"], cfg["n_basis"], generator=gen)
    params = None
    state = {}

    def step(i):
        b = batches[i % pool_size]
        for p in P.values():
            p.grad = None
        out = orc.cgvae_forward(P, spec, b, eps=eps)
        loss = orc.training_loss(out, b, cfg["beta"], cfg["gamma"])[0]
        loss.backward()
        if "opt" not in state:
            used = [p for p in P.values() if p.grad is not None]
            state["used"] = used
            state["opt"] = torch.optim.Adam(used, lr=1e-4)
        torch.nn.utils.clip_grad_norm_(state["used"], 0.01)
        state["opt"].step()
        return float(loss)

    del params
    return step


REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _reference_step_fn(cfg, pool_size, threads):
    """The UNMODIFIED reference (pip-installed into the git-ignored baseline/_ref by tools/install_reference.sh; it travels
    to the GPU box with the snapshot) driven through its own public API on the host CPU: model construction as in
    scripts/run_ala.py:184-209, batches from the reference's get_neighbor_list (data.py:65-82) + CG_collate (data.py:255-289),
    and one iteration of the training loop of scripts/utils.py:112-157 per step (scripts/ itself needs ase / mdtraj, which
    are absent, so the dozen lines of that loop are restated here around the reference's model call).  Returns None when
    baseline/_ref is missing (then the oracle port is timed and reported as kind "port")."""
    if not os.path.isdir(os.path.join(REF_DIR, "CoarseGrainingVAE")):
        return None
    os.environ["CGVAE_REFERENCE_ROOT"] = REF_DIR
    import torch
    from torch import nn
    from coarsegrainingvae_b200 import synthetic
    from oracle import ref_shim
    ref_shim.REFERENCE_ROOT = REF_DIR
    try:
        _, _, ref_cgvae, ref_data = ref_shim.import_reference()
    except Exception:
        return None
    torch.set_num_threads(threads)
    torch.manual_seed(123)
    F, R, act = cfg["n_basis"], cfg["n_rbf"], "swish"
    decoder = ref_cgvae.EquivariantPsuedoDecoder(n_atom_basis=F, n_rbf=R, cutoff=cfg["atom_cutoff"], num_conv=cfg["dec_nconv"],
                                                 activation=act, breaksym=cfg["n_cgs"] == 3)
    encoder = ref_cgvae.EquiEncoder(n_conv=cfg["enc_nconv"], n_atom_basis=F, n_rbf=R, cutoff=cfg["cg_cutoff"], activation=act,
                                    cg_mp=False, dir_mp=False)
    prior = ref_cgvae.CGprior(n_conv=cfg["enc_nconv"], n_atom_basis=F, n_rbf=R, cutoff=cfg["cg_cutoff"], activation=act, dir_mp=False)
    atom_mu = nn.Sequential(nn.Linear(F, F), nn.ReLU(), nn.Linear(F, F))
    atom_sigma = nn.Sequential(nn.Linear(F, F), nn.ReLU(), nn.Linear(F, F))
    model = ref_cgvae.CGequiVAE(encoder, decoder, atom_mu, atom_sigma, cfg["n_cgs"], feature_dim=F, prior_net=prior, det=False,
                                equivariant=True)
    model.train()
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)            # scripts/run_ala.py:211

    def ref_radius(xyz, cutoff):
        return ref_data.get_neighbor_list(torch.as_tensor(xyz), "cpu", cutoff, True).numpy()

    batches = [synthetic.cgvae_batch(cfg, i, ref_radius, ref_data.CG_collate) for i in range(pool_size)]
    beta, gamma, EPS = cfg["beta"], cfg["gamma"], 1e-6

    def step(i):
        batch = batches[i % pool_size]
        S_mu, S_sigma, H_prior_mu, H_prior_sigma, xyz, xyz_recon = model(batch)                     # utils.py:114
        loss_kl = 0.5 * ((S_sigma.pow(2) / H_prior_sigma.pow(2)).sum(-1) + ((S_mu - H_prior_mu).pow(2) / H_prior_sigma).sum(-1)
                         + torch.log(H_prior_sigma.pow(2)).sum(-1) - torch.log(S_sigma.pow(2)).sum(-1) - S_sigma.shape[-1]).mean()
        loss_recon = (xyz_recon - xyz).pow(2).mean()                                                # utils.py:124
        edge_list = batch["bond_edge_list"]
        gen = ((xyz_recon[edge_list[:, 0]] - xyz_recon[edge_list[:, 1]]).pow(2).sum(-1) + EPS).sqrt()
        dat = ((xyz[edge_list[:, 0]] - xyz[edge_list[:, 1]]).pow(2).sum(-1) + EPS).sqrt()
        loss = loss_recon + loss_kl * beta + (gen - dat).pow(2).mean() * gamma                       # utils.py:141
        if loss.item() >= gamma * 200.0 or torch.isnan(loss):                                       # utils.py:145-148
            return float(loss)
        optimizer.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 0.01)
        optimizer.step()
        return float(loss)

    return step


def _cpu_step_fn(cfg, pool_size, threads):
    """(step, kind): the unmodified reference when baseline/_ref is present, else the oracle port."""
    step = _reference_step_fn(cfg, pool_size, threads)
    if step is not None:
        return step, "reference"
    return _oracle_step_fn(cfg, pool_size, threads), "port"


def run_reference(args, cfg):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    step, kind = _cpu_step_fn(cfg, args.pool, threads)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    ms = 1e3 * dt / max(args.steps, 1)
    value = cfg["batch"] / (ms / 1e3)
    sample = "%d full steps of the %s batch (%d conformations each) after %d warm-up" % (args.steps, args.workload,
                                                                                          cfg["batch"], args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": _config_json(args.workload, cfg, args.gpus),
            "reference_impl": ("unmodified wwang2/CoarseGrainingVAE from baseline/_ref on the host CPU cores, torch %s"
                               if kind == "reference" else "oracle port of the reference (baseline/_ref missing), torch %s")
                              % torch.__version__,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))



# --------------------------------------------------------------------------------------------- kernel families / extras

FAMILY_RULES = (("message_atom_fwd", ("message_tc_fwd", "message_fwd_kernel")), ("message_atom_bwd", ("message_bwd_kernel", "filter_grad_finalize")),
                ("message9", ("message9_",)), ("gemm_stream", ("gemm_nt_stream", "gemm_nn_stream")),
                ("gemm_tcgen05", ("gemm_tc_kernel",)), ("gemm_simt", ("gemm_kernel", "gemm_skinny", "gemm_mma", "colsum")),
                ("wgrad_grouped", ("wgrad_grouped",)), ("adam_clip", ("adam_clip", "sumsq_partial")),
                ("graph_build", ("csr_", "scan_kernel", "sort_rows", "edge_geometry", "edge_orientation", "segment_", "tile_count", "tile_fill",
                                 "radius_", "zero_words")),
                ("nodewise", ("update_", "lift_", "gather_rows", "vec_to_planar", "vec_from_planar", "loss_")))


def _family_of(kernel_name):
    for fam, keys in FAMILY_RULES:
        if any(k in kernel_name for k in keys):
            return fam
    return "torch_aten" if ("at::" in kernel_name or "elementwise" in kernel_name or "reduce" in kernel_name
                            or "Memcpy" in kernel_name or "Memset" in kernel_name or "cub::" in kernel_name) else "other"


def _family_shares(run, n_steps):
    """CUPTI timeline (torch.profiler) of n_steps steps -> ({family: us per step}, {family: launches per step}, sum us per step).
    The message family is split by graph size: only the atom-graph launches (the long ones) count as message_atom_*."""
    import collections
    import tempfile
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n_steps):
            run(i)
        torch.cuda.synchronize()
    path = os.path.join(tempfile.gettempdir(), "cgvae_bench_trace_%d.json" % os.getpid())
    prof.export_chrome_trace(path)
    with open(path) as fh:
        ev = json.load(fh)["traceEvents"]
    os.remove(path)
    dur, cnt = collections.defaultdict(float), collections.defaultdict(int)
    for e in ev:
        if e.get("cat") not in ("kernel", "gpu_memset", "gpu_memcpy") or "dur" not in e:
            continue
        fam = _family_of(e["name"])
        if fam in ("message_atom_fwd", "message_atom_bwd") and e["dur"] < 20.0 and "finalize" not in e["name"]:
            fam = "message_small_graphs"            # prior / contraction / bead-graph launches of the same kernels
        dur[fam] += e["dur"]
        cnt[fam] += 1
    fams = {k: v / n_steps for k, v in dur.items()}
    return fams, {k: v / n_steps for k, v in cnt.items()}, sum(fams.values())


def _timeit(fn, warm, iters):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


DUMP_SAMPLE = 1 << 22          # floats kept per buffer: 2 x 16 MB at most


def _dump_outputs(out_dir, loss, trainer):
    """loss / parameters / gradients of the step that just ran as float32 DIR/<name>.npy (see --dump-outputs).  The sample
    positions depend only on the buffer length (fixed seed), so runs of the same workload keep the same elements."""
    import numpy as np
    import torch
    params = torch.cat([p.detach().reshape(-1) for p in trainer.flat.params])
    grads = trainer.flat.flat
    idx = None
    if params.numel() > DUMP_SAMPLE:
        pick = np.random.default_rng(0).choice(params.numel(), DUMP_SAMPLE, replace=False)
        idx = torch.from_numpy(np.sort(pick)).to(params.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", loss.detach().reshape(-1)), ("parameters", params), ("gradients", grads)):
        if idx is not None and name != "loss":
            t = t[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.to(torch.float32).cpu().numpy())


def _extra_c3(dev, world, rank):
    """BASELINE config 3: chignolin sampling, n_ensemble 8 -- the prior once + 8 decoder passes per conformation as ONE CUDA
    graph replay (train.GraphedSampler); under torchrun the 8 members are sharded over the ranks and all-gathered."""
    import torch
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops, synthetic
    from coarsegrainingvae_b200.factory import build_cgvae
    from coarsegrainingvae_b200.train import GraphedSampler, sample_ensemble_sharded, to_static_batch
    cfg = dict(synthetic.CONFIGS["c2_chignolin"]); cfg["batch"] = 1
    rad = lambda xyz, c: ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=dev), c).cpu().numpy()
    torch.manual_seed(123)
    model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"], cfg["cg_cutoff"], cfg["n_cgs"]).to(dev)
    raw = [synthetic.cgvae_batch(cfg, i, rad, cg.CG_collate) for i in range(4)]
    n, ncg, n_ens = cfg["n_atoms"], cfg["n_cgs"], 8
    eps = torch.randn(n_ens, ncg, cfg["n_basis"], device=dev)
    out = {"what": "1 prior + %d decoder passes per conformation, chignolin model (35 conformations in the config; 4 cycled here)" % n_ens}
    if world == 1:
        caps = {"nbr_list": n * (n - 1) // 2, "CG_nbr_list": ncg * (ncg - 1) // 2, "bond_edge_list": max(b["bond_edge_list"].shape[0] for b in raw) + 64}
        sconfs = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in to_static_batch(b, caps).items()} for b in raw]
        sampler = GraphedSampler(model, sconfs[0], n_ens)
        it = [0]
        def step():
            sampler.sample(sconfs[it[0] % 4], eps); it[0] += 1
        ms = _timeit(step, 3, 30)
        out.update(ms_per_conformation=ms, decoder_passes_per_s=n_ens / ms * 1e3, mode="one CUDA graph per conformation, 1 GPU")
    else:
        import torch.distributed as dist
        from coarsegrainingvae_b200.train import ShardedGraphedSampler
        caps = {"nbr_list": n * (n - 1) // 2, "CG_nbr_list": ncg * (ncg - 1) // 2, "bond_edge_list": max(b["bond_edge_list"].shape[0] for b in raw) + 64}
        sconfs = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in to_static_batch(b, caps).items()} for b in raw]
        sampler = ShardedGraphedSampler(model, sconfs[0], n_ens)
        it = [0]
        def step():
            sampler.sample(sconfs[it[0] % 4], eps); it[0] += 1
        ms = _timeit(step, 3, 30)
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
        out.update(ms_per_conformation=ms, decoder_passes_per_s=n_ens / ms * 1e3,
                   mode="members sharded m %% world over %d ranks: one CUDA graph per rank and conformation (prior + %d members) + one "
                        "all_gather of [members, n_atoms, 3]" % (world, sampler.per))
    return out


def _extra_c5(dev, world, rank):
    """BASELINE config 5: one EquiMessageBlock layer on a 20 000-atom graph (message-pass edges/s) + radius-graph build."""
    import numpy as np
    import torch
    from coarsegrainingvae_b200 import ops, synthetic
    cfg = synthetic.CONFIGS["c5_large"]
    F, R, cutoff = cfg["n_basis"], cfg["n_rbf"], 8.5
    xyz = torch.as_tensor(synthetic.lattice_points(cfg["n_atoms"], cfg["spacing"], np.random.default_rng(55), rotate=False), device=dev)
    n = xyz.shape[0]
    ms_graph = _timeit(lambda: ops.radius_graph(xyz, 12.0, True), 1, 3)
    half = ops.radius_graph(xyz, cutoff, True)
    pairs = torch.cat([half, half.flip(1)], 0)
    graph = ops.build_graph(pairs, n)
    geom = ops.edge_geometry(graph, xyz, xyz, R, cutoff)
    g = torch.Generator().manual_seed(1)
    phi = torch.randn(n, 3, F, generator=g).to(dev)
    v = torch.randn(n, 3, F, generator=g).to(dev)
    s_ = torch.randn(n, F, generator=g).to(dev)
    Wf = (torch.randn(3 * F, R, generator=g) * 0.3).to(dev)
    bf = (torch.randn(3 * F, generator=g) * 0.3).to(dev)
    gs, gv = torch.randn(n, F, generator=g).to(dev), torch.randn(n, 3, F, generator=g).to(dev)
    E = graph.n_edges
    ms_f = _timeit(lambda: ops.message_fwd(3, phi, v, None, geom, Wf, bf, s_, v), 2, 5)
    ms_b = _timeit(lambda: ops.message_bwd(3, phi, v, None, None, geom, Wf, bf, gs, gv, True, sink=False), 2, 5)
    flops = 2.0 * (R + 1) * 3 * F * E
    return {"what": "one fused message layer (K=3, F=%d, R=%d) on %d atoms, cutoff %.1f A: %d directed edges; replicas only under "
                    "torchrun (no graph partitioning)" % (F, R, n, cutoff, E),
            "fwd_ms": ms_f, "bwd_ms": ms_b, "fwd_edges_per_s": E / ms_f * 1e3, "fwd_bwd_edges_per_s": E / (ms_f + ms_b) * 1e3,
            "fwd_filter_tflops": flops / ms_f * 1e-9, "bwd_filter_tflops": 2 * flops / ms_b * 1e-9,
            "radius_graph_12A_ms": ms_graph, "radius_graph_12A_pairs": int(ops.radius_graph(xyz, 12.0, True).shape[0])}


def _extra_c4(dev, world, rank):
    """BASELINE config 4: PCN (run_pdb path), ~2000-atom proteins, alpha-carbon CG; global batch 64 split over the ranks
    (strong scaling: 64 / world proteins per rank), one NCCL all-reduce of the flat gradient buffer per step."""
    import torch
    from coarsegrainingvae_b200 import ops, synthetic
    from coarsegrainingvae_b200.factory import build_pcn
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    per_rank = max(1, cfg["batch"] // world)
    rad = lambda xyz, c: ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=dev), c).cpu().numpy()
    raw = synthetic.pcn_batch(cfg, rank, rad, n_proteins=per_rank)
    torch.manual_seed(123)
    model = build_pcn(cfg["n_basis"], cfg["n_rbf"], cfg["cg_cutoff"], cfg["dec_nconv"]).to(dev)

    from coarsegrainingvae_b200.train import GraphedTrainStep, PCNTrainStep, to_static_pcn_batch
    caps = {k: int(raw[k].shape[0]) + 64 for k in ("CG_nbr_list", "bond_edge_list", "dihe_idxs", "ca_idx")}
    batch = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in to_static_pcn_batch(raw, caps).items()}
    # loss = MSE + gamma * bond-graph term + kappa * dihedral term (scripts/pcn_utils.py:160-183), skip guard on the device
    tr = PCNTrainStep(model, 1.0, 0.1, lr=1e-4, capturable=True)
    tr.prepare(batch, None)
    graphed = GraphedTrainStep(tr, batch, None)
    ms = _timeit(lambda: graphed.step(batch), 2, 4)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    out = {"what": "PCN train step (EquivariantDecoder cross_flag=True, F=%d, 9 layers), %d proteins x %d atoms per rank, global batch %d, "
                   "one CUDA graph per step (PCNTrainStep, static-capacity batch; loss = MSE + bond + 0.1 x dihedral)" % (cfg["n_basis"], per_rank, cfg["n_res"] * cfg["atoms_per_res"], per_rank * world),
           "ms_per_step": ms, "conformations_per_s": per_rank * world / ms * 1e3, "scaling": "strong (global batch 64)",
           "max_memory_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
    graphed = None
    tr.flat.release()
    return out

# --------------------------------------------------------------------------------------------- CUDA arm

def run_cuda(args, cfg):
    import numpy as np
    import torch
    import torch.distributed as dist
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops, synthetic
    from coarsegrainingvae_b200.factory import build_cgvae
    from coarsegrainingvae_b200.train import GraphedTrainStep, TrainStep, to_static_batch

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl cuda needs a CUDA device: there is no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    def gpu_radius(xyz, cutoff):
        return ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=dev), cutoff).cpu().numpy()

    # synthetic data: `pool` distinct batches per rank (different conformations on every rank: weak scaling)
    raw_batches = [synthetic.cgvae_batch(cfg, rank * 1000 + i, gpu_radius, cg.CG_collate) for i in range(args.pool)]
    edges = int(np.mean([2 * b["nbr_list"].shape[0] for b in raw_batches]))
    use_graph = not args.no_graph
    if use_graph:
        # static capacities: dense upper bounds for the radius graphs, pool maximum (+ slack) for the bond list
        B, n, ncg = cfg["batch"], cfg["n_atoms"], cfg["n_cgs"]
        caps = {"nbr_list": B * n * (n - 1) // 2, "CG_nbr_list": max(B * ncg * (ncg - 1) // 2, 1),
                "bond_edge_list": max(b["bond_edge_list"].shape[0] for b in raw_batches) + 64}
        raw_batches = [to_static_batch(b, caps) for b in raw_batches]
    host_batches = [{k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()} for b in raw_batches]
    dev_batches = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()} for b in host_batches]
    h2d_bytes = int(np.mean([sum(v.numel() * v.element_size() for v in b.values() if torch.is_tensor(v)) for b in host_batches]))

    torch.manual_seed(123)                                   # identical replicas on every rank
    model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"], cfg["cg_cutoff"],
                        cfg["n_cgs"]).to(dev)
    # the reparametrisation noise is DRAWN INSIDE the step (torch.randn_like under the graph-safe philox generator: a new
    # draw every replay, as cgvae.py:445-449 does); --fixed-eps passes one tensor instead (parity runs)
    eps = torch.randn(cfg["batch"] * cfg["n_cgs"], cfg["n_basis"], generator=torch.Generator().manual_seed(7)).to(dev) \
        if args.fixed_eps else None
    trainer = TrainStep(model, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01, capturable=use_graph)
    used = trainer.prepare(dev_batches[0], eps)
    n_used = int(trainer.flat.flat.numel())
    if use_graph:
        graphed = GraphedTrainStep(trainer, dev_batches[0], eps)
        # batches packed once (dataset-preparation time) into the byte layout of the graph's static input buffer:
        # loading a batch is ONE copy -- D2D for `value`, H2D from pinned host memory for `e2e`
        packed_dev = [graphed.pack(b, device=dev) for b in dev_batches]
        packed_host = [graphed.pack(b, pin=True) for b in host_batches]
        h2d_bytes = int(packed_host[0].numel())
        run_step = lambda i: graphed.step(packed_dev[i])
    else:
        run_step = lambda i: trainer.step(dev_batches[i], eps)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: batch resident in HBM
    for i in range(max(args.warmup, 3)):
        run_step(i % args.pool)
    sync_all()
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for i in range(args.steps):
        step_loss = run_step(i % args.pool)
    e1.record()
    sync_all()
    launches = (graphed.launches_per_step * args.steps) if use_graph else (ops.launch_count() - launches0)
    clock_info = clocks.stop()
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, step_loss, trainer)
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms = float(ms_total) / max(args.steps, 1)
    value = cfg["batch"] * n_gpus / (ms / 1e3)

    # ---- e2e: pinned host batch -> H2D -> step -> D2H loss, every step
    def e2e_step(i):
        hb = host_batches[i % args.pool]
        if use_graph:
            loss = graphed.step(packed_host[i % args.pool])  # pinned host -> static device buffer (one async H2D), then replay
        else:
            db = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in hb.items()}
            loss = trainer.step(db, eps)
        return loss.item()                                   # the reference reads loss.item() every step (utils.py:145)

    for i in range(3):
        e2e_step(i)
    sync_all()
    e0.record()
    last = 0.0
    for i in range(args.steps):
        last = e2e_step(i)
    e1.record()
    sync_all()
    ms_e = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e) / max(args.steps, 1)
    e2e_value = cfg["batch"] * n_gpus / (ms_e2e / 1e3)

    # ---- extra timed regions (same K steps each): run-to-run spread of the headline number
    reps_ms = [ms]
    for _ in range(2):
        sync_all()
        e0.record()
        for i in range(args.steps):
            run_step(i % args.pool)
        e1.record()
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        reps_ms.append(float(t) / max(args.steps, 1))

    peaks = _peaks()
    tf32_peak = 0.5 * peaks["bf16_sustained"]
    hbm_peak = peaks["hbm_gbs"]
    R, F = cfg["n_rbf"], cfg["n_basis"]

    # ---- where the step time goes: CUPTI kernel timeline of graph replays (torch.profiler), grouped into kernel families
    families, fam_launches, timeline_note = {}, {}, None
    ms_no_pdl = None
    pdl_was_on = ops.set_pdl(False)
    try:
        # Programmatic dependent launch (on in the timed runs above) makes a dependent grid resident while it still waits for
        # its predecessor, so a profiler's per-kernel durations overlap and overstate every family.  The timeline is
        # therefore taken from a SECOND capture of the same step with PDL off (its step time is reported next to it).
        timeline_step = run_step
        if use_graph and pdl_was_on and world == 1:
            graphed_tl = GraphedTrainStep(trainer, dev_batches[0], eps)
            timeline_step = lambda i: graphed_tl.step(packed_dev[i])
            for i in range(3):
                timeline_step(i % args.pool)
            sync_all()
            e0.record()
            for i in range(args.steps):
                timeline_step(i % args.pool)
            e1.record()
            sync_all()
            ms_no_pdl = e0.elapsed_time(e1) / max(args.steps, 1)
        families, fam_launches, span_us = _family_shares(lambda i: timeline_step(i % args.pool), 3)
        timeline_note = ("torch.profiler (CUPTI) over 3 %s%s; share = sum of the family's kernel durations / sum of all kernel "
                         "durations of a step (%.0f us; branches of the captured graph overlap, so the sum exceeds ms_per_step)"
                         % ("graph replays" if use_graph else "eager steps",
                            (" of a second capture WITHOUT programmatic dependent launch (%.3f ms per step; the timed runs use PDL: "
                             "weight copies of the streaming GEMMs start before the dependency wait)" % ms_no_pdl) if ms_no_pdl else "",
                            span_us))
    except Exception as exc:                        # the timeline is evidence, not a dependency of the headline number
        timeline_note = "unavailable: %r" % (exc,)
    ops.set_pdl(pdl_was_on)

    # ---- algorithmic work of one step per family: shapes recorded during ONE eager step of the same workload
    ops.TIMER = ops.KernelTimer(["gemm", "wgrad_grouped", "message_fwd", "message_bwd", "adam_clip"], keep_operands=False)
    trainer.step(dev_batches[0], eps)
    sync_all()
    rec, ops.TIMER = ops.TIMER, None
    rsum = rec.summary()
    E = float(edges)

    def gemm_family(m):
        Mr, Nr, Kr, form = m["M"], m["N"], m["K"], m["form"]
        if (form == ops.GEMM_NT and Mr <= 48) or (form == ops.GEMM_NN and Mr <= 16):
            return "gemm_stream"
        if form != ops.GEMM_TN and Mr >= 256 and Nr >= 64 and 64 <= Kr <= 1280:
            return "gemm_tcgen05"
        return "gemm_simt"

    work = {"gemm_stream": 0.0, "gemm_simt": 0.0, "gemm_tcgen05": 0.0}
    for _, m in rsum.get("gemm", []):
        fam = gemm_family(m)
        work[fam] += 4.0 * m["N"] * m["K"] if fam == "gemm_stream" else 2.0 * m["M"] * m["N"] * m["K"]
    msg_f = [m for _, m in rsum.get("message_fwd", []) if m["E"] >= edges // 2 and m["n_recv"] == m["n_send"]]
    msg_b = [m for _, m in rsum.get("message_bwd", []) if m["E"] >= edges // 2 and m["n_recv"] == m["n_send"]]
    filt = 2.0 * (R + 1) * 3 * F * E                 # filter contraction incl. the bias column per launch (SURVEY 8d)
    work["message_atom_fwd"] = filt * len(msg_f)
    work["message_atom_bwd"] = 2.0 * filt * len(msg_b)
    work["wgrad_grouped"] = 4.0 * sum(m.get("out_floats", 0) for _, m in rsum.get("wgrad_grouped", []))
    work["adam_clip"] = 32.0 * n_used
    tc_fwd = any(m.get("tc") for m in msg_f)

    MODELS = {
        "message_atom_fwd": ("tensor", "message_tc_fwd_kernel (filter on tcgen05, 3xTF32)" if tc_fwd else "message_fwd_kernel<3,%d>" % (ops.rb_for(R) // 4),
                             "filter flops 2(R+1)*3F per directed edge"),
        "message_atom_bwd": ("tensor", "message_bwd_kernel<3,%d> (fp32 SIMT)" % (ops.rb_for(R) // 4), "2x the forward filter flops"),
        "gemm_simt": ("tensor", "gemm_kernel<48,32,32,3,2> family (fp32 SIMT tiles with cluster split-K: the 36-row update-block mixes of the 12-bead decoder)", "2MNK per call"),
        "gemm_tcgen05": ("tensor", "tc::gemm_tc_kernel (tcgen05, 3xTF32: every contraction with >= 64 rows -- atom-level Dense layers, input and weight gradients)", "2MNK per call"),
        "gemm_stream": ("hbm", "gemm_nt_stream / gemm_nn_stream (12-bead Dense layers, TMA weight streaming)", "the weight matrix once per launch"),
        "wgrad_grouped": ("hbm", "wgrad_grouped_kernel (small-graph weight / bias gradients)", "gradients written once"),
        "adam_clip": ("hbm", "sumsq_partial + adam_clip_kernel", "4 (norm pass) + 28 (p, g, m, v read; p, m, v written) bytes per parameter"),
    }
    other = {}
    tot_us = sum(families.values()) or 1.0
    for fam, (bound, kernel, per_unit) in MODELS.items():
        t_us = families.get(fam)
        if not t_us or not work.get(fam):
            continue
        if bound == "tensor":
            ach, peak, unit = work[fam] / (t_us * 1e-6) / 1e12, tf32_peak, "TFLOP/s"
            src = "derived: 0.5 x bf16_tflops_sustained of %s MEASURED_PEAKS (TF32 is not measured there)" % peaks["source"]
        else:
            ach, peak, unit = work[fam] / (t_us * 1e-6) / 1e9, hbm_peak, "GB/s"
            src = "hbm_gbs of %s MEASURED_PEAKS" % peaks["source"]
        other[fam] = {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                      "traffic": NCU_DRAM_BYTES.get(fam), "algorithmic_work_per_step": work[fam], "work_model": per_unit,
                      "time_per_step_us": t_us, "launches_per_step": fam_launches.get(fam), "share_of_step": t_us / tot_us,
                      "peak_source": src}
        if fam in NCU_TRAFFIC_NOTE:
            other[fam]["traffic_source"] = ("dram__bytes_read.sum + dram__bytes_write.sum in profiles/r2_ncu_full_hot_kernels_raw.csv: "
                                            + NCU_TRAFFIC_NOTE[fam])
        if fam.startswith("message_atom"):
            n_l = max(fam_launches.get(fam) or 1, 1)
            other[fam].update(avg_launch_us=t_us / n_l, edges_per_launch=E, edges_per_s=E / (t_us / n_l * 1e-6),
                              traffic_source="dram__bytes_read.sum + dram__bytes_write.sum of this launch in " + NCU_SOURCE)
    # the roofline entry = the modelled family with the largest share of the graph-replay time
    roof = max(other.values(), key=lambda e: e["share_of_step"]) if other else None
    family_shares = {k: {"us_per_step": v, "share": v / tot_us, "launches": fam_launches.get(k)} for k, v in
                     sorted(families.items(), key=lambda kv: -kv[1])}
    # step-level HBM floor: every used parameter is read in forward and backward, its gradient written, and the optimiser
    # pass moves 32 bytes per parameter
    step_bytes = 44.0 * n_used
    hbm_floor = {"bytes_per_step": step_bytes, "floor_ms": step_bytes / (hbm_peak * 1e9) * 1e3,
                 "frac_of_floor": (step_bytes / (hbm_peak * 1e9) * 1e3) / ms,
                 "model": "used parameters x (4 fwd read + 4 bwd read + 4 gradient write + 32 clip/Adam) bytes"}

    # ---- secondary workloads of BASELINE.json (bounded; failures are reported, never fatal)
    extra = {}
    if not args.no_extra:
        graphed = None
        trainer.flat.release()
        for name, fn in (("c3_sampling", _extra_c3), ("c5_layer", _extra_c5), ("c4_protein", _extra_c4)):
            try:
                torch.cuda.empty_cache()
                extra[name] = fn(dev, world, rank)
            except Exception as exc:
                extra[name] = {"error": repr(exc)[:300]}
            sync_all()

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": _config_json(args.workload, cfg, n_gpus),
            "workload_details": {
                "directed_atom_edges_per_batch": edges, "used_gradient_floats": n_used, "used_parameters": len(used),
                "launch_mode": ("one CUDA graph per step over static-capacity input buffers (edge counts read on the device)"
                                if use_graph else "eager launches")},
            "clocks": clock_info,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "last_loss": last},
            "gpu_launches": int(launches),
            "roofline": roof, "roofline_kernels": other, "kernel_family_shares": family_shares, "timeline": timeline_note,
            "hbm_floor": hbm_floor, "ms_per_step_repeats": reps_ms, "ms_per_step_median": statistics.median(reps_ms),
            "message_pass_edges_per_s": (other.get("message_atom_fwd") or {}).get("edges_per_s"),
            "other_workloads": extra}

    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        step, kind = _cpu_step_fn(cfg, 2, threads)
        step(0)
        t0 = time.perf_counter()
        n = 0
        while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 8):
            step(n + 1)
            n += 1
        dt = (time.perf_counter() - t0) / n
        line["cpu_baseline"] = {"value": cfg["batch"] / dt, "unit": UNIT, "cores": threads, "kind": kind,
                                "sample": "%d full train steps of the same %s batch on the host CPU (%s, torch %s), after 1 "
                                          "warm-up" % (n, args.workload, "the unmodified reference from baseline/_ref"
                                                       if kind == "reference" else "oracle port of the reference", torch.__version__)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = _args()
    from coarsegrainingvae_b200 import synthetic
    cfg = dict(synthetic.CONFIGS[args.workload])
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_cuda(args, cfg)


if __name__ == "__main__":
    main()
