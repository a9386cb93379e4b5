"""The opt-in TF32 precision mode (``ops.set_matmul_precision("high")``, C ABI ``cgvae_set_matmul_precision(1)``).

"highest" (the default) runs every tensor-core contraction as 3xTF32; "high" runs the tcgen05 GEMMs and the filter of the
tensor-core message forward as 1xTF32 (operands rounded to nearest TF32, fp32 accumulation) through their own kernels
(``gemm_tc1_kernel``, ``gemm_tc1_persistent_kernel``, ``message_tc1_fwd_kernel``) with the dispatch of the default.

Stated bound per contraction with zero-mean operands: 4 * 2^-11 scale-relative (tests.golden_util.rel_err) against
float64.  Model-level gates (policy): loss 1e-3 relative, every output 1e-2 scale-relative, whole gradient 1e-2 relative L2.

Checked here: the default kernels, grids and result bits are untouched by a "high" block; every tcgen05 path and epilogue
of tests/test_gpu_dense_paths.py in "high" against float64 with the one-pass kernel confirmed by the profiler; rounding is
to nearest (a truncating pass fails the positive-operand case); kernels outside the mode give the same bits in both modes;
the message forward, the c2 step and the reduced c4 PCN step in "high"; CUDA-graph capture keeps its mode; a short training
run in both modes.  The switch itself (argument errors, context manager) is also checked without a GPU."""
import json
import math
import os
import tempfile

import numpy as np
import pytest
import torch

from coarsegrainingvae_b200 import _lib

TF32_BOUND = 4.0 * 2.0 ** -11          # stated per-contraction bound of the "high" mode
NUM_SM = 148
NAN = float("nan")
DEV = "cuda"


# ------------------------------------------------------------------------------------------ switch (no GPU needed)

def test_set_matmul_precision_abi_argument_error():
    if not os.path.exists(_lib.LIB_PATH):
        from coarsegrainingvae_b200.build import build
        build()
    lib = _lib.load()
    before = lib.cgvae_get_matmul_precision()
    rc = lib.cgvae_set_matmul_precision(7)
    assert rc < 0 and "set_matmul_precision" in _lib.last_error() and "7" in _lib.last_error()
    assert lib.cgvae_get_matmul_precision() == before == 0
    assert lib.cgvae_set_matmul_precision(1) == 0
    assert lib.cgvae_get_matmul_precision() == 1
    assert lib.cgvae_set_matmul_precision(0) == 1
    assert lib.cgvae_get_matmul_precision() == 0


def test_matmul_precision_switch_and_context_manager():
    import coarsegrainingvae_b200 as cg
    assert cg.get_matmul_precision() == "highest"
    assert cg.set_matmul_precision("high") == "highest"
    assert cg.set_matmul_precision("highest") == "high"
    for bad in ("medium", "HIGH", 1, None):
        with pytest.raises(ValueError):
            cg.set_matmul_precision(bad)
        with pytest.raises(ValueError):
            with cg.matmul_precision(bad):
                pass
    assert cg.get_matmul_precision() == "highest"
    with pytest.raises(KeyError):
        with cg.matmul_precision("high"):
            assert cg.get_matmul_precision() == "high"
            with cg.matmul_precision("highest"):
                assert cg.get_matmul_precision() == "highest"
            assert cg.get_matmul_precision() == "high"
            raise KeyError("inside the block")
    assert cg.get_matmul_precision() == "highest"
    # torch's own flag is not read
    prev = torch.get_float32_matmul_precision()
    try:
        torch.set_float32_matmul_precision("high")
        assert cg.get_matmul_precision() == "highest"
    finally:
        torch.set_float32_matmul_precision(prev)


# ------------------------------------------------------------------------------------------ GPU helpers

def _rel_err(a, b):
    assert tuple(a.shape) == tuple(b.shape), (tuple(a.shape), tuple(b.shape))
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _kernel_name(name):
    """'void cgvae::tc::gemm_tc1_kernel<true, false>(CUtensorMap_st, ...)' -> 'gemm_tc1_kernel<true, false>': namespace and
    argument list dropped, template arguments kept."""
    name = name.replace("(anonymous namespace)", "anon")
    depth = 0
    for i, ch in enumerate(name):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            name = name[:i]
            break
    name = name.strip()
    if name.startswith("void "):
        name = name[5:]
    head, sep, args = name.partition("<")
    return head.rsplit("::", 1)[-1] + sep + args


def _base(name):
    return name.split("<", 1)[0]


def _probe(fn):
    """fn() under torch.profiler with CUDA activities -> (result, [(kernel name with template arguments, grid)]) for the
    kernels of this library, in launch order.  A profile without kernel events fails."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e.get("ts", 0))
    assert kernels, "the profile holds no CUDA kernel events: the kernel that ran cannot be confirmed"
    return result, [(_kernel_name(e["name"]), tuple(e.get("args", {}).get("grid", ()))) for e in kernels
                    if "cgvae::" in e["name"]]


ONE_PASS = {"gemm_tc_kernel": "gemm_tc1_kernel", "gemm_tc_persistent_kernel": "gemm_tc1_persistent_kernel",
            "message_tc_fwd_kernel": "message_tc1_fwd_kernel"}


def _one_pass_of(launches):
    """the launches the "high" mode must make for a default-mode launch list: same kernels with the one-pass names, same
    template arguments, same grids"""
    out = []
    for name, grid in launches:
        base = _base(name)
        out.append((ONE_PASS.get(base, base) + name[len(base):], grid))
    return out


# ------------------------------------------------------------------------------------------ GEMM paths

def _gemm_setup():
    from tests import test_gpu_dense_paths as dp
    return dp


def _gemm_tf32_case(form, M, N, K, path, seed, bias=False, act=0, z_out=False, dact=None, add=False, view=False, shift=0,
                    const_pdl=False):
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops
    from tests.emulator import _act, _dact
    dp = _gemm_setup()
    gen = torch.Generator(device=DEV).manual_seed(seed)
    sa, sb = dp._shapes(form, M, N, K)
    A = dp._operand(sa, gen, 1.0, view, shift)
    B = dp._operand(sb, gen, 1.0 / math.sqrt(K), view)
    b = torch.randn(N, device=DEV, generator=gen) if bias else None
    zin = torch.randn(M, N, device=DEV, generator=gen) * 2 if dact is not None else None
    ad = torch.randn(M, N, device=DEV, generator=gen) if add else None
    v = dp._mm64(form, A, B)
    z = v + b.double() if bias else v
    y = _act(act, z)
    if zin is not None:
        y = y * _dact(dact, zin.double())
    if add:
        y = y + ad.double()
    tol = TF32_BOUND * (max(1.0, float(z.abs().max() / y.abs().max())) if (act or zin is not None) else 1.0)
    out_kind = ("rows" if z_out else "cols") if view else None

    def call(out):
        return ops.gemm(form, A, B, M, N, K, bias=b, act=act, z_out=z_out, z_in=zin, dact=dact or 0, add=ad, out=out)

    def run(mode, probe=False):
        _, C = dp._nan_out(M, N, out_kind)
        if z_out:
            dp._poison_allocator(M, N)
        with cg.matmul_precision(mode):
            if probe:
                res, launches = _probe(lambda: call(C))
            else:
                res, launches = call(C), None
        return C, (res[1].clone() if z_out else None), launches

    # the default: its kernels and bits before and after a "high" block
    C0, Z0, l0 = run("highest", probe=True)
    dp._assert_launches([(_base(n), g) for n, g in l0], dp._want(path))
    assert all(_base(n) not in ONE_PASS.values() for n, _ in l0), l0
    parent, C1 = dp._nan_out(M, N, out_kind)
    if z_out:
        dp._poison_allocator(M, N)
    with cg.matmul_precision("high"):
        res, l1 = _probe(lambda: call(C1))
    Z1 = res[1] if z_out else None
    # the one-pass kernel with the default's template arguments and grid
    assert l1 == _one_pass_of(l0), (l1, l0)
    err = _rel_err(C1, y)
    assert err <= tol, (err, tol)
    if z_out:
        ez = _rel_err(Z1, z)
        assert ez <= TF32_BOUND, ez
        err = max(err, ez)
    if view:                                                # nothing outside the output window was touched
        outside = parent.clone()
        outside[2:2 + M, (4 if out_kind == "cols" else 0):(4 if out_kind == "cols" else 0) + N] = 0.0
        assert int(torch.isnan(outside).sum()) == outside.numel() - M * N
    C2, Z2, _ = run("high")                                 # repeatable
    assert torch.equal(C2, C1) and (not z_out or torch.equal(Z2, Z1))
    C3, Z3, l3 = run("highest", probe=True)                 # default untouched
    assert l3 == l0 and torch.equal(C3, C0) and (not z_out or torch.equal(Z3, Z0))
    if const_pdl:
        # weight prefetch before the PDL dependency wait (b_const branch of the one-pass kernel), then PDL off
        prev = ops.set_pdl(True)
        try:
            ops.register_const_range(B)
            with cg.matmul_precision("high"):
                _, C4 = dp._nan_out(M, N, out_kind)
                _, l4 = _probe(lambda: call(C4))
                ops.set_pdl(False)
                _, C5 = dp._nan_out(M, N, out_kind)
                call(C5)
        finally:
            ops.register_const_range(None)
            ops.set_pdl(prev)
        assert l4 == l1 and torch.equal(C4, C1) and torch.equal(C5, C1)
    # the 3xTF32 result stays well inside the TF32 bound too: the two modes differ by TF32 rounding only
    print("TF32 %s %dx%d<-%d %s: rel err %.2e (bound %.2e), default %.2e"
          % ("NT NN TN".split()[form], M, N, K, path[0], err, tol, _rel_err(C0, y)))
    return err


def _tc_cases():
    dp = _gemm_setup()
    return [c for c in dp.GEMM_CASES if c[5][0] in ("persistent", "cluster", "grouped")]


TC_CASES = _tc_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("case", TC_CASES, ids=[c[0] for c in TC_CASES])
def test_tf32_gemm_path_vs_float64(case):
    name, form, M, N, K, path, kw = case
    _gemm_tf32_case(form, M, N, K, path, seed=(M * 31 + N * 7 + K) % 100003, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("form,M,N,K,path", [
    (0, 256, 256, 16000, ("cluster", 8)),            # NT, 63 k-steps per CTA
    (2, 2048, 512, 16000, ("cluster", 6)),           # TN (MN-major operands)
    (1, 16000, 512, 1024, ("persistent",)),          # NN, persistent kernel
])
def test_tf32_rounds_to_nearest(form, M, N, K, path):
    """positive operands uniform in [0.5, 1): every product has the same sign, so a truncating operand pass (what the tensor
    core does to raw fp32) leaves a one-sided error of ~2^-11 x 1.5 (~7e-4) that does not average out; round to nearest
    leaves ~2e-5 at K = 16 000 (calculated, not measured).  Gate 1e-4."""
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops
    dp = _gemm_setup()
    gen = torch.Generator(device=DEV).manual_seed(K + M)
    sa, sb = dp._shapes(form, M, N, K)
    A = torch.rand(*sa, device=DEV, generator=gen) * 0.5 + 0.5
    B = torch.rand(*sb, device=DEV, generator=gen) * 0.5 + 0.5
    with cg.matmul_precision("high"):
        C, launches = _probe(lambda: ops.gemm(form, A, B, M, N, K))
    want = [(ONE_PASS[n], axes) for n, axes in dp._want(path)]
    dp._assert_launches([(_base(n), g) for n, g in launches], want)
    err = _rel_err(C, dp._mm64(form, A, B))
    print("TF32 positive operands %s %dx%d<-%d: rel err %.2e" % ("NT NN TN".split()[form], M, N, K, err))
    assert err <= 1e-4, err


# ------------------------------------------------------------------------------------------ what the mode does not touch

def _both_modes(fn):
    import coarsegrainingvae_b200 as cg
    with cg.matmul_precision("highest"):
        a, la = _probe(fn)
    with cg.matmul_precision("high"):
        b, lb = _probe(fn)
    assert la == lb, (la, lb)
    assert all(_base(n) not in ONE_PASS and _base(n) not in ONE_PASS.values() for n, _ in la), la
    return a, b, la


@pytest.mark.gpu
@pytest.mark.parametrize("form,M,N,K,kind,kw", [
    (2, 2048, 2048, 50000, "gemm_kernel", dict()),             # SIMT: grouped partials beyond the workspace
    (0, 2000, 600, 598, "gemm_kernel", dict()),                 # SIMT: ld % 4 != 0
    (0, 36, 600, 600, None, dict(bias=True)),                   # weight streaming NT (decoder graphs)
    (1, 12, 600, 600, None, dict()),                            # weight streaming NN
])
def test_mode_does_not_touch_fp32_gemms(form, M, N, K, kind, kw):
    from coarsegrainingvae_b200 import ops
    dp = _gemm_setup()
    gen = torch.Generator(device=DEV).manual_seed(M + N + K)
    sa, sb = dp._shapes(form, M, N, K)
    A = torch.randn(*sa, device=DEV, generator=gen)
    B = torch.randn(*sb, device=DEV, generator=gen) / math.sqrt(K)
    bias = torch.randn(N, device=DEV, generator=gen) if kw.get("bias") else None
    a, b, launches = _both_modes(lambda: ops.gemm(form, A, B, M, N, K, bias=bias))
    if kind is not None:
        assert kind in [_base(n) for n, _ in launches], launches
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_mode_does_not_touch_colsum_and_wgrad_grouped():
    from coarsegrainingvae_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(3)
    X = torch.randn(48000, 512, device=DEV, generator=gen)
    a, b, launches = _both_modes(lambda: ops.colsum(X))
    assert "colsum_tall_kernel" in [_base(n) for n, _ in launches]
    assert torch.equal(a, b)
    gy = torch.randn(350, 600, device=DEV, generator=gen)
    x = torch.randn(350, 600, device=DEV, generator=gen)

    def wg():
        dW, db = torch.empty(600, 600, device=DEV), torch.empty(600, device=DEV)
        ops.wgrad_grouped([(gy, x, dW, db)])
        return dW, db
    (a1, a2), (b1, b2), launches = _both_modes(wg)
    assert "wgrad_grouped_kernel" in [_base(n) for n, _ in launches]
    assert torch.equal(a1, b1) and torch.equal(a2, b2)


# ------------------------------------------------------------------------------------------ message layer

def _message_case(n_split, n, F, R, cutoff, seed):
    from coarsegrainingvae_b200 import ops, synthetic
    g = torch.Generator().manual_seed(seed)
    xyz = synthetic.lattice_points(n, 2.2, np.random.default_rng(seed), rotate=False)
    half = ops.radius_graph(torch.as_tensor(xyz, device=DEV), cutoff, True)
    graph = ops.build_graph(torch.cat([half, half.flip(1)], 0), n)
    x = torch.as_tensor(xyz, device=DEV)
    geom = ops.edge_geometry(graph, x, x, R, cutoff)
    phi = torch.randn(n, n_split, F, generator=g).to(DEV)
    v = torch.randn(n, 3, F, generator=g).to(DEV)
    Wf = (torch.randn(n_split * F, R, generator=g) * 0.5).to(DEV)
    bf = (torch.randn(n_split * F, generator=g) * 0.5).to(DEV)
    res_s = torch.randn(n, F, generator=g).to(DEV)
    res_v = torch.randn(n, 3, F, generator=g).to(DEV)
    return graph, geom, phi, v, Wf, bf, res_s, res_v


def _message_truth(n_split, graph, geom, phi, v, Wf, bf, res_s, res_v):
    """float64 layer from the same per-edge records (basis, unit): conv.py:505-563 / 358-402"""
    n, F, R = graph.n_recv, phi.shape[-1], Wf.shape[1]
    col = graph.col.long()
    recv = torch.repeat_interleave(torch.arange(n, device=DEV), (graph.rowptr[1:] - graph.rowptr[:-1]).long())
    E = int(graph.rowptr[-1])
    col, recv = col[:E], recv[:E]
    Wfull = torch.zeros(n_split * F, geom.rb, dtype=torch.float64, device=DEV)
    Wfull[:, :R] = Wf.double()
    Wfull[:, R] = bf.double()
    w = (geom.basis[:E].double() @ Wfull.t()).view(E, n_split, F)
    m = phi.double()[col] * w
    u = geom.unit[:E, :3].double()
    ds = torch.zeros(n, F, dtype=torch.float64, device=DEV).index_add_(0, recv, m[:, 1])
    dv_e = m[:, 2, None, :] * u[:, :, None] + m[:, 0, None, :] * v.double()[col]
    if n_split == 4:
        dv_e = dv_e + m[:, 3, None, :] * torch.linalg.cross(v.double()[recv], v.double()[col], dim=1)
    dv = torch.zeros(n, 3, F, dtype=torch.float64, device=DEV).index_add_(0, recv, dv_e)
    return ds + res_s.double(), dv + res_v.double()


@pytest.mark.gpu
@pytest.mark.parametrize("n_split,n,F,R,cutoff", [
    (3, 350, 600, 10, 12.0),          # c2 atom graph: 2 x 175 atoms, F = 600, 10 radial functions
    (4, 2000, 512, 8, 7.0),           # cross block at the PCN width, 2 000 beads
], ids=["c2_atom_k3", "cross_k4_2000"])
def test_message_forward_tf32_vs_float64(n_split, n, F, R, cutoff):
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import ops
    graph, geom, phi, v, Wf, bf, res_s, res_v = _message_case(n_split, n, F, R, cutoff, seed=5 + n_split)
    ds, dv = _message_truth(n_split, graph, geom, phi, v, Wf, bf, res_s, res_v)
    vr = v if n_split == 4 else None
    old = ops.MSG_TC
    try:
        ops.MSG_TC = "1"
        fwd = lambda: ops.message_fwd(n_split, phi, v, vr, geom, Wf, bf, res_s, res_v, want_q=n_split == 4)  # noqa: E731
        fwd()                                   # builds the column tiles of the graph once (cached on geom)
        with cg.matmul_precision("highest"):
            d0, l0 = _probe(fwd)
        with cg.matmul_precision("high"):
            h1, l1 = _probe(fwd)
            h2 = fwd()
        with cg.matmul_precision("highest"):
            d1, l2 = _probe(fwd)
    finally:
        ops.MSG_TC = old
    assert [_base(k) for k, _ in l0 if _base(k).startswith("message")] == ["message_tc_fwd_kernel"], l0
    assert l1 == _one_pass_of(l0) and l2 == l0, (l0, l1, l2)
    assert all(torch.equal(a, b) for a, b in zip(d0[:2], d1[:2]))          # default untouched
    assert all(torch.equal(a, b) for a, b in zip(h1[:2], h2[:2]))          # repeatable
    es, ev = _rel_err(h1[0], ds), _rel_err(h1[1], dv)
    print("TF32 message forward K=%d n=%d: s %.2e v %.2e (default %.2e %.2e)"
          % (n_split, n, es, ev, _rel_err(d0[0], ds), _rel_err(d0[1], dv)))
    assert es <= TF32_BOUND and ev <= TF32_BOUND, (es, ev)


@pytest.mark.gpu
@pytest.mark.parametrize("n_split", [3, 4])
def test_mode_does_not_touch_message_backward(n_split):
    from coarsegrainingvae_b200 import ops
    graph, geom, phi, v, Wf, bf, _, _ = _message_case(n_split, 350, 256, 8, 9.0, seed=21 + n_split)
    g = torch.Generator().manual_seed(2)
    gs = torch.randn(350, 256, generator=g).to(DEV)
    gv = torch.randn(350, 3, 256, generator=g).to(DEV)
    q = None
    if n_split == 4:
        q = ops.message_fwd(4, phi, v, v, geom, Wf, bf, None, None, want_q=True)[2]
    a, b, launches = _both_modes(lambda: ops.message_bwd(n_split, phi, v, v if n_split == 4 else None, q, geom, Wf, bf, gs, gv,
                                                         True, sink=False))
    assert launches
    assert all(torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------ model level

LOSS_GATE, OUT_GATE, GRAD_GATE = 1e-3, 1e-2, 1e-2


def _grad_l2(model, P64):
    num = den = 0.0
    for k, p in model.named_parameters():
        truth = P64[k].grad
        if truth is None:
            continue
        got = p.grad.detach().cpu().double() if p.grad is not None else torch.zeros_like(truth)
        num += float((got - truth).pow(2).sum())
        den += float(truth.pow(2).sum())
    return (num / den) ** 0.5


def _gpu_radius(xyz, cutoff):
    from coarsegrainingvae_b200 import ops
    return ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=DEV), cutoff).cpu().numpy()


def _to(batch, dev):
    return {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in batch.items()}


@pytest.mark.gpu
def test_c2_step_tf32_vs_float64_oracle():
    """the c2 (chignolin, F = 600) train step of test_cgvae_step_at_config_width under "high" against the float64 oracle"""
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import synthetic
    from oracle import cgvae_oracle as orc
    from tests import parity_cases as pc
    from tests.golden_util import rel_err
    cfg = dict(synthetic.CONFIGS["c2_chignolin"])
    n_conf = cfg["batch"] = 2
    batch = synthetic.cgvae_batch(cfg, 0, _gpu_radius, cg.CG_collate)
    torch.manual_seed(123)
    model = pc.build_vae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"],
                         cfg["cg_cutoff"], cfg["n_cgs"] == 3, cfg["n_cgs"]).to(DEV)
    eps = torch.randn(n_conf * cfg["n_cgs"], cfg["n_basis"], generator=torch.Generator().manual_seed(7))
    P = pc._oracle_params(model)
    with cg.matmul_precision("high"):
        out = model(_to(batch, DEV), eps=eps.to(DEV))
        loss = orc.training_loss(out, _to(batch, DEV), cfg["beta"], cfg["gamma"])[0]
        loss.backward()
        torch.cuda.synchronize()
    spec = dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], enc_nconv=cfg["enc_nconv"], dec_nconv=cfg["dec_nconv"],
                atom_cutoff=cfg["atom_cutoff"], cg_cutoff=cfg["cg_cutoff"], decoder="pseudo", breaksym=cfg["n_cgs"] == 3,
                activation="swish")
    P64 = {k: v.detach().double().requires_grad_(v.dtype.is_floating_point) for k, v in P.items()}
    b64 = {k: (v.double() if torch.is_tensor(v) and v.dtype.is_floating_point else v) for k, v in batch.items()}
    o64 = orc.cgvae_forward(P64, spec, b64, eps=eps.double())
    l64 = orc.training_loss(o64, b64, cfg["beta"], cfg["gamma"])[0]
    l64.backward()
    e_out = {k: rel_err(a, b) for a, b, k in zip(out, o64, ("mu", "sigma", "pmu", "pstd", "xyz", "xyz_recon"))}
    e_loss, e_grad = rel_err(loss, l64), _grad_l2(model, P64)
    print("TF32 c2 step: loss %.2e, worst output %.2e (%s), gradient L2 %.2e"
          % (e_loss, max(e_out.values()), max(e_out, key=e_out.get), e_grad))
    assert e_loss <= LOSS_GATE and max(e_out.values()) <= OUT_GATE and e_grad <= GRAD_GATE, (e_loss, e_out, e_grad)


@pytest.mark.gpu
def test_pcn_reduced_step_tf32_vs_float64_oracle():
    """the reduced c4 PCN step (F = 512, 9 cross layers, 2 proteins x 60 residues) under "high" against the float64 oracle"""
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import synthetic
    from oracle import cgvae_oracle as orc
    from tests import parity_cases as pc
    from tests.golden_util import rel_err
    cfg = dict(synthetic.CONFIGS["c4_protein"])
    cfg["n_res"] = 60
    batch = synthetic.pcn_batch(cfg, 0, _gpu_radius, n_proteins=2)
    torch.manual_seed(123)
    net = cg.EquivariantDecoder(n_atom_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], cutoff=cfg["cg_cutoff"],
                                num_conv=cfg["dec_nconv"], activation="swish", cross_flag=True)
    model = cg.PCN(net, feature_dim=cfg["n_basis"], offset=False).to(DEV)
    P = pc._oracle_params(model)
    with cg.matmul_precision("high"):
        out = model(_to(batch, DEV))
        loss = (out[5] - out[4]).pow(2).mean()
        loss.backward()
        torch.cuda.synchronize()
    spec = dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], dec_nconv=cfg["dec_nconv"], atom_cutoff=cfg["cg_cutoff"],
                decoder="cross", activation="swish")
    P64 = {k: v.detach().double().requires_grad_(v.dtype.is_floating_point) for k, v in P.items()}
    b64 = {k: (v.double() if torch.is_tensor(v) and v.dtype.is_floating_point else v) for k, v in batch.items()}
    o64 = orc.pcn_forward(P64, spec, b64)
    l64 = (o64[5] - o64[4]).pow(2).mean()
    l64.backward()
    e_out, e_loss, e_grad = rel_err(out[5], o64[5]), rel_err(loss, l64), _grad_l2(model, P64)
    print("TF32 reduced c4 PCN step: loss %.2e, output %.2e, gradient L2 %.2e" % (e_loss, e_out, e_grad))
    assert e_loss <= LOSS_GATE and e_out <= OUT_GATE and e_grad <= GRAD_GATE, (e_loss, e_out, e_grad)


# ------------------------------------------------------------------------------------------ graphs and training

def _c1_setup(n_batches, caps_slack=8):
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200 import synthetic
    from coarsegrainingvae_b200.train import to_static_batch
    cfg = dict(synthetic.CONFIGS["c1_dipeptide"])
    cfg["batch"] = 4
    raw = [synthetic.cgvae_batch(cfg, i, _gpu_radius, cg.CG_collate) for i in range(n_batches)]
    B, n, ncg = cfg["batch"], cfg["n_atoms"], cfg["n_cgs"]
    caps = {"nbr_list": B * n * (n - 1) // 2, "CG_nbr_list": max(B * ncg * (ncg - 1) // 2, 1),
            "bond_edge_list": max(b["bond_edge_list"].shape[0] for b in raw) + caps_slack}
    return cfg, [_to(to_static_batch(b, caps), DEV) for b in raw]


def _c1_model(cfg):
    from coarsegrainingvae_b200.factory import build_cgvae
    torch.manual_seed(123)
    return build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"], cfg["cg_cutoff"],
                       cfg["n_cgs"]).to(DEV)


@pytest.mark.gpu
def test_graph_captured_in_high_mode_keeps_it():
    """a GraphedTrainStep captured under "high" replays bit for bit what the same steps give eagerly under "high", and keeps
    running the one-pass kernels after the global mode is back to "highest"."""
    import copy
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200.train import GraphedTrainStep, TrainStep
    cfg, static = _c1_setup(3)
    model_a = _c1_model(cfg)
    model_b = copy.deepcopy(model_a)
    eps = torch.randn(cfg["batch"] * cfg["n_cgs"], cfg["n_basis"], generator=torch.Generator().manual_seed(7)).to(DEV)
    eager = TrainStep(model_a, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01, capturable=True)
    eager.prepare(static[0], eps)
    graph_tr = TrainStep(model_b, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01, capturable=True)
    graph_tr.prepare(static[0], eps)
    with cg.matmul_precision("high"):
        graphed = GraphedTrainStep(graph_tr, static[0], eps)   # three eager warm-up steps, then the capture
        for _ in range(3):
            eager.step(static[0], eps)
        assert graphed.matmul_precision == "high"
        losses_a = [float(eager.step(static[i], eps)) for i in (1, 2)]
    assert cg.get_matmul_precision() == "highest"
    losses_b = [float(graphed.step(static[1]))]
    _, launches = _probe(lambda: graphed.step(static[2]))
    losses_b.append(float(graphed.loss))
    names = [_base(n) for n, _ in launches]
    assert "gemm_tc1_kernel" in names and "gemm_tc_kernel" not in names and "gemm_tc_persistent_kernel" not in names, names
    assert graphed.matmul_precision == "high"
    assert losses_a == losses_b, (losses_a, losses_b)
    for (k, pa), (_, pb) in zip(model_a.named_parameters(), model_b.named_parameters()):
        assert torch.equal(pa, pb), k
    graph_tr.flat.release()
    eager.flat.release()


@pytest.mark.gpu
def test_training_in_both_modes_tracks():
    """20 graphed c1 steps (batch 4) in each mode from the same weights and batches: both losses fall, and the per-step
    relative loss difference stays within 1e-2 (policy)."""
    import coarsegrainingvae_b200 as cg
    from coarsegrainingvae_b200.train import GraphedTrainStep, TrainStep
    cfg, static = _c1_setup(4)
    eps = torch.randn(cfg["batch"] * cfg["n_cgs"], cfg["n_basis"], generator=torch.Generator().manual_seed(7)).to(DEV)
    curves = {}
    for mode in ("highest", "high"):
        model = _c1_model(cfg)
        tr = TrainStep(model, cfg["beta"], cfg["gamma"], lr=1e-4, max_norm=0.01, capturable=True)   # the bench.py settings
        tr.prepare(static[0], eps)
        with cg.matmul_precision(mode):
            graphed = GraphedTrainStep(tr, static[0], eps)
        curves[mode] = [float(graphed.step(static[i % len(static)])) for i in range(20)]
        graphed = None
        tr.flat.release()
    a, b = np.array(curves["highest"]), np.array(curves["high"])
    diff = np.abs(b - a) / np.abs(a)
    print("c1 training, 20 steps: highest %.4f -> %.4f, high %.4f -> %.4f, worst relative loss difference %.2e"
          % (a[0], a[-1], b[0], b[-1], diff.max()))
    assert a[-4:].mean() < a[:4].mean() and b[-4:].mean() < b[:4].mean(), (a, b)
    assert diff.max() <= 1e-2, diff
