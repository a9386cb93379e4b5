"""GPU (B200): every branch of the dense-contraction dispatcher that the PCN protein step (c4: F = 512, 16 000 beads,
48 000 planar vector rows) runs, against float64 torch on the device, with the kernel that ran confirmed by the profiler.

The dispatcher is ``cgvae_gemm`` / ``cgvae_colsum`` (csrc/gemm.cu), ``launch_gemm_tcgen05`` (csrc/gemm_tc.cu) and
``launch_gemm_stream`` (csrc/gemm_stream.cu).  Paths are chosen by shape and alignment alone, so every case names the kernel
and grid (and for the decoder-sized shapes the block) its shape must reach, and ``_probe`` checks them in the CUDA trace:

  * persistent tcgen05 kernel: >= 296 output tiles, K <= 1280, grid.x = 148;
  * one-CTA-per-tile tcgen05 kernel, K split over a cluster of S CTAs (grid.z = S); S = 1 for long K-loops on many tiles;
  * grouped split-K: reductions over more than 8 x 96 k-steps, grid.z = 8 x groups, then splitk_reduce_kernel adds the
    group partials in order and applies the epilogue;
  * the SIMT gemm_kernel for what TMA cannot take (misaligned bases, ld % 4 != 0) and for group partials that do not
    fit the 32 MB split-K workspace (one unsplit fp32 chain over K);
  * below 64 rows (decoder graphs: 12 beads, 36 vector rows): the TMA weight-streaming kernels (NT up to 48 rows, NN up to
    16, cgvae_dense_pair_fwd), the column-per-thread gemm_skinny_kernel (NT, <= 16 rows, N >= 1024, where the streaming
    kernel declines), SIMT cluster split-K (grid.z = S) and SIMT workspace split-K + splitk_reduce_kernel (TN);
  * colsum_tall_kernel from 4096 rows, rows split over a cluster of S = 8 / 4 / 1 CTAs (grid.y);
  * the rank-segmented grouped weight gradient (data-parallel factor exchange);
  * the message-layer forward: message_fwd_kernel (SIMT) and message_tc_fwd_kernel (tensor cores, RC = 8).

Every output is pre-filled with NaN (an element nobody writes fails), every case runs twice and must be bitwise repeatable.
Metric: tests.golden_util.rel_err (max|a - b| / max|b|), evaluated on the device."""
import json
import math
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import coarsegrainingvae_b200 as cg
from coarsegrainingvae_b200 import ops, synthetic
from oracle import cgvae_oracle as orc
from tests import parity_cases as pc
from tests.emulator import _act, _dact

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
NT, NN, TN = ops.GEMM_NT, ops.GEMM_NN, ops.GEMM_TN
NUM_SM = 148
NAN = float("nan")


def _rel_err(a, b):
    """tests.golden_util.rel_err computed on the device (the operands here reach 10^8 elements)."""
    assert tuple(a.shape) == tuple(b.shape), (tuple(a.shape), tuple(b.shape))
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


# ------------------------------------------------------------------------------------------ path probe

def _base_name(name):
    """'void cgvae::tc::gemm_tc_kernel<true, false>(CUtensorMap_st, ...)' -> 'gemm_tc_kernel'"""
    name = name.replace("(anonymous namespace)", "anon")
    head = re.split(r"[<(]", name, maxsplit=1)[0].strip()
    return head.split()[-1].rsplit("::", 1)[-1]


def _probe(fn):
    """run fn() under torch.profiler with CUDA activities; returns (fn's result, [(kernel base name, grid, block)]) for
    the kernels of this library (namespace cgvae), in launch order -- torch's own kernels (tensor set-up, a launch still
    draining when the profile starts) are left out.  A profile without kernel events fails: a path check that cannot see
    the kernels proves nothing."""
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
    assert kernels, "the profile holds no CUDA kernel events: the kernel this case must reach cannot be confirmed"
    return result, [(_base_name(e["name"]), tuple(e.get("args", {}).get("grid", ())), tuple(e.get("args", {}).get("block", ())))
                    for e in kernels if "cgvae::" in e["name"]]


# expected launches per path: [(kernel, {grid axis: extent}[, block.x])]
def _want(path):
    kind = path[0]
    if kind == "persistent":
        return [("gemm_tc_persistent_kernel", {0: NUM_SM})]
    if kind == "cluster":                                   # ("cluster", S): one tcgen05 launch, S K-slices per tile
        return [("gemm_tc_kernel", {2: path[1]})]
    if kind == "grouped":                                   # ("grouped", groups): clusters of 8 + the ordered reduction
        return [("gemm_tc_kernel", {2: 8 * path[1]}), ("splitk_reduce_kernel", {})]
    if kind == "simt":
        return [("gemm_kernel", {2: 1})]
    # (kind, grid, block): the whole launch shape is pinned
    grid = dict(enumerate(path[1]))
    if kind == "simt_cluster":                              # K split over a cluster of grid.z CTAs, reduced through DSMEM
        return [("gemm_kernel", grid, path[2])]
    if kind == "simt_splitk":                               # grid.z partial matrices, added in order by the reduce kernel
        return [("gemm_kernel", grid, path[2]), ("splitk_reduce_kernel", {})]
    if kind in ("gemm_skinny_kernel", "gemm_nt_stream_kernel", "gemm_nn_stream_kernel"):
        return [(kind, grid, path[2])]
    raise ValueError(path)


def _assert_launches(launches, want):
    """launches: [(name, grid[, block])]; want: [(name, {grid axis: extent}[, block.x])]"""
    assert [k[0] for k in launches] == [w[0] for w in want], (launches, want)
    for (name, grid, *block), (_, axes, *blk) in zip(launches, want):
        for axis, extent in axes.items():
            assert grid[axis] == extent, (name, grid, axes)
        if blk:
            assert block[0][0] == blk[0], (name, block, blk)


# ------------------------------------------------------------------------------------------ GEMM cases

def _mm64(form, A, B):
    A, B = A.double(), B.double()
    return {NT: lambda: A @ B.t(), NN: lambda: A @ B, TN: lambda: A.t() @ B}[form]()


def _shapes(form, M, N, K):
    return {NT: ((M, K), (N, K)), NN: ((M, K), (K, N)), TN: ((K, M), (K, N))}[form]


def _operand(shape, gen, scale, view, shift=0):
    """randn(shape) * scale; view: a column window [4, 4 + cols) of a NaN-filled buffer 8 columns wider (row pitch % 4 == 0,
    16-byte aligned base) -- the tensor maps must use the logical extent, not the pitch; shift: base moved by one float."""
    rows, cols = shape
    x = torch.randn(rows, cols, device=DEV, generator=gen) * scale
    if view:
        buf = torch.full((rows, cols + 8), NAN, device=DEV)
        buf[:, 4:4 + cols] = x
        return buf[:, 4:4 + cols]
    if shift:
        buf = torch.full((rows * cols + shift,), NAN, device=DEV)
        buf[shift:] = x.reshape(-1)
        return buf[shift:].view(rows, cols)
    return x


def _nan_out(M, N, kind):
    """(parent, C): C pre-filled with NaN; 'cols' = C is a window of a NaN parent with a wider row pitch, 'rows' = a row
    window (row pitch N, as a z_out call needs)."""
    if kind == "cols":
        parent = torch.full((M + 4, N + 12), NAN, device=DEV)
        return parent, parent[2:2 + M, 4:4 + N]
    if kind == "rows":
        parent = torch.full((M + 4, N), NAN, device=DEV)
        return parent, parent[2:2 + M]
    out = torch.full((M, N), NAN, device=DEV)
    return out, out


def _poison_allocator(M, N, *shapes):
    """hand the caching allocator NaN blocks of the pre-activation's size (and of `shapes`): a z_out the kernel does not
    write reads NaN."""
    t = [torch.full(s, NAN, device=DEV) for s in ((M, N),) + shapes]
    del t


def _gemm_case(form, M, N, K, path, seed, bias=False, act=0, z_out=False, dact=None, add=False, view=False, shift=0,
               const_pdl=False):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    sa, sb = _shapes(form, M, N, K)
    scale_b = 1.0 / math.sqrt(K)
    A = _operand(sa, gen, 1.0, view, shift)
    B = _operand(sb, gen, scale_b, view)
    b = torch.randn(N, device=DEV, generator=gen) if bias else None
    zin = torch.randn(M, N, device=DEV, generator=gen) * 2 if dact is not None else None
    ad = torch.randn(M, N, device=DEV, generator=gen) if add else None
    # float64 ground truth, epilogue in the kernels' order: + bias, (z_out), act, * act'(z_in), + add
    v = _mm64(form, A, B)
    z = v + b.double() if bias else v
    y = _act(act, z)
    if zin is not None:
        y = y * _dact(dact, zin.double())
    if add:
        y = y + ad.double()
    # activation outputs: the error budget is set by the pre-activation scale (as in test_gemm_forms_and_epilogues)
    tol = TOL * (max(1.0, float(z.abs().max() / y.abs().max())) if (act or zin is not None) else 1.0)
    out_kind = ("rows" if z_out else "cols") if view else None
    assert not (view and (zin is not None or add)), "aux operands share the output's row pitch"

    def call(out):
        return ops.gemm(form, A, B, M, N, K, bias=b, act=act, z_out=z_out, z_in=zin, dact=dact or 0, add=ad, out=out)

    parent, C = _nan_out(M, N, out_kind)
    if z_out:
        _poison_allocator(M, N)
    res, launches = _probe(lambda: call(C))
    _assert_launches(launches, _want(path))
    Z = res[1] if z_out else None
    err = _rel_err(C, y)
    assert err < tol, (err, tol)
    if z_out:                                               # first call of this shape: Z is freshly written
        ez = _rel_err(Z, z)
        assert ez < TOL, ez
        err = max(err, ez)
    if view:                                                # nothing outside the output window was touched
        outside = parent.clone()
        outside[2:2 + M, (4 if out_kind == "cols" else 0):(4 if out_kind == "cols" else 0) + N] = 0.0
        assert int(torch.isnan(outside).sum()) == outside.numel() - M * N
    # deterministic: a second call is bitwise identical
    parent2, C2 = _nan_out(M, N, out_kind)
    res2 = call(C2)
    assert torch.equal(C2, C)
    if z_out:
        assert torch.equal(res2[1], Z)
    if const_pdl:
        # B inside a registered constant range with PDL on: the producer prefetches B before the dependency wait
        # (gemm_tc_kernel's b_const branch); then PDL off.  Both bitwise equal to the plain run.
        prev = ops.set_pdl(True)
        try:
            ops.register_const_range(B)
            parent3, C3 = _nan_out(M, N, out_kind)
            _, launches3 = _probe(lambda: call(C3))
            _assert_launches(launches3, _want(path))
            ops.set_pdl(False)
            parent4, C4 = _nan_out(M, N, out_kind)
            call(C4)
        finally:
            ops.register_const_range(None)
            ops.set_pdl(prev)
        assert torch.equal(C3, C) and torch.equal(C4, C)
    print("%s %dx%d<-%d %s: rel err %.2e (tol %.1e)" % ("NT NN TN".split()[form], M, N, K, path[0], err, tol))
    return err


P, S1 = ("persistent",), ("cluster", 1)
GEMM_CASES = [
    # ---- persistent kernel (>= 296 tiles, K <= 1280): epilogue modes 0, 1, 2, 3, 4, 5, 6 and the TN form
    ("p_nt_phi_fwd_bias", NT, 16000, 2048, 512, P, dict(bias=True)),                        # mode 1
    ("p_nt_bias_swish_zout", NT, 16000, 512, 1024, P, dict(bias=True, act=1, z_out=True)),  # mode 6
    ("p_nt_bias_swish", NT, 16000, 512, 512, P, dict(bias=True, act=1)),                    # mode 2
    ("p_nt_plain", NT, 48000, 512, 512, P, dict()),                                         # mode 0
    ("p_nt_bias_relu_view", NT, 15997, 1800, 600, P, dict(bias=True, act=2, view=True)),    # mode 3, strided views
    ("p_nt_bias_tanh", NT, 15997, 1800, 600, P, dict(bias=True, act=3)),
    ("p_nt_bias_sigmoid", NT, 15997, 1800, 600, P, dict(bias=True, act=4)),
    ("p_nt_bias_ssp", NT, 15997, 1800, 600, P, dict(bias=True, act=5)),
    ("p_nt_bias_leaky", NT, 15997, 1800, 600, P, dict(bias=True, act=6)),
    ("p_nt_bias_elu", NT, 15997, 1800, 600, P, dict(bias=True, act=7)),
    ("p_nt_bias_relu_zout", NT, 15997, 1800, 600, P, dict(bias=True, act=2, z_out=True)),
    ("p_nn_uv_input_grad_add", NN, 48000, 512, 1024, P, dict(add=True)),                    # mode 5
    ("p_nn_plain", NN, 16000, 512, 512, P, dict()),                                         # mode 0
    ("p_nn_dswish", NN, 16000, 512, 512, P, dict(dact=1)),                                  # mode 4
    ("p_nn_dtanh", NN, 16000, 512, 512, P, dict(dact=3)),                                   # mode 3
    ("p_nn_dswish_add", NN, 16000, 512, 512, P, dict(dact=1, add=True)),                    # mode 3
    ("p_tn_plain", TN, 2560, 2048, 1000, P, dict()),
    ("p_tn_bias", TN, 2560, 2048, 1000, P, dict(bias=True)),
    # ---- one tile per CTA, S = 1
    ("s1_nn_phi_bwd_dswish", NN, 16000, 512, 2048, S1, dict(dact=1)),                       # 64 k-steps > 40
    ("s1_nt_bias_const_pdl", NT, 2000, 1800, 600, S1, dict(bias=True, const_pdl=True)),
    ("s1_nt_bias_swish", NT, 2000, 1800, 600, S1, dict(bias=True, act=1)),
    ("s1_nt_1kstep", NT, 128, 256, 32, S1, dict()),
    ("s1_nt_2ksteps", NT, 128, 256, 36, S1, dict()),
    ("s1_nt_3ksteps", NT, 128, 256, 96, S1, dict()),
    # ---- cluster split-K, S = 2 .. 8 (cluster_reduce_rows row slices 64, 32, 26, 22, 19, 16)
    ("c6_tn_phi_w1_grad", TN, 2048, 512, 16000, ("cluster", 6), dict()),
    ("c8_tn", TN, 512, 512, 16000, ("cluster", 8), dict()),
    ("c6_tn_s_dense1_grad", TN, 1536, 512, 16000, ("cluster", 6), dict()),
    ("c5_nt_bias_view", NT, 640, 640, 600, ("cluster", 5), dict(bias=True, view=True)),
    ("c5_nt_bias_swish_const_pdl", NT, 640, 640, 600, ("cluster", 5), dict(bias=True, act=1, const_pdl=True)),
    ("c5_nt_bias_swish_zout", NT, 640, 640, 600, ("cluster", 5), dict(bias=True, act=1, z_out=True)),
    ("c7_nt_bias_tanh", NT, 384, 896, 600, ("cluster", 7), dict(bias=True, act=3)),
    ("c6_nn_dswish", NN, 768, 512, 1000, ("cluster", 6), dict(dact=1)),
    ("c6_nn_add", NN, 768, 512, 1000, ("cluster", 6), dict(add=True)),
    ("c4_tn", TN, 600, 600, 350, ("cluster", 4), dict()),
    ("c2_nt", NT, 128, 256, 100, ("cluster", 2), dict()),
    # ---- grouped split-K + splitk_reduce_kernel
    ("g2_tn_uv_pair_grad", TN, 1024, 512, 48000, ("grouped", 2), dict()),
    ("g2_tn_uv_grad", TN, 512, 512, 48000, ("grouped", 2), dict()),
    ("g6_tn", TN, 600, 1800, 128000, ("grouped", 6), dict()),
    ("g2_nt_bias_swish_zout_view", NT, 256, 192, 30000, ("grouped", 2), dict(bias=True, act=1, z_out=True, view=True)),
    # ---- SIMT fallbacks
    ("simt_tn_ws_overflow", TN, 2048, 2048, 50000, ("simt",), dict()),                       # 3 x 16 MB partials > 32 MB
    ("simt_nt_misaligned_base", NT, 2000, 600, 600, ("simt",), dict(shift=1)),
    ("simt_nt_lda_not_4", NT, 2000, 600, 598, ("simt",), dict()),
    # ---- fewer than 64 rows (decoder graphs: 12 beads, 36 vector rows), and the tcgen05 row threshold
    ("skinny_nt_k100", NT, 12, 1024, 100, ("gemm_skinny_kernel", (16, 1, 2), 64), dict(bias=True, act=1)),   # K < 128
    ("simt_cluster_nn_m36", NN, 36, 600, 600, ("simt_cluster", (19, 1, 5), 256), dict()),       # update-block mixes
    ("simt_cluster_nt_m63", NT, 63, 256, 256, ("simt_cluster", (4, 1, 2), 256), dict()),
    ("tc_cluster_nt_m64", NT, 64, 256, 256, ("cluster", 4), dict()),
    ("simt_splitk_tn_m48", TN, 48, 600, 2000, ("simt_splitk", (10, 1, 16), 256), dict()),
    ("stream_nt_m12", NT, 12, 600, 600, ("gemm_nt_stream_kernel", (75, 1, 1), 64), dict(bias=True, act=1)),
    ("stream_nt_m36", NT, 36, 600, 600, ("gemm_nt_stream_kernel", (100, 1, 1), 128), dict(bias=True, act=1)),
    ("stream_nn_m12", NN, 12, 600, 600, ("gemm_nn_stream_kernel", (10, 1, 8), 512), dict(dact=1)),
    ("stream_nn_m12_s1", NN, 12, 19000, 256, ("gemm_nn_stream_kernel", (149, 1, 1), 512), dict()),    # cluster of one
]


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_path_vs_float64(case):
    name, form, M, N, K, path, kw = case
    _gemm_case(form, M, N, K, path, seed=(M * 31 + N * 7 + K) % 100003, **kw)


def test_linear_pair_adjacent_weights_one_stream_launch():
    """ops.linear_pair_fwd with W1 / W2 adjacent in one buffer (u_mat / v_mat of an update block): one NT weight-streaming
    launch over both weight matrices, each output against float64"""
    M, N1, N2, K = 36, 600, 600, 600
    gen = torch.Generator(device=DEV).manual_seed(36)
    x = torch.randn(M, K, device=DEV, generator=gen)
    W = torch.randn(N1 + N2, K, device=DEV, generator=gen) / math.sqrt(K)
    W1, W2 = W[:N1], W[N1:]
    _poison_allocator(M, N1, (M, N2))
    (C1, C2), launches = _probe(lambda: ops.linear_pair_fwd(x, W1, W2))
    _assert_launches(launches, [("gemm_nt_stream_kernel", {0: 120, 1: 1, 2: 1}, 256)])
    for got, Wi in ((C1, W1), (C2, W2)):
        err = _rel_err(got, _mm64(NT, x, Wi))
        assert err < TOL, err
    again = ops.linear_pair_fwd(x, W1, W2)
    assert torch.equal(again[0], C1) and torch.equal(again[1], C2)


# ------------------------------------------------------------------------------------------ message-layer forward

def _message64(n_split, graph, geom, phi, v, Wf, bf, res_s, res_v):
    """float64 message layer from the same per-edge records (basis, unit): conv.py:505-563 / 358-402"""
    n, F = phi.shape[0], phi.shape[2]
    E = int(graph.rowptr[-1])
    col = graph.col.long()[:E]
    recv = torch.repeat_interleave(torch.arange(n, device=DEV), (graph.rowptr[1:] - graph.rowptr[:-1]).long())[:E]
    Wfull = torch.zeros(n_split * F, geom.rb, dtype=torch.float64, device=DEV)
    Wfull[:, :geom.n_rbf] = Wf.double()
    Wfull[:, geom.n_rbf] = bf.double()
    m = phi.double()[col] * (geom.basis[:E].double() @ Wfull.t()).view(E, n_split, F)
    dv_e = m[:, 2, None, :] * geom.unit[:E, :3].double()[:, :, None] + m[:, 0, None, :] * v.double()[col]
    if n_split == 4:
        dv_e = dv_e + m[:, 3, None, :] * torch.linalg.cross(v.double()[recv], v.double()[col], dim=1)
    ds = torch.zeros(n, F, dtype=torch.float64, device=DEV).index_add_(0, recv, m[:, 1])
    dv = torch.zeros(n, 3, F, dtype=torch.float64, device=DEV).index_add_(0, recv, dv_e)
    return ds + res_s.double(), dv + res_v.double()


# (n_split, MSG_TC, receivers, F, R, cutoff, expected launch (kernel, {grid axis: extent}, block.x))
MESSAGE_CASES = [
    ("simt_k3", 3, "0", 350, 600, 10, 12.0, ("message_fwd_kernel", {0: 88, 1: 19, 2: 1}, 128)),    # grid.x = ceil(350 / 4)
    ("tc_k3_rc8", 3, "1", 350, 600, 10, 12.0, ("message_tc_fwd_kernel", {}, 320)),                  # 8 consumer warps
    ("tc_k4_rc8", 4, "1", 250, 512, 8, 7.0, ("message_tc_fwd_kernel", {}, 320)),
]


@pytest.mark.parametrize("case", MESSAGE_CASES, ids=[c[0] for c in MESSAGE_CASES])
def test_message_fwd_path_vs_float64(case):
    _, n_split, tc, n, F, R, cutoff, want = case
    gen = torch.Generator().manual_seed(n + F)
    xyz = torch.as_tensor(synthetic.lattice_points(n, 2.2, np.random.default_rng(n), rotate=False), device=DEV)
    half = ops.radius_graph(xyz, cutoff, True)
    graph = ops.build_graph(torch.cat([half, half.flip(1)], 0), n)
    geom = ops.edge_geometry(graph, xyz, xyz, R, cutoff)
    phi = torch.randn(n, n_split, F, generator=gen).to(DEV)
    v = torch.randn(n, 3, F, generator=gen).to(DEV)
    Wf = (torch.randn(n_split * F, R, generator=gen) * 0.5).to(DEV)
    bf = (torch.randn(n_split * F, generator=gen) * 0.5).to(DEV)
    res_s, res_v = torch.randn(n, F, generator=gen).to(DEV), torch.randn(n, 3, F, generator=gen).to(DEV)
    old = ops.MSG_TC, ops.MSG_TC_RC, ops.MSG_TC_CROSS_RC
    try:
        ops.MSG_TC, ops.MSG_TC_RC, ops.MSG_TC_CROSS_RC = tc, 8, 8
        if tc == "1":
            ops.message_tiles(geom, False, 8)               # built once per graph, outside the profiled call

        def call():
            _poison_allocator(n, F, (n, 3, F))
            return ops.message_fwd(n_split, phi, v, v if n_split == 4 else None, geom, Wf, bf, res_s, res_v)

        got, launches = _probe(call)
        again = call()
    finally:
        ops.MSG_TC, ops.MSG_TC_RC, ops.MSG_TC_CROSS_RC = old
    _assert_launches([k for k in launches if k[0] == want[0]], [want])
    ds, dv = _message64(n_split, graph, geom, phi, v, Wf, bf, res_s, res_v)
    for a, b in ((got[0], ds), (got[1], dv)):
        err = _rel_err(a, b)
        assert err < TOL, err
    assert torch.equal(again[0], got[0]) and torch.equal(again[1], got[1])


# ------------------------------------------------------------------------------------------ column sums

def _colsum_cluster(N):
    S = min(8, max(1, (2 * NUM_SM) // ((N + 31) // 32)))
    while S & (S - 1):
        S &= S - 1
    return S


def _colsum_case(X):
    M, N = X.shape
    want = torch.zeros(N, dtype=torch.float64, device=DEV)
    for r0 in range(0, M, 16384):
        want += X[r0:r0 + 16384].double().sum(0)
    got, launches = _probe(lambda: ops.colsum(X))
    if M >= 4096:
        _assert_launches(launches, [("colsum_tall_kernel", {0: (N + 31) // 32, 1: _colsum_cluster(N)})])
    else:
        _assert_launches(launches, [("colsum_kernel", {})])
    err = _rel_err(got, want)
    assert err < TOL, err
    assert torch.equal(ops.colsum(X), got)
    print("colsum %dx%d: rel err %.2e" % (M, N, err))
    return err


@pytest.mark.parametrize("N", [1, 33, 512, 2048, 5400])
@pytest.mark.parametrize("M", [4095, 4096, 16000, 48000, 128000])
def test_colsum_vs_float64(M, N):
    """bias gradients: colsum_kernel below 4096 rows, colsum_tall_kernel (cluster sizes 8, 4, 1 over these widths) above"""
    gen = torch.Generator(device=DEV).manual_seed(M + N)
    X = torch.randn(M, N, device=DEV, generator=gen) + 0.5        # non-zero mean: no column sum near zero by chance
    _colsum_case(X)
    assert _colsum_cluster(N) == {1: 8, 33: 8, 512: 8, 2048: 4, 5400: 1}[N]


def test_colsum_strided_rows():
    gen = torch.Generator(device=DEV).manual_seed(5)
    buf = torch.full((16000, 512 + 7), NAN, device=DEV)
    buf[:, 3:3 + 512] = torch.randn(16000, 512, device=DEV, generator=gen) + 0.5
    _colsum_case(buf[:, 3:3 + 512])


# ------------------------------------------------------------------------------------------ rank-segmented weight gradients

WG_SHAPES = [(600, 600), (1800, 600), (600, 10), (7, 5)]


def _segmented_case(world, misaligned, seed):
    """A factor table laid out like train.TrainStep._pack_factors: every rank's gy / x pieces packed into an arena of L
    floats (pieces padded to 4 floats; the padding is NaN here), the arenas of `world` ranks gathered back to back, one
    problem over rows * world rows with seg_rows = rows and segment stride L.  misaligned: L % 4 != 0."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    specs = []                                              # (rows, n_out, n_in, has_w, has_b)
    for seg in (12, 36, 350):
        for n_out, n_in in WG_SHAPES:
            specs += [(seg, n_out, n_in, True, True), (seg, n_out, n_in, True, False), (seg, n_out, n_in, False, True)]
    specs += [(12 + i, 17 + 5 * i, 9 + 3 * i, True, i % 2 == 0) for i in range(14)]       # > 48 problems: two launches
    layout, off = [], 0

    def place(n):
        nonlocal off
        start = off
        off += n
        off += (-off) % 4
        return start

    for rows, n_out, n_in, has_w, has_b in specs:
        layout.append((place(rows * n_out), place(rows * n_in) if has_w else None))
    L = off + (1 if misaligned else 0)
    gathered = torch.full((world * L,), NAN, device=DEV)
    for r in range(world):
        for (rows, n_out, n_in, has_w, _), (g_off, x_off) in zip(specs, layout):
            gathered[r * L + g_off:r * L + g_off + rows * n_out] = torch.randn(rows * n_out, device=DEV, generator=gen)
            if has_w:
                gathered[r * L + x_off:r * L + x_off + rows * n_in] = torch.randn(rows * n_in, device=DEV, generator=gen)
    table = np.zeros(len(specs), dtype=ops._wgrad_dtype())
    base = gathered.data_ptr()
    outs, plain, want = [], [], []
    for i, ((rows, n_out, n_in, has_w, has_b), (g_off, x_off)) in enumerate(zip(specs, layout)):
        dW = torch.full((n_out, n_in), NAN, device=DEV) if has_w else None
        db = torch.full((n_out,), NAN, device=DEV) if has_b else None
        table[i] = (base + 4 * g_off, (base + 4 * x_off) if has_w else 0, dW.data_ptr() if has_w else 0,
                    db.data_ptr() if has_b else 0, rows * world, n_out, n_in if has_w else 0, n_out, n_in if has_w else 0,
                    rows, L, L)
        gys = [gathered[r * L + g_off:r * L + g_off + rows * n_out].view(rows, n_out) for r in range(world)]
        xs = [gathered[r * L + x_off:r * L + x_off + rows * n_in].view(rows, n_in) for r in range(world)] if has_w else None
        w64 = sum(g.double().t() @ x.double() for g, x in zip(gys, xs)) if has_w else None
        b64 = sum(g.double().sum(0) for g in gys) if has_b else None
        outs.append((dW, db))
        want.append((w64, b64))
        # the same rows physically concatenated, through the unsegmented table
        plain.append((torch.cat(gys), torch.cat(xs) if has_w else None,
                      torch.full((n_out, n_in), NAN, device=DEV) if has_w else None,
                      torch.full((n_out,), NAN, device=DEV) if has_b else None))
    _, launches = _probe(lambda: ops.wgrad_grouped_table(table))
    n_launch = (len(specs) + ops.WGRAD_PROBLEMS_PER_LAUNCH - 1) // ops.WGRAD_PROBLEMS_PER_LAUNCH
    _assert_launches(launches, [("wgrad_grouped_kernel", {})] * n_launch)
    worst = 0.0
    for spec, (dW, db), (w64, b64) in zip(specs, outs, want):
        for got, ref in ((dW, w64), (db, b64)):
            if got is not None:
                e = _rel_err(got, ref)
                assert e < TOL, (spec, e)
                worst = max(worst, e)
    ops.wgrad_grouped(plain)
    for (dW, db), (_, _, pW, pb) in zip(outs, plain):           # rows are summed in the same order either way
        assert (dW is None or torch.equal(dW, pW)) and (db is None or torch.equal(db, pb))
    first = [t.clone() for pair in outs for t in pair if t is not None]
    ops.wgrad_grouped_table(table)
    assert all(torch.equal(a, b) for a, b in zip(first, [t for pair in outs for t in pair if t is not None]))
    return worst


@pytest.mark.parametrize("world,misaligned", [(2, False), (4, False), (8, False), (4, True)])
def test_wgrad_rank_segmented_vs_float64(world, misaligned):
    """cgvae_wgrad_grouped with seg_rows > 0 (the all-gathered factors of the data-parallel factor exchange):
    dW = sum_r gy_r^T x_r and db = sum_r colsum(gy_r), float64 reference, bitwise equal to the concatenated rows"""
    err = _segmented_case(world, misaligned, seed=world * 10 + int(misaligned))
    print("wgrad segmented world %d%s: rel err %.2e" % (world, " L % 4 != 0" if misaligned else "", err))


# ------------------------------------------------------------------------------------------ one update block at c4 size

def _on_cpu(P):
    """oracle parameters with their gradients, on the CPU (parity_cases._check_grads compares there)"""
    out = {}
    for k, t in P.items():
        c = t.detach().cpu().requires_grad_()
        c.grad = t.grad.detach().cpu() if t.grad is not None else None
        out[k] = c
    return out


@pytest.mark.parametrize("paired", [False, True], ids=["separate", "paired_uv"])
def test_update_block_c4_size_vs_float64(paired):
    """UpdateBlock(feat_dim=512) on 16 000 nodes, forward and backward, against the oracle in float64 on the device.
    paired: u_mat / v_mat adjacent views of one buffer (TrainStep's layout), which takes the paired backward: NN over
    [3N, 2F] + add and one grouped TN into [2F, F]."""
    n, F = 16000, 512
    torch.manual_seed(7)
    blk = cg.UpdateBlock(feat_dim=F, activation="swish", dropout=0.0).to(DEV)
    with torch.no_grad():                                   # non-zero biases: the bias epilogues must show in the result
        for lin in blk.s_dense:
            lin.bias.normal_(0.0, 0.5)
    if paired:
        buf = torch.cat([blk.u_mat.weight.detach().reshape(-1), blk.v_mat.weight.detach().reshape(-1)])
        blk.u_mat.weight.data = buf[:F * F].view(F, F)
        blk.v_mat.weight.data = buf[F * F:].view(F, F)
    gen = torch.Generator(device=DEV).manual_seed(11)
    s0 = torch.randn(n, F, device=DEV, generator=gen)
    v0 = torch.randn(n, F, 3, device=DEV, generator=gen)
    gs = torch.randn(n, F, device=DEV, generator=gen)
    gv = torch.randn(n, F, 3, device=DEV, generator=gen)
    s, v = s0.clone().requires_grad_(), v0.clone().requires_grad_()
    ds, dv = blk(s, v)
    loss = (ds * gs).sum() + (dv * gv).sum()
    _, launches = _probe(loss.backward)
    names = [k for k, _, _ in launches]
    grids = [(k, g) for k, g, _ in launches]
    assert ("gemm_tc_persistent_kernel", (NUM_SM, 1, 1)) in grids, launches
    assert "colsum_tall_kernel" in names, launches
    grouped = [i for i, (k, g) in enumerate(grids) if k == "gemm_tc_kernel" and g[2] == 16]
    assert grouped and "splitk_reduce_kernel" in names[grouped[0]:], launches
    if paired:      # [gU; gV] over 48 000 rows as ONE [1024, 512] contraction (4 x 8 tiles, 2 groups of 8)
        assert ("gemm_tc_kernel", (4, 8, 16)) in grids, launches
    # oracle: fp32 (for the conditioning-aware criterion) and float64 (the truth), both on the device
    outs = {}
    for dt in (torch.float32, torch.float64):
        P = {"blk." + k: t.detach().clone().to(dt).requires_grad_() for k, t in blk.state_dict().items()}
        so, vo = s0.to(dt, copy=True).requires_grad_(), v0.to(dt, copy=True).requires_grad_()
        ods, odv = orc.update_block(P, "blk", so, vo)
        ((ods * gs.to(dt)).sum() + (odv * gv.to(dt)).sum()).backward()
        outs[dt] = (_on_cpu(P), ods.detach(), odv.detach(), so.grad, vo.grad)
    P32, P64 = outs[torch.float32][0], outs[torch.float64][0]
    _, ds64, dv64, gs64, gv64 = outs[torch.float64]
    _, _, _, gs32, gv32 = outs[torch.float32]
    assert _rel_err(ds, ds64) < TOL and _rel_err(dv, dv64) < TOL
    for got, ref32, truth in ((s.grad, gs32, gs64), (v.grad, gv32, gv64)):
        assert _rel_err(got, truth) < max(TOL, 10.0 * _rel_err(ref32, truth))
    worst = pc._check_grads(blk, P32, TOL, "blk.", P64=P64)
    print("update block c4 (%s): outputs %.2e / %.2e, worst fp32-vs-fp32 parameter gradient %.2e"
          % ("paired" if paired else "separate", _rel_err(ds, ds64), _rel_err(dv, dv64), worst))


# ------------------------------------------------------------------------------------------ wrapper checks

def test_gemm_rejects_mismatched_epilogue_operands():
    M, N, K = 256, 192, 64
    A = torch.randn(M, K, device=DEV)
    W = torch.randn(N, K, device=DEV)
    ok = torch.randn(N, device=DEV)
    aux = torch.randn(M, N, device=DEV)
    assert _rel_err(ops.gemm(NT, A, W, M, N, K, bias=ok), _mm64(NT, A, W) + ok.double()) < TOL
    for bad in (ok.double(), torch.randn(2 * N, device=DEV)[::2], torch.randn(N + 1, device=DEV), ok.cpu(),
                torch.randn(1, N, device=DEV)):
        with pytest.raises(RuntimeError):
            ops.gemm(NT, A, W, M, N, K, bias=bad)
    wide = torch.randn(M, N + 8, device=DEV)
    for bad in (aux.double(), torch.randn(N, M, device=DEV).t(), wide[:, :N], torch.randn(M, N + 1, device=DEV),
                aux.cpu()):
        with pytest.raises(RuntimeError):
            ops.gemm(NN, A, W.t().contiguous(), M, N, K, z_in=bad, dact=1)
        with pytest.raises(RuntimeError):
            ops.gemm(NN, A, W.t().contiguous(), M, N, K, add=bad)
    # an aux operand with the row pitch of a strided output is accepted
    out = torch.full((M, N + 8), NAN, device=DEV)[:, :N]
    got = ops.gemm(NN, A, W.t().contiguous(), M, N, K, add=wide[:, :N], out=out)
    assert got.data_ptr() == out.data_ptr() and _rel_err(got, _mm64(NN, A, W.t()) + wide[:, :N].double()) < TOL
    # z_out writes a contiguous (M, N) copy with the output's row pitch: only an output of row pitch N may ask for it
    with pytest.raises(RuntimeError):
        ops.gemm(NT, A, W, M, N, K, bias=ok, act=1, z_out=True, out=torch.empty(M, N + 4, device=DEV)[:, :N])
    for bad_out in (torch.empty(M, N, device=DEV, dtype=torch.float64), torch.empty(N, M, device=DEV).t(),
                    torch.empty(M + 1, N, device=DEV)):
        with pytest.raises(RuntimeError):
            ops.gemm(NT, A, W, M, N, K, out=bad_out)


def test_colsum_rejects_non_unit_inner_stride():
    X = torch.randn(5000, 64, device=DEV)
    with pytest.raises(RuntimeError):
        ops.colsum(X.t())
    with pytest.raises(RuntimeError):
        ops.colsum(X.double())
    assert _rel_err(ops.colsum(X), X.double().sum(0)) < TOL
