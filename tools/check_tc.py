"""tcgen05 3xTF32 GEMM (csrc/gemm_tc.cu) vs float64, all operand forms, timed inside a CUDA graph (20 launches per replay,
operands rotated through 4 buffers).
    python tools/check_tc.py [--big]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from coarsegrainingvae_b200 import ops
dev = "cuda"
def rel(a, b):
    return float((a.double().cpu() - b).abs().max() / b.abs().max())
def graph_time(fn, reps=20):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for i in range(3): fn(i)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for i in range(reps): fn(i)
    g.replay(); torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 5 / reps * 1e3     # us per launch
shapes = [(350, 1800, 600), (350, 600, 600), (350, 600, 1800), (704, 600, 600), (97, 130, 77), (1000, 130, 77), (2000, 600, 600),
          (4000, 2048, 512)]
if "--big" in sys.argv:
    shapes += [(16000, 2048, 512), (128000, 600, 600)]
for (M, N, K) in shapes:
    g = torch.Generator().manual_seed(M + N)
    A = torch.randn(M, K, generator=g); W = torch.randn(N, K, generator=g) / K ** 0.5; b = torch.randn(N, generator=g)
    gy = torch.randn(M, N, generator=g)
    Ad, Wd, bd, gyd = A.to(dev), W.to(dev), b.to(dev), gy.to(dev)
    ref = A.double() @ W.double().t() + b.double()
    y, z = ops.gemm(ops.GEMM_NT, Ad, Wd, M, N, K, bias=bd, act=1, z_out=True)
    torch.cuda.synchronize()
    e_nt = rel(z, ref)
    got = ops.gemm(ops.GEMM_NN, gyd, Wd, M, K, N)
    e_nn = rel(got, gy.double() @ W.double())
    got = ops.gemm(ops.GEMM_TN, gyd, Ad, N, K, M)
    e_tn = rel(got, gy.double().t() @ A.double())
    nb = 4 if M * max(N, K) < 5e7 else 1
    As = [Ad.clone() for _ in range(nb)]; Ws = [Wd.clone() for _ in range(nb)]; Gs = [gyd.clone() for _ in range(nb)]
    o_nt = torch.empty(M, N, device=dev); o_nn = torch.empty(M, K, device=dev); o_tn = torch.empty(N, K, device=dev)
    us_nt = graph_time(lambda i: ops.gemm(ops.GEMM_NT, As[i % nb], Ws[i % nb], M, N, K, bias=bd, act=1, out=o_nt))
    us_nn = graph_time(lambda i: ops.gemm(ops.GEMM_NN, Gs[i % nb], Ws[i % nb], M, K, N, out=o_nn))
    us_tn = graph_time(lambda i: ops.gemm(ops.GEMM_TN, Gs[i % nb], As[i % nb], N, K, M, out=o_tn))
    fl = 2.0 * M * N * K / 1e6
    print("M%6d N%5d K%5d  err NT %.2e NN %.2e TN %.2e | NT %8.1f us %6.1f TF  NN %8.1f us %6.1f TF  TN %8.1f us %6.1f TF" %
          (M, N, K, e_nt, e_nn, e_tn, us_nt, fl / us_nt, us_nn, fl / us_nn, us_tn, fl / us_tn), flush=True)
if "--long" in sys.argv:
    for (M, N, K) in [(512, 512, 48000), (1536, 512, 16000), (600, 1800, 128000)]:
        g = torch.Generator().manual_seed(1)
        X = torch.randn(K, M, generator=g).to(dev); Y = torch.randn(K, N, generator=g).to(dev)
        ref = X.double().cpu().t() @ Y.double().cpu()
        got = ops.gemm(ops.GEMM_TN, X, Y, M, N, K)
        o = torch.empty(M, N, device=dev)
        us = graph_time(lambda i: ops.gemm(ops.GEMM_TN, X, Y, M, N, K, out=o), reps=5)
        print("TN M%5d N%5d K%7d err %.2e  %8.1f us %6.1f TF" % (M, N, K, rel(got, ref), us, 2.0 * M * N * K / us / 1e6), flush=True)
