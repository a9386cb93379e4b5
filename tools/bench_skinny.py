"""Isolated timing of the decoder-shaped skinny GEMMs (M = 12 / 36 rows), weights rotated through > L2 worth of buffers."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from coarsegrainingvae_b200 import ops
dev = "cuda"
def bench(fn_list, iters=5):
    """the launches are captured in a CUDA graph so the host wrapper (~12 us per call) is out of the measurement"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for f in fn_list: f()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for f in fn_list: f()
    g.replay(); torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (iters * len(fn_list)) * 1e3
shapes = [("W1", 600, 600), ("W2", 5400, 600), ("A0", 600, 1200), ("A1", 1800, 600)]
for M in (12, 36):
    for name, n_out, n_in in shapes:
        nbuf = max(2, int(300e6 // (n_out * n_in * 4)))
        nbuf = min(nbuf, 64)
        Ws = [torch.randn(n_out, n_in, device=dev) for _ in range(nbuf)]
        x = torch.randn(M, n_in, device=dev); gy = torch.randn(M, n_out, device=dev); b = torch.randn(n_out, device=dev)
        t_nt = bench([lambda W=W: ops.gemm(ops.GEMM_NT, x, W, M, n_out, n_in, bias=b, act=1) for W in Ws])
        t_nn = bench([lambda W=W: ops.gemm(ops.GEMM_NN, gy, W, M, n_in, n_out) for W in Ws])
        t_tn = bench([lambda: ops.gemm(ops.GEMM_TN, gy, x, n_out, n_in, M) for _ in Ws])
        mb = n_out * n_in * 4 / 1e6
        print("M=%2d %s [%4dx%4d] %5.1f MB | NT %6.1f us (%5.2f TB/s)  NN %6.1f us (%5.2f TB/s)  TN %6.1f us (%5.2f TB/s write)" %
              (M, name, n_out, n_in, mb, t_nt, mb / t_nt, t_nn, mb / t_nn, t_tn, mb / t_tn), flush=True)

# all decoder-layer parameter gradients of one chignolin step in one grouped launch (cgvae_wgrad_grouped)
for M in (12,):
    probs = []
    for layer in range(9):
        for name, n_out, n_in in shapes:
            rows = 3 * M if name == "U" else M
            probs.append((torch.randn(rows, n_out, device=dev), torch.randn(rows, n_in, device=dev),
                          torch.empty(n_out, n_in, device=dev), torch.empty(n_out, device=dev)))
        for _ in range(2):      # u_mat / v_mat: 36 rows
            probs.append((torch.randn(3 * M, 600, device=dev), torch.randn(3 * M, 600, device=dev),
                          torch.empty(600, 600, device=dev), None))
    mb = sum(p[2].numel() for p in probs) * 4 / 1e6
    t = bench([lambda: ops.wgrad_grouped(probs)], iters=10)
    print("grouped wgrad: %d problems, %.0f MB written, %.1f us (%.2f TB/s)" % (len(probs), mb, t, mb / t), flush=True)
