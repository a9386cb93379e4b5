"""Tensor-level wrappers over the C ABI (include/cgvae_b200.h).

Every function here takes CUDA tensors, allocates outputs / scratch with torch (PyTorch owns all
memory), and launches hand-written sm_100a kernels on the current stream through ctypes.  There is no
CPU path: a non-CUDA tensor raises.  Layouts: scalars [N,F]; vectors planar [N,3,F]; phi [N,K,F].
"""
import contextlib as _contextlib
import ctypes

import numpy as np
import torch

from . import _lib

ACT_CODES = {None: 0, "none": 0, "linear": 0, "swish": 1, "ReLU": 2, "relu": 2, "Tanh": 3, "tanh": 3}
GEMM_NT, GEMM_NN, GEMM_TN = 0, 1, 2


def _p(t):
    if t is None:
        return None
    return t.data_ptr()


_raw_stream = torch._C._cuda_getCurrentRawStream if hasattr(torch._C, "_cuda_getCurrentRawStream") else None


def _stream():
    # torch.cuda.current_stream() costs ~65 us per call in this torch build (it re-probes device availability);
    # the raw accessor is a plain C call.  ~500 launches per training step go through here.
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("coarsegrainingvae_b200 runs on CUDA tensors only (sm_100a kernels, no CPU fallback); "
                               "got a %s tensor" % t.device)


def _f32(t):
    if t.dtype != torch.float32:
        raise RuntimeError("expected float32, got %s" % t.dtype)
    return t.contiguous()


def launch_count():
    return _lib.launch_count()


# Device-side index validation (cgvae_set_error_flags): one int32 word per device, owned here.  Kernels skip an
# out-of-range index and OR a bit into it; check_device_errors() reads it (one host sync) and raises what the
# reference raises.  The model forwards call it in eager mode (VALIDATE) -- never while a CUDA graph is being captured;
# static-capacity batches are validated on the host instead (train.validate_batch).
VALIDATE = True
_ERR_FLAGS = {}
_ERR_TEXT = {1: "a bead holds more atoms than feature channels (cg_v[mapping, CG2atomChannel], cgvae.py:473)",
             2: "embedding index out of range (nn.Embedding, cgvae.py:273,380,591)",
             4: "CG_mapping entry outside [0, n_beads)",
             8: "edge-list entry outside [0, n_nodes)",
             16: "a collated batch exceeds its capacities, or selects an item outside the dataset"}


def error_flags(device):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    t = _ERR_FLAGS.get(idx)
    if t is None:
        t = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", idx))
        _ERR_FLAGS[idx] = t
        _lib.check(_lib.load().cgvae_set_error_flags(idx, t.data_ptr()), "set_error_flags")
    return t


def check_device_errors(device, force=False):
    """raise IndexError if a kernel rejected an index since the last check (synchronises the device)."""
    if not (VALIDATE or force) or device.type != "cuda" or torch.cuda.is_current_stream_capturing():
        return
    t = error_flags(device)
    bits = int(t.item())
    if bits:
        t.zero_()
        raise IndexError("; ".join(msg for bit, msg in _ERR_TEXT.items() if bits & bit))


class KernelTimer(object):
    """Optional CUDA-event timing of individual kernel launches on the launching stream (bench.py uses it for the
    live roofline figure).  ``records[name]`` = list of (start_event, end_event, meta)."""

    def __init__(self, names, keep_operands=False):
        self.names = set(names)
        self.records = {}
        self.keep_operands = keep_operands      # also keep the operand tensors of gemm / wgrad_grouped calls (bench.py
                                                # replays those exact launches in isolation inside a CUDA graph)

    def begin(self, name):
        if name not in self.names:
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream())
        return ev

    def end(self, name, start, meta):
        if start is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream())
        self.records.setdefault(name, []).append((start, ev, meta))

    def summary(self):
        """name -> list of (milliseconds, meta); call after a synchronize."""
        return {k: [(a.elapsed_time(b), m) for a, b, m in v] for k, v in self.records.items()}


TIMER = None      # set to a KernelTimer to time launches; None (default) adds no events

_SIDE_STREAMS = {}
FORK_ENABLED = True


class Fork(object):
    """fork / join of a side stream inside one autograd node: weight- and bias-gradient contractions do not feed the
    rest of the backward pass, so they run on a forked branch and overlap with the input-gradient chain (inside a CUDA
    graph capture this becomes a parallel branch of the graph).  Every branch is joined before the node returns, so all
    tensors it touches are still referenced -- no cross-stream allocator hazards."""

    def __init__(self, device, enabled=True):
        self.enabled = enabled and FORK_ENABLED and device.type == "cuda"
        if not self.enabled:
            return
        idx = device.index if device.index is not None else torch.cuda.current_device()
        side = _SIDE_STREAMS.get(idx)
        if side is None:
            side = torch.cuda.Stream(device=idx)
            _SIDE_STREAMS[idx] = side
        self.side = side
        self.main = torch.cuda.current_stream(idx)
        self.sync()

    def sync(self):
        """side branch sees everything the main stream has enqueued so far"""
        if self.enabled:
            ev = torch.cuda.Event()
            ev.record(self.main)
            self.side.wait_event(ev)

    def branch(self):
        if self.enabled:
            return torch.cuda.stream(self.side)
        import contextlib
        return contextlib.nullcontext()

    def join(self):
        if self.enabled:
            ev = torch.cuda.Event()
            ev.record(self.side)
            self.main.wait_event(ev)


# Optional gradient sinks: data_ptr of a parameter -> (flat buffer, offset).  When a training step registers its flat
# gradient buffer here (train.FlatGrads), the weight / bias / filter gradient kernels write straight into that buffer and
# autograd adopts the view as ``p.grad`` -- no per-parameter accumulate kernels, no flatten copy before the all-reduce.
# Valid only when every registered parameter is used once per backward (true for every model of the reference).
GRAD_SINK = {}


def _has_sink(param):
    """the parameter's gradient region of a flat buffer will be ADOPTED by autograd (registered sink, no gradient yet): the
    only situation in which a deferred (still unwritten) gradient tensor may be returned from a backward node -- with
    gradient accumulation or a parameter used twice autograd would add the uninitialised tensor before the flush."""
    return (param is not None and bool(GRAD_SINK) and param.grad is None and GRAD_SINK.get(param.data_ptr()) is not None)


def _grad_out(param, shape):
    hit = GRAD_SINK.get(param.data_ptr()) if GRAD_SINK else None
    if hit is None or param.grad is not None:
        return torch.empty(shape, dtype=param.dtype, device=param.device)
    flat, off = hit
    n = 1
    for s in shape:
        n *= s
    return flat[off:off + n].view(shape)


# --------------------------------------------------------------------------------------------------
# graphs
# --------------------------------------------------------------------------------------------------

class Graph(object):
    """Receiver CSR + sender CSR of a directed edge list, plus cached per-edge geometry.

    rowptr[n_recv+1], col[E] (sender per slot), eid[E] (original edge id per slot),
    rowptr_t[n_send+1], col_t[E] (receiver), perm_t[E] (receiver-CSR slot of the same edge).
    """

    def __init__(self, n_recv, n_send, n_edges, rowptr, col, eid, rowptr_t, col_t, perm_t):
        self.n_recv, self.n_send, self.n_edges = int(n_recv), int(n_send), int(n_edges)
        self.rowptr, self.col, self.eid = rowptr, col, eid
        self.rowptr_t, self.col_t, self.perm_t = rowptr_t, col_t, perm_t


class Geometry(object):
    """basis[E,RB] = [rbf*env | env | 0...], unit[E,4] = (ux,uy,uz,d) in receiver-CSR order."""

    def __init__(self, graph, basis, unit, n_rbf, rb, cutoff):
        self.graph, self.basis, self.unit = graph, basis, unit
        self.n_rbf, self.rb, self.cutoff = int(n_rbf), int(rb), float(cutoff)


class Segments(object):
    """bead CSR: rowptr[n_beads+1], atoms[N] ascending per bead, slot[N], rank[N] (int64), mapping[N]."""

    def __init__(self, n_beads, mapping, rowptr, atoms, slot, rank):
        self.n_beads, self.mapping = int(n_beads), mapping
        self.rowptr, self.atoms, self.slot, self.rank = rowptr, atoms, slot, rank
        self.n = int(mapping.shape[0])


def rb_for(n_rbf):
    """padded basis width: R+1 rounded up to a multiple of 4 (float4 edge records)."""
    rb = ((n_rbf + 1 + 3) // 4) * 4
    if rb < 8:
        rb = 8
    if rb > 16:
        raise RuntimeError("n_rbf up to 15 supported (got %d)" % n_rbf)
    return rb


_COEF_CACHE = {}


def rbf_coefficients(n_rbf, cutoff, device):
    """n * pi / cutoff evaluated exactly like the reference (modules.py:145,156): fp32 CPU tensor ops, then kept on the
    device (cached: a pageable H2D copy per layer would serialise the stream and cannot be graph-captured)."""
    key = (int(n_rbf), float(cutoff), str(device))
    hit = _COEF_CACHE.get(key)
    if hit is None:
        n = torch.arange(1, n_rbf + 1).float()
        hit = (n * np.pi / cutoff).to(device)
        _COEF_CACHE[key] = hit
    return hit


def exclusive_scan(counts_i32, out_dtype=torch.int64):
    _need_cuda(counts_i32)
    lib = _lib.load()
    n = counts_i32.shape[0]
    out = torch.empty(n + 1, dtype=out_dtype, device=counts_i32.device)
    if out_dtype == torch.int64:
        _lib.check(lib.cgvae_exclusive_scan(_p(counts_i32), n, _p(out), _stream()), "exclusive_scan")
    else:
        _lib.check(lib.cgvae_scan_i32(_p(counts_i32), n, _p(out), _stream()), "scan_i32")
    return out


def radius_graph(xyz, cutoff, undirected=True, frame_ptr=None, use_cells=None, capacity=None, max_frame=None):
    """get_neighbor_list (data.py:65-82) on the GPU, optionally batched over frames.

    xyz [n,3] fp32 CUDA; frame_ptr int64 [n_frames+1] (defaults to one frame).  Returns int64 [E,2]
    sorted by (i, j) -- identical, bit for bit, to the reference's per-frame lists offset and
    concatenated by CG_collate (data.py:255-270).  One host read (the edge count).

    capacity (with max_frame = atoms of the largest frame, known to the caller): static mode -- NO host read; returns
    (pairs zero-padded to [capacity, 2], count int64 [1] on the device).  The capacity must cover the worst case
    (every pair of every frame within the cutoff), which is checked on the host from the frame sizes.
    """
    _need_cuda(xyz)
    lib = _lib.load()
    xyz = _f32(xyz)
    n = xyz.shape[0]
    dev = xyz.device
    if frame_ptr is None:
        frame_ptr = torch.tensor([0, n], dtype=torch.int64, device=dev)
        max_frame = n
    else:
        frame_ptr = frame_ptr.to(device=dev, dtype=torch.int64).contiguous()
    n_frames = frame_ptr.shape[0] - 1
    if capacity is not None:
        if max_frame is None:
            raise ValueError("radius_graph(capacity=...) needs max_frame (atoms of the largest frame): no host read in static mode")
        worst = n_frames * max_frame * (max_frame - 1) // (2 if undirected else 1)
        if capacity < worst:
            raise ValueError("capacity %d below the worst case %d (%d frames of <= %d atoms)" % (capacity, worst, n_frames, max_frame))
    if use_cells is None:
        if max_frame is None:
            max_frame = int((frame_ptr[1:] - frame_ptr[:-1]).max().item()) if n_frames > 0 else 0
        use_cells = max_frame > 1024
    if n == 0:
        if capacity is not None:
            return torch.zeros((capacity, 2), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
        return torch.zeros((0, 2), dtype=torch.int64, device=dev)
    ws_bytes = int(lib.cgvae_radius_graph_ws_bytes(n, n_frames)) if use_cells else 0
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
    deg = torch.empty(n, dtype=torch.int32, device=dev)
    st = _stream()
    _lib.check(lib.cgvae_radius_graph_count(_p(xyz), n, _p(frame_ptr), n_frames, float(np.float32(cutoff)), int(bool(undirected)),
                                            int(bool(use_cells)), _p(deg), _p(ws), ws_bytes, st), "radius_graph_count")
    rowptr = exclusive_scan(deg, torch.int64)
    if capacity is not None:
        pairs = torch.zeros((capacity, 2), dtype=torch.int64, device=dev)
        _lib.check(lib.cgvae_radius_graph_fill(_p(xyz), n, _p(frame_ptr), n_frames, float(np.float32(cutoff)), int(bool(undirected)),
                                               int(bool(use_cells)), _p(rowptr), _p(pairs), _p(ws), ws_bytes, st),
                   "radius_graph_fill")
        return pairs, rowptr[-1:].clone()
    n_edges = int(rowptr[-1].item())
    pairs = torch.empty((n_edges, 2), dtype=torch.int64, device=dev)
    if n_edges:
        _lib.check(lib.cgvae_radius_graph_fill(_p(xyz), n, _p(frame_ptr), n_frames, float(np.float32(cutoff)), int(bool(undirected)),
                                               int(bool(use_cells)), _p(rowptr), _p(pairs), _p(ws), ws_bytes, st),
                   "radius_graph_fill")
    return pairs


def edge_orientation(pairs):
    """(any(col0 > col1), any(col1 > col0)) -- the two host reads of make_directed (conv.py:12-13)."""
    _need_cuda(pairs)
    lib = _lib.load()
    flags = torch.empty(2, dtype=torch.int32, device=pairs.device)
    pairs = pairs.contiguous()
    _lib.check(lib.cgvae_edge_orientation(_p(pairs), pairs.shape[0], _p(flags), _stream()), "edge_orientation")
    f = flags.tolist()
    return bool(f[0]), bool(f[1])


def build_graph(pairs, n_recv, n_send=None, symmetrize=False, n_edges_dev=None):
    """CSR views of an int64 edge list [E,2] (col 0 receiver, col 1 sender).

    symmetrize: ``pairs`` is one-directional and the flipped half of make_directed (conv.py:19) is generated inside the
    kernels (directed edge E+e = pairs[e] flipped).  n_edges_dev: int64 device scalar with the live number of rows of
    ``pairs`` (its shape is then a static capacity) -- fixed launch shapes for CUDA-graph replay."""
    _need_cuda(pairs)
    lib = _lib.load()
    if n_send is None:
        n_send = n_recv
    pairs = pairs.to(torch.int64).contiguous()
    E_in = pairs.shape[0]
    E = 2 * E_in if symmetrize else E_in
    dev = pairs.device
    st = _stream()
    sym = int(bool(symmetrize))
    error_flags(dev)
    deg_r = torch.empty(n_recv, dtype=torch.int32, device=dev)
    deg_s = torch.empty(n_send, dtype=torch.int32, device=dev)
    _lib.check(lib.cgvae_csr_count(_p(pairs), E_in, _p(n_edges_dev), sym, n_recv, n_send, _p(deg_r), _p(deg_s), st), "csr_count")
    rowptr = exclusive_scan(deg_r, torch.int32)
    rowptr_t = exclusive_scan(deg_s, torch.int32)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    eid = torch.empty(E, dtype=torch.int32, device=dev)
    col_t = torch.empty(E, dtype=torch.int32, device=dev)
    perm_t = torch.empty(E, dtype=torch.int32, device=dev)
    scratch = torch.empty(n_recv + n_send + 2 * E + 4, dtype=torch.int32, device=dev)
    _lib.check(lib.cgvae_csr_fill(_p(pairs), E_in, _p(n_edges_dev), sym, n_recv, n_send, _p(rowptr), _p(rowptr_t), _p(scratch),
                                  _p(col), _p(eid), _p(col_t), _p(perm_t), st), "csr_fill")
    return Graph(n_recv, n_send, E, rowptr, col, eid, rowptr_t, col_t, perm_t)


def build_segments(mapping, n_beads):
    """bead CSR + CG2ChannelIdx ranks (cgvae.py:451-460) for an int64 mapping [N]."""
    _need_cuda(mapping)
    lib = _lib.load()
    mapping = mapping.to(torch.int64).contiguous()
    n = mapping.shape[0]
    dev = mapping.device
    st = _stream()
    error_flags(dev)
    deg = torch.empty(n_beads, dtype=torch.int32, device=dev)
    _lib.check(lib.cgvae_segment_count(_p(mapping), n, n_beads, _p(deg), st), "segment_count")
    rowptr = exclusive_scan(deg, torch.int32)
    atoms = torch.empty(n, dtype=torch.int32, device=dev)
    slot = torch.empty(n, dtype=torch.int32, device=dev)
    rank = torch.empty(n, dtype=torch.int64, device=dev)
    scratch = torch.empty(n_beads + 4, dtype=torch.int32, device=dev)
    _lib.check(lib.cgvae_segment_rank(_p(mapping), n, n_beads, _p(rowptr), _p(scratch), _p(atoms), _p(slot), _p(rank), st),
               "segment_rank")
    return Segments(n_beads, mapping, rowptr, atoms, slot, rank)


def contraction_graph(seg):
    """atoms -> beads bipartite graph of ContractiveMessageBlock (conv.py:725-731): receiver = bead,
    sender = atom; receiver CSR is the bead CSR, the sender CSR has exactly one edge per atom."""
    dev = seg.mapping.device
    n = seg.n
    rowptr_t = torch.arange(n + 1, dtype=torch.int32, device=dev)
    col_t = seg.mapping.to(torch.int32)
    return Graph(seg.n_beads, n, n, seg.rowptr, seg.atoms, seg.atoms, rowptr_t, col_t, seg.slot)


def edge_geometry(graph, xyz_send, xyz_recv, n_rbf, cutoff, edge_wgt=None, r_edge=None):
    """per-edge basis / unit vectors in receiver-CSR order, from coordinates or from r_edge [E,3]
    (original edge order)."""
    _need_cuda(xyz_send, xyz_recv, r_edge)
    lib = _lib.load()
    dev = (r_edge if r_edge is not None else xyz_send).device
    rb = rb_for(n_rbf)
    E = graph.n_edges
    basis = torch.empty((E, rb), dtype=torch.float32, device=dev)
    unit = torch.empty((E, 4), dtype=torch.float32, device=dev)
    coef = rbf_coefficients(n_rbf, cutoff, dev)
    xs = _f32(xyz_send) if xyz_send is not None else None
    xr = _f32(xyz_recv) if xyz_recv is not None else None
    re = _f32(r_edge) if r_edge is not None else None
    w = _f32(edge_wgt) if edge_wgt is not None else None
    _lib.check(lib.cgvae_edge_geometry(_p(xs), _p(xr), _p(re), _p(graph.rowptr), _p(graph.col), graph.n_recv, E, _p(coef), n_rbf, rb,
                                       float(np.float32(cutoff)), _p(w), _p(graph.eid), _p(basis), _p(unit), _stream()),
               "edge_geometry")
    return Geometry(graph, basis, unit, n_rbf, rb, cutoff)


def edge_geometry_bwd(graph, n_rbf, cutoff, xyz_send, xyz_recv, d_basis, d_unit, edge_wgt=None, r_edge=None):
    """cotangent of the edge displacements from those of the basis / unit records of edge_geometry (either may be None =
    zero): [E,3] in receiver-CSR slot order, or, with r_edge, the gradient of r_edge in its original edge order."""
    _need_cuda(xyz_send, xyz_recv, r_edge)
    lib = _lib.load()
    g = graph
    E = g.n_edges
    dev = g.rowptr.device
    coef = rbf_coefficients(n_rbf, cutoff, dev)
    dr = torch.empty((E, 3), dtype=torch.float32, device=dev)
    xs = _f32(xyz_send) if xyz_send is not None else None
    xr = _f32(xyz_recv) if xyz_recv is not None else None
    re = _f32(r_edge) if r_edge is not None else None
    w = _f32(edge_wgt) if edge_wgt is not None else None
    db = _f32(d_basis) if d_basis is not None else None
    du = _f32(d_unit) if d_unit is not None else None
    _lib.check(lib.cgvae_edge_geometry_bwd(_p(xs), _p(xr), _p(re), _p(g.rowptr), _p(g.col), g.n_recv, E, _p(coef), n_rbf, rb_for(n_rbf),
                                           float(np.float32(cutoff)), _p(w), _p(g.eid), _p(db), _p(du), _p(dr), _stream()),
               "edge_geometry_bwd")
    return dr


def edge_coord_reduce(graph, dr, same):
    """(g_send [n_send,3], g_recv [n_recv,3] or None when ``same``) from per-slot displacement cotangents dr."""
    _need_cuda(dr)
    lib = _lib.load()
    g_send = torch.empty((graph.n_send, 3), dtype=torch.float32, device=dr.device)
    g_recv = None if same else torch.empty((graph.n_recv, 3), dtype=torch.float32, device=dr.device)
    _lib.check(lib.cgvae_edge_coord_reduce(_p(dr), _p(graph.rowptr), graph.n_recv, _p(graph.rowptr_t), _p(graph.perm_t), graph.n_send,
                                           int(bool(same)), _p(g_send), _p(g_recv), _stream()), "edge_coord_reduce")
    return g_send, g_recv


# --------------------------------------------------------------------------------------------------
# dense
# --------------------------------------------------------------------------------------------------

_SPLITK_WS_BYTES = 32 << 20


def gemm(form, A, B, M, N, K, bias=None, act=0, z_out=False, z_in=None, dact=0, add=None, out=None):
    """C[M,N] = epilogue(op(A) op(B)); see cgvae_gemm in the header.  A, B 2-D contiguous views."""
    _need_cuda(A, B)
    if A.dtype != torch.float32 or B.dtype != torch.float32 or A.stride(-1) != 1 or B.stride(-1) != 1:
        raise RuntimeError("gemm: operands must be float32 with unit inner stride (got %s %s, %s %s)"
                           % (A.dtype, tuple(A.stride()), B.dtype, tuple(B.stride())))
    lib = _lib.load()
    dev = A.device
    if out is not None and (out.dtype != torch.float32 or out.device != dev or tuple(out.shape) != (M, N)
                            or (N > 1 and out.stride(1) != 1)):
        raise RuntimeError("gemm: out must be a float32 (%d, %d) tensor with unit inner stride on %s (got %s %s %s on %s)"
                           % (M, N, dev, out.dtype, tuple(out.shape), tuple(out.stride()), out.device))
    C = out if out is not None else torch.empty((M, N), dtype=torch.float32, device=dev)
    # the kernels read bias[n] and z_in / add / z_out at m * ldc + n, with ldc = C's row stride
    ldc = C.stride(0)
    if bias is not None and (bias.dtype != torch.float32 or bias.dim() != 1 or bias.numel() != N
                             or not bias.is_contiguous() or bias.device != dev):
        raise RuntimeError("gemm: bias must be a contiguous float32 vector of length %d on %s (got %s %s %s on %s)"
                           % (N, dev, bias.dtype, tuple(bias.shape), tuple(bias.stride()), bias.device))
    for name, t in (("z_in", z_in), ("add", add)):
        if t is not None and (t.dtype != torch.float32 or tuple(t.shape) != (M, N) or (N > 1 and t.stride(1) != 1)
                              or (M > 1 and t.stride(0) != ldc) or t.device != dev):
            raise RuntimeError("gemm: %s must be a float32 (%d, %d) tensor on %s with the row stride of the output (%d) "
                               "and unit inner stride (got %s %s %s on %s)"
                               % (name, M, N, dev, ldc, t.dtype, tuple(t.shape), tuple(t.stride()), t.device))
    if z_out and M > 1 and ldc != N:
        raise RuntimeError("gemm: z_out=True needs an output with row stride %d (the pre-activation copy is a contiguous "
                           "(M, N) tensor indexed with the output's row stride); got row stride %d" % (N, ldc))
    Z = torch.empty((M, N), dtype=torch.float32, device=dev) if z_out else None
    tiles = ((M + 63) // 64) * ((N + 63) // 64) if M > 32 else ((N + 31) // 32)
    st = _stream()
    ws = None
    if (tiles < 148 and K >= 512) or (K > 24576 and M >= 64):      # split-K workspace (SIMT tiles; tcgen05 group partials)
        ws = torch.empty(_SPLITK_WS_BYTES, dtype=torch.uint8, device=dev)
    t0 = TIMER.begin("gemm") if TIMER is not None else None
    _lib.check(lib.cgvae_gemm(form, _p(A), A.stride(0), _p(B), B.stride(0), _p(C), ldc, M, N, K, _p(bias), act, _p(Z),
                              _p(z_in), dact, _p(add), _p(ws), _SPLITK_WS_BYTES if ws is not None else 0, None, 0, st),
               "gemm")
    if t0 is not None:
        meta = dict(form=form, M=M, N=N, K=K, lda=A.stride(0), ldb=B.stride(0))
        if TIMER.keep_operands:
            meta.update(A=A, B=B, bias=bias, act=act, z_in=z_in, dact=dact, add=add)
        TIMER.end("gemm", t0, meta)
    return (C, Z) if z_out else C


def linear_fwd(x, W, b, act=0, save_pre=False):
    """y = act(x W^T + b)   (Dense.forward, modules.py:99-112)"""
    M, K = x.shape
    N = W.shape[0]
    return gemm(GEMM_NT, x, W, M, N, K, bias=b, act=act, z_out=save_pre)


def linear_pair_fwd(x, W1, W2):
    """(x W1^T, x W2^T) for two bias-free Dense layers on the same input.  When the two weight matrices are adjacent in
    memory (consecutive parameters of the flat parameter buffer of train.TrainStep) this is ONE weight-streaming launch
    (cgvae_dense_pair_fwd); otherwise two."""
    M, K = x.shape
    N1, N2 = W1.shape[0], W2.shape[0]
    adjacent = (W1.is_contiguous() and W2.is_contiguous() and W1.shape[1] == K and W2.shape[1] == K
                and W2.data_ptr() == W1.data_ptr() + 4 * W1.numel())
    if not adjacent:
        return linear_fwd(x, W1, None, 0), linear_fwd(x, W2, None, 0)
    _need_cuda(x, W1)
    lib = _lib.load()
    C1 = torch.empty((M, N1), dtype=torch.float32, device=x.device)
    C2 = torch.empty((M, N2), dtype=torch.float32, device=x.device)
    _lib.check(lib.cgvae_dense_pair_fwd(_p(x), x.stride(0), _p(W1), K, M, N1, N2, K, _p(C1), _p(C2), _stream()), "dense_pair_fwd")
    return C1, C2


def linear_bwd_input(gy, W, z_in=None, dact=0, add=None):
    """gx = (gy W) [* act'(z_in)] [+ add]"""
    M, N = gy.shape
    K = W.shape[1]
    return gemm(GEMM_NN, gy, W, M, K, N, z_in=z_in, dact=dact, add=add)


# Deferred parameter gradients.  Weight / bias gradients of Dense layers on small node sets (decoder graphs: 12..96
# rows) cost as much as writing them; one launch per layer cannot keep enough stores in flight (1.2 ms per chignolin
# step in 92 + 56 launches).  Nothing in the backward pass reads them, so while a DeferredGrads scope is open
# (train.TrainStep opens one around loss.backward() when gradient sinks are registered) they are only RECORDED, and
# flush() produces all of them with cgvae_wgrad_grouped: one launch per 48 problems.  The recorded operands stay
# referenced until the flush, which is enqueued on the stream the backward ran on.
DEFER_MAX_ROWS = 128
_DEFERRED = None


def deferring(rows):
    return _DEFERRED is not None and rows <= DEFER_MAX_ROWS


WGRAD_PROBLEMS_PER_LAUNCH = 48


class DeferredGrads(object):
    """flush=True: the grouped launch is issued when the scope closes.  flush=False: the merged problem list is left in
    ``self.pending`` for the caller (data-parallel training gathers the FACTORS of all ranks first, train.TrainStep)."""

    def __init__(self, flush=True):
        self.flush = flush
        self.pending = []

    def __enter__(self):
        global _DEFERRED
        if _DEFERRED is not None:
            raise RuntimeError("DeferredGrads scopes do not nest")
        _DEFERRED = []
        return self

    def flush_now(self):
        """launch what has been recorded so far (data-parallel overlap: the decoder's gradients must be final before their
        all-reduce starts, while the encoder's backward is still to come)."""
        global _DEFERRED
        pending, _DEFERRED = _DEFERRED, []
        if pending:
            wgrad_grouped(merge_deferred(pending))

    def __exit__(self, exc_type, exc, tb):
        global _DEFERRED
        pending, _DEFERRED = _DEFERRED, None
        if exc_type is None:
            self.pending = merge_deferred(pending)
            if self.flush:
                wgrad_grouped(self.pending)
        return False


_WGRAD_DTYPE = None


def _wgrad_dtype():
    global _WGRAD_DTYPE
    if _WGRAD_DTYPE is None:
        import numpy as np
        _WGRAD_DTYPE = np.dtype([("gy", np.uint64), ("x", np.uint64), ("dW", np.uint64), ("db", np.uint64),
                                 ("rows", np.int32), ("n_out", np.int32), ("n_in", np.int32), ("ldg", np.int32),
                                 ("ldx", np.int32), ("seg_rows", np.int32), ("seg_stride_g", np.int64),
                                 ("seg_stride_x", np.int64)], align=True)
        assert _WGRAD_DTYPE.itemsize == 72
    return _WGRAD_DTYPE


def wgrad_table(problems):
    """numpy table (struct cgvae_wgrad_problem) of a list of (gy [rows,n_out], x [rows,n_in] or None, dW or None, db or None)."""
    import numpy as np
    table = np.zeros(len(problems), dtype=_wgrad_dtype())
    for i, (gy, x, dW, db) in enumerate(problems):
        _need_cuda(gy)
        if gy.stride(1) != 1 or (x is not None and x.stride(1) != 1):
            raise ValueError("wgrad_grouped: operands must have unit column stride")
        if dW is not None and not dW.is_contiguous():
            raise ValueError("wgrad_grouped: dW must be contiguous")
        table[i] = (gy.data_ptr(), x.data_ptr() if x is not None else 0, dW.data_ptr() if dW is not None else 0,
                    db.data_ptr() if db is not None else 0, gy.shape[0], gy.shape[1], x.shape[1] if x is not None else 0,
                    gy.stride(0), x.stride(0) if x is not None else 0, 0, 0, 0)
    return table


def wgrad_grouped_table(table, out_floats=0, keep=None):
    """launch cgvae_wgrad_grouped on a prepared table (device pointers inside; the table itself is host memory)."""
    if len(table) == 0:
        return
    lib = _lib.load()
    t0 = TIMER.begin("wgrad_grouped") if TIMER is not None else None
    _lib.check(lib.cgvae_wgrad_grouped(table.ctypes.data, len(table), _stream()), "wgrad_grouped")
    if t0 is not None:
        TIMER.end("wgrad_grouped", t0, dict(problems=len(table), table=(keep if TIMER.keep_operands else None),
                                           out_floats=out_floats))


def wgrad_grouped(problems):
    """problems: list of (gy [rows,n_out], x [rows,n_in] or None, dW [n_out,n_in] or None, db [n_out] or None);
    cgvae_wgrad_grouped: every dW = gy^T x and db = colsum(gy) in one launch per 48 problems."""
    if not problems:
        return
    out_floats = sum((p[2].numel() if p[2] is not None else 0) + (p[3].numel() if p[3] is not None else 0) for p in problems)
    wgrad_grouped_table(wgrad_table(problems), out_floats, list(problems))


def merge_deferred(pending):
    """merge the bias problem of a layer into its weight problem (same gy)."""
    merged, by_gy = [], {}
    for gy, x, dW, db in pending:
        key = (gy.data_ptr(), gy.shape[0], gy.shape[1], gy.stride(0))
        hit = by_gy.get(key)
        if hit is not None and ((db is not None and merged[hit][3] is None and dW is None)
                                or (dW is not None and merged[hit][2] is None and db is None)):
            g0, x0, w0, b0 = merged[hit]
            merged[hit] = (g0, x if x0 is None else x0, dW if w0 is None else w0, db if b0 is None else b0)
            continue
        by_gy[key] = len(merged)
        merged.append((gy, x, dW, db))
    return merged


def flush_deferred(pending):
    """merge and launch."""
    wgrad_grouped(merge_deferred(pending))


def linear_bwd_weight(gy, x, param=None, shape=None):
    """gW[out,in] = gy^T x (written into the parameter's gradient sink when one is registered).  shape: the output covers
    SEVERAL parameters adjacent in the flat buffers, starting at ``param`` (u_mat / v_mat of an UpdateBlock: [2F, F])."""
    rows, n_out = gy.shape
    n_in = x.shape[1]
    if shape is not None and tuple(shape) != (n_out, n_in):
        raise ValueError("linear_bwd_weight: shape %s does not match gy^T x = (%d, %d)" % (tuple(shape), n_out, n_in))
    out = _grad_out(param, (n_out, n_in)) if param is not None else None
    if deferring(rows) and _has_sink(param) and gy.is_cuda and gy.stride(1) == 1 and x.stride(1) == 1:
        # record an ALIAS of the output: autograd only adopts a returned gradient without copying when nothing else
        # references the tensor object (AccumulateGrad's use_count test); gy / x are recorded as they are so that
        # nobody accumulates into them in place before the flush
        _DEFERRED.append((gy, x, out.detach(), None))
        return out
    return gemm(GEMM_TN, gy, x, n_out, n_in, rows, out=out)


def colsum(X, param=None):
    _need_cuda(X)
    M, N = X.shape
    if X.dtype != torch.float32 or (N > 1 and X.stride(1) != 1):     # the kernels read X[m * ldx + n]
        raise RuntimeError("colsum: X must be float32 with unit inner stride (got %s %s)" % (X.dtype, tuple(X.stride())))
    lib = _lib.load()
    out = _grad_out(param, (N,)) if param is not None else torch.empty(N, dtype=torch.float32, device=X.device)
    if deferring(M) and _has_sink(param) and X.stride(1) == 1:
        _DEFERRED.append((X, None, None, out.detach()))
        return out
    _lib.check(lib.cgvae_colsum(_p(X), X.stride(0), M, N, _p(out), _stream()), "colsum")
    return out


# --------------------------------------------------------------------------------------------------
# message layers
# --------------------------------------------------------------------------------------------------

class MessageTiles(object):
    """column tiles of a CSR for the tensor-core message kernels (cgvae_msg_tiles_build): bptr[n_chunks+1] batch offsets,
    ngroups[n_chunks], rec = batch records (uint8), rc = rows per chunk."""

    def __init__(self, rc, bptr, ngroups, rec, n_batches_cap, n_edges):
        self.rc, self.bptr, self.ngroups, self.rec = int(rc), bptr, ngroups, rec
        self.n_batches_cap, self.n_edges = int(n_batches_cap), int(n_edges)
        self.fill = None              # live edges / columns, measured once in eager mode (one host read)


# Tensor-core message path policy.  CGVAE_MSG_TC=0 disables it; =1 forces it wherever it applies (homogeneous graph,
# R <= 15).  Default "auto": 3-split layers on graphs with at least MSG_TC_MIN_EDGES directed edge slots and a mean degree
# of at least MSG_TC_MIN_DEGREE, and -- measured once per graph SHAPE outside CUDA-graph capture -- a column fill (edges /
# columns of the tiles) of at least MSG_TC_MIN_FILL.  Measured on B200 (tools/bench_message.py, profiles/r2_bench_message*):
# at chignolin density (fill 0.89) the tensor-core kernel is 1.7x the SIMT one (85 vs 142 us), at fill 0.5 (20 000 atoms,
# 12 A) 1.2x, below 0.4 it loses: the zero columns then cost more than the register re-use of the gathered sender rows
# saves, and the SIMT kernel of message.cu (L1 re-use across 4 receivers) is the better path.  The cross block (4 splits;
# PCN residue graph, fill 0.45-0.5) measured 0.7x and stays on the SIMT kernel unless forced.
import os as _os
MSG_TC = _os.environ.get("CGVAE_MSG_TC", "auto")
MSG_TC_RC = int(_os.environ.get("CGVAE_MSG_TC_RC", "8"))
MSG_TC_CROSS_RC = int(_os.environ.get("CGVAE_MSG_TC_CROSS_RC", "8"))
MSG_TC_MIN_EDGES = 4096
MSG_TC_MIN_DEGREE = 12.0
MSG_TC_MIN_FILL = float(_os.environ.get("CGVAE_MSG_TC_MIN_FILL", "0.40"))
_TC_DECISIONS = {}


def message_tiles(geom, transposed=False, rc=None):
    """forward (receiver-chunk) or backward (sender-chunk) column tiles of a Geometry, built once and cached on it."""
    rc = int(rc or MSG_TC_RC)
    cache = geom.__dict__.setdefault("_tiles", {})
    key = (rc, bool(transposed))
    hit = cache.get(key)
    if hit is not None:
        return hit
    lib = _lib.load()
    g = geom.graph
    if transposed:
        rowptr, col, slot_map, n_rows, n_part = g.rowptr_t, g.col_t, g.perm_t, g.n_send, g.n_recv
    else:
        rowptr, col, slot_map, n_rows, n_part = g.rowptr, g.col, None, g.n_recv, g.n_send
    dev = geom.basis.device
    n_chunks = (n_rows + rc - 1) // rc
    cap = int(lib.cgvae_msg_tiles_batches_cap(n_rows, n_part, g.n_edges, rc))
    rec_bytes = int(lib.cgvae_msg_tiles_rec_bytes())
    nbatch = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    bptr = torch.empty(n_chunks + 1, dtype=torch.int32, device=dev)
    ngroups = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    rec = torch.empty(cap * rec_bytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.cgvae_msg_tiles_build(_p(rowptr), _p(col), _p(slot_map), n_rows, n_part, g.n_edges, _p(geom.basis),
                                         _p(geom.unit), geom.rb, rc, _p(nbatch), _p(bptr), _p(ngroups), _p(rec), cap, _stream()),
               "msg_tiles_build")
    tiles = MessageTiles(rc, bptr, ngroups, rec, cap, g.n_edges)
    cache[key] = tiles
    return tiles


def _tc_applies(geom, n_split):
    """policy decision (see MSG_TC above); returns the forward tiles or None."""
    if MSG_TC == "0":
        return False
    g = geom.graph
    if g.n_recv != g.n_send or g.n_recv == 0 or geom.n_rbf > 15 or g.n_recv > 262144:
        return False
    if MSG_TC == "1":
        return True
    if n_split not in (3, 4):
        return False
    if g.n_edges < MSG_TC_MIN_EDGES or g.n_edges < MSG_TC_MIN_DEGREE * g.n_recv:
        return False
    key = (g.n_recv, (g.n_edges // g.n_recv) // 4, MSG_TC_RC)     # per graph shape: nodes, degree bucket
    hit = _TC_DECISIONS.get(key)
    if hit is None:
        if torch.cuda.is_current_stream_capturing():
            return True                     # no host read inside a capture: the warm-up steps normally decide first
        tiles = message_tiles(geom, False)
        if tiles.fill is None:
            live_edges = int(g.rowptr[-1].item())
            n_batches = int(tiles.bptr[-1].item())
            tiles.fill = live_edges / max(1.0, 64.0 * n_batches)
        hit = tiles.fill >= MSG_TC_MIN_FILL
        _TC_DECISIONS[key] = hit
    return hit


def message_tc_fwd(n_split, phi, v_send, v_recv, geom, Wf, bf, res_s, res_v, want_q=False):
    """cgvae_message_tc_fwd: the fused message layer with the filter contraction on the tensor cores."""
    lib = _lib.load()
    g = geom.graph
    F = phi.shape[-1]
    dev = phi.device
    rc = MSG_TC_RC if n_split == 3 else min(MSG_TC_RC, MSG_TC_CROSS_RC)   # cross block: 7 accumulators per receiver
    tiles = message_tiles(geom, False, rc)
    out_s = torch.empty((g.n_recv, F), dtype=torch.float32, device=dev)
    out_v = torch.empty((g.n_recv, 3, F), dtype=torch.float32, device=dev)
    q = torch.empty((g.n_recv, 3, F), dtype=torch.float32, device=dev) if (want_q and n_split == 4) else None
    ws_bytes = int(lib.cgvae_message_tc_ws_bytes(n_split, tiles.rc, g.n_recv, F))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    t0 = TIMER.begin("message_fwd") if TIMER is not None else None
    _lib.check(lib.cgvae_message_tc_fwd(n_split, _p(phi), _p(v_send), _p(v_recv), _p(tiles.bptr), _p(tiles.ngroups), _p(tiles.rec),
                                        tiles.n_batches_cap, tiles.rc, _p(Wf), _p(bf), g.n_recv, F, geom.n_rbf, _p(res_s),
                                        _p(res_v), int(v_send is None), _p(out_s), _p(out_v), _p(q), _p(ws), ws_bytes, _stream()),
               "message_tc_fwd")
    if t0 is not None:
        TIMER.end("message_fwd", t0, dict(n_split=n_split, E=g.n_edges, n_recv=g.n_recv, n_send=g.n_send, F=F,
                                          R=geom.n_rbf, v_zero=v_send is None, tc=True))
    return out_s, out_v, q


def message_fwd(n_split, phi, v_send, v_recv, geom, Wf, bf, res_s, res_v, want_q=False):
    """returns (out_s [n_recv,F], out_v [n_recv,3,F], q or None).  v_send None == all-zero vectors."""
    _need_cuda(phi)
    if _tc_applies(geom, n_split):
        return message_tc_fwd(n_split, phi, v_send, v_recv, geom, Wf, bf, res_s, res_v, want_q)
    lib = _lib.load()
    g = geom.graph
    F = phi.shape[-1]
    dev = phi.device
    out_s = torch.empty((g.n_recv, F), dtype=torch.float32, device=dev)
    out_v = torch.empty((g.n_recv, 3, F), dtype=torch.float32, device=dev)
    q = torch.empty((g.n_recv, 3, F), dtype=torch.float32, device=dev) if (want_q and n_split == 4) else None
    t0 = TIMER.begin("message_fwd") if TIMER is not None else None
    _lib.check(lib.cgvae_message_fwd(n_split, _p(phi), _p(v_send), _p(v_recv), _p(g.rowptr), _p(g.col), _p(geom.basis),
                                     _p(geom.unit), _p(Wf), _p(bf), g.n_recv, g.n_send, F, geom.n_rbf, geom.rb, _p(res_s),
                                     _p(res_v), int(v_send is None), _p(out_s), _p(out_v), _p(q), _stream()), "message_fwd")
    if t0 is not None:
        TIMER.end("message_fwd", t0, dict(n_split=n_split, E=g.n_edges, n_recv=g.n_recv, n_send=g.n_send, F=F,
                                          R=geom.n_rbf, v_zero=v_send is None))
    return out_s, out_v, q


def message_bwd(n_split, phi, v_send, v_recv, q, geom, Wf, bf, g_out_s, g_out_v, residual, sink=True):
    """returns (g_phi [n_send,K,F], g_v_send [n_send,3,F], dWf [K*F,R], dbf [K*F])."""
    _need_cuda(phi)
    lib = _lib.load()
    g = geom.graph
    F = phi.shape[-1]
    dev = phi.device
    g_phi = torch.empty((g.n_send, n_split, F), dtype=torch.float32, device=dev)
    g_v = torch.empty((g.n_send, 3, F), dtype=torch.float32, device=dev)
    dWf = _grad_out(Wf, (n_split * F, geom.n_rbf)) if sink else torch.empty((n_split * F, geom.n_rbf), dtype=torch.float32, device=dev)
    dbf = _grad_out(bf, (n_split * F,)) if sink else torch.empty((n_split * F,), dtype=torch.float32, device=dev)
    ws_bytes = int(lib.cgvae_message_bwd_ws_bytes(n_split, F, geom.rb, g.n_send))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    t0 = TIMER.begin("message_bwd") if TIMER is not None else None
    _lib.check(lib.cgvae_message_bwd(n_split, _p(phi), _p(v_send), _p(v_recv), _p(q), _p(g.rowptr_t), _p(g.col_t), _p(g.perm_t),
                                     _p(geom.basis), _p(geom.unit), _p(Wf), _p(bf), g.n_recv, g.n_send, F, geom.n_rbf, geom.rb,
                                     _p(g_out_s), _p(g_out_v), int(bool(residual)), int(v_send is None), _p(g_phi), _p(g_v),
                                     _p(dWf), _p(dbf), _p(ws), ws_bytes, _stream()), "message_bwd")
    if t0 is not None:
        TIMER.end("message_bwd", t0, dict(n_split=n_split, E=g.n_edges, n_recv=g.n_recv, n_send=g.n_send, F=F,
                                          R=geom.n_rbf, v_zero=v_send is None))
    return g_phi, g_v, dWf, dbf


def message_geom_bwd(n_split, phi, v_send, v_recv, geom, Wf, bf, g_out_s, g_out_v):
    """geometry cotangents of one message layer: (d_basis [E,RB], d_unit [E,4]); n_split 9 returns (None, d_unit)."""
    _need_cuda(phi)
    lib = _lib.load()
    g = geom.graph
    F = phi.shape[-1]
    dev = phi.device
    d_basis = torch.empty((g.n_edges, geom.rb), dtype=torch.float32, device=dev) if n_split != 9 else None
    d_unit = torch.empty((g.n_edges, 4), dtype=torch.float32, device=dev)
    _lib.check(lib.cgvae_message_geom_bwd(n_split, _p(phi), _p(v_send), _p(v_recv), _p(g.rowptr), _p(g.col), g.n_recv, g.n_edges,
                                          _p(geom.basis), _p(geom.unit), _p(Wf), _p(bf), F, geom.n_rbf, geom.rb, _p(g_out_s),
                                          _p(g_out_v), int(v_send is None), _p(d_basis), _p(d_unit), _stream()), "message_geom_bwd")
    return d_basis, d_unit


def message9_geom_bwd(phi, geom, Wf, bf, gw, g_v):
    """geometry cotangents of a 9-split layer: d_basis = gw [Wf | bf] with cgvae_gemm (gw from message9_bwd, padded
    basis columns zero), d_unit from the unit-only form of cgvae_message_geom_bwd."""
    g = geom.graph
    E, R, F = g.n_edges, geom.n_rbf, phi.shape[-1]
    d_basis = fill((E, geom.rb), 0.0, phi)
    if E > 0:
        with matmul_precision("highest"):           # fp32 in both precision modes, like every coordinate-gradient kernel
            gemm(GEMM_NN, gw, Wf, E, R, 9 * F, out=d_basis[:, :R])
            gemm(GEMM_NN, gw, bf.view(9 * F, 1), E, 1, 9 * F, out=d_basis[:, R:R + 1])
    _, d_unit = message_geom_bwd(9, phi, None, None, geom, Wf, bf, None, g_v)
    return d_basis, d_unit


def message9_fwd(phi, s, sbar, v, vbar, geom, Wf, bf, residual):
    _need_cuda(phi)
    lib = _lib.load()
    g = geom.graph
    n, F = s.shape
    outs = [torch.empty_like(s), torch.empty_like(sbar), torch.empty_like(v), torch.empty_like(vbar)]
    _lib.check(lib.cgvae_message9_fwd(_p(phi), _p(s), _p(sbar), _p(v), _p(vbar), _p(g.rowptr), _p(g.col), _p(geom.basis),
                                      _p(geom.unit), _p(Wf), _p(bf), n, F, geom.n_rbf, geom.rb, int(bool(residual)),
                                      _p(outs[0]), _p(outs[1]), _p(outs[2]), _p(outs[3]), _stream()), "message9_fwd")
    return outs


def message9_bwd(phi, s, sbar, v, vbar, geom, Wf, bf, residual, g_s, g_sbar, g_v, g_vbar, keep_gw=False):
    """returns (gi_s, gi_sbar, gi_v, gi_vbar, g_phi [n,9,F], dWf [9F,R], dbf [9F]), and gw [E,9F] last with keep_gw."""
    _need_cuda(phi)
    lib = _lib.load()
    g = geom.graph
    n, F = s.shape
    dev = s.device
    gi = [torch.empty_like(s), torch.empty_like(sbar), torch.empty_like(v), torch.empty_like(vbar)]
    g_phi = torch.empty((n, 9, F), dtype=torch.float32, device=dev)
    gw = torch.empty((g.n_edges, 9 * F), dtype=torch.float32, device=dev)
    _lib.check(lib.cgvae_message9_bwd(_p(phi), _p(s), _p(sbar), _p(v), _p(vbar), _p(g.rowptr), _p(g.col), _p(g.rowptr_t),
                                      _p(g.col_t), _p(g.perm_t), _p(geom.basis), _p(geom.unit), _p(Wf), _p(bf), n, g.n_edges, F,
                                      geom.n_rbf, geom.rb, int(bool(residual)), _p(g_s), _p(g_sbar), _p(g_v), _p(g_vbar), _p(gi[0]),
                                      _p(gi[1]), _p(gi[2]), _p(gi[3]), _p(g_phi), _p(gw), _stream()), "message9_bwd")
    # dWf[9F,R] = gw^T basis[:, :R] ; dbf[9F] = gw^T basis[:, R]   (DistanceEmbed weight / bias gradients)
    R = geom.n_rbf
    E = g.n_edges
    if E > 0 and deferring(E):
        dWf = linear_bwd_weight(gw, geom.basis[:, :R], Wf)
        dbf = linear_bwd_weight(gw, geom.basis[:, R:R + 1], bf).reshape(9 * F)
    elif E > 0:
        # forked branch; it is joined by the caller's next Fork.join() on the same side stream
        # (functions.Message9Block.backward -> _phi_backward), i.e. before the autograd node returns
        fork = Fork(dev)
        with fork.branch():
            dWf = gemm(GEMM_TN, gw, geom.basis, 9 * F, R, E, out=_grad_out(Wf, (9 * F, R)))
            dbf = gemm(GEMM_TN, gw, geom.basis[:, R:], 9 * F, 1, E, out=_grad_out(bf, (9 * F,)).view(9 * F, 1)).reshape(9 * F)
        if deferring(n):          # the caller's forks are disabled when its own parameter gradients are deferred
            fork.join()
    else:
        dWf = torch.zeros((9 * F, R), dtype=torch.float32, device=dev)
        dbf = torch.zeros((9 * F,), dtype=torch.float32, device=dev)
    if keep_gw:
        return gi[0], gi[1], gi[2], gi[3], g_phi, dWf, dbf, gw
    return gi[0], gi[1], gi[2], gi[3], g_phi, dWf, dbf


# --------------------------------------------------------------------------------------------------
# update block, pooling, lifting
# --------------------------------------------------------------------------------------------------

def update_norm_fwd(s, Vv):
    _need_cuda(s)
    lib = _lib.load()
    N, F = s.shape
    x = torch.empty((N, 2 * F), dtype=torch.float32, device=s.device)
    _lib.check(lib.cgvae_update_norm_fwd(_p(s), _p(Vv), N, F, _p(x), _stream()), "update_norm_fwd")
    return x


def update_combine_fwd(s, v, Uv, Vv, q, residual):
    _need_cuda(Uv)
    lib = _lib.load()
    N, _, F = Uv.shape
    s_out = torch.empty((N, F), dtype=torch.float32, device=Uv.device)
    v_out = torch.empty((N, 3, F), dtype=torch.float32, device=Uv.device)
    _lib.check(lib.cgvae_update_combine_fwd(_p(s), _p(v), _p(Uv), _p(Vv), _p(q), N, F, int(bool(residual)), _p(s_out), _p(v_out),
                                            _stream()), "update_combine_fwd")
    return s_out, v_out


def update_combine_bwd(Uv, Vv, q, g_s, g_v, cat=False):
    """cat: gUv and gVv are returned as the two column halves (views) of ONE [N, 3, 2F] tensor."""
    _need_cuda(Uv)
    lib = _lib.load()
    N, _, F = Uv.shape
    gq = torch.empty_like(q)
    if cat:
        gUV = torch.empty((N, 3, 2 * F), dtype=torch.float32, device=Uv.device)
        gUv, gVv = gUV[:, :, :F], gUV[:, :, F:]
        _lib.check(lib.cgvae_update_combine_bwd_ld(_p(Uv), _p(Vv), _p(q), _p(g_s), _p(g_v), N, F, _p(gq), _p(gUV), gUV.data_ptr() + 4 * F,
                                                   2 * F, _stream()), "update_combine_bwd_ld")
        return gq, gUv, gVv
    gUv = torch.empty_like(Uv)
    gVv = torch.empty_like(Vv)
    _lib.check(lib.cgvae_update_combine_bwd(_p(Uv), _p(Vv), _p(q), _p(g_s), _p(g_v), N, F, _p(gq), _p(gUv), _p(gVv), _stream()),
               "update_combine_bwd")
    return gq, gUv, gVv


def update_norm_bwd(x, Vv, gx, g_s, gVv, residual):
    """in place on gVv; returns gs_in"""
    _need_cuda(x)
    lib = _lib.load()
    N, _, F = Vv.shape
    gs_in = torch.empty((N, F), dtype=torch.float32, device=x.device)
    if not gVv.is_contiguous():                      # column half of a [N, 3, 2F] tensor (update_combine_bwd(cat=True))
        _lib.check(lib.cgvae_update_norm_bwd_ld(_p(x), _p(Vv), _p(gx), _p(g_s), N, F, int(bool(residual)), _p(gs_in), _p(gVv),
                                                gVv.stride(1), _stream()), "update_norm_bwd_ld")
        return gs_in
    _lib.check(lib.cgvae_update_norm_bwd(_p(x), _p(Vv), _p(gx), _p(g_s), N, F, int(bool(residual)), _p(gs_in), _p(gVv), _stream()),
               "update_norm_bwd")
    return gs_in


def segment_reduce_fwd(X, seg, mean, param=None):
    _need_cuda(X)
    lib = _lib.load()
    X = _f32(X)
    W = int(np.prod(X.shape[1:]))
    shape = (seg.n_beads,) + tuple(X.shape[1:])
    out = _grad_out(param, shape) if param is not None else torch.empty(shape, dtype=torch.float32, device=X.device)
    _lib.check(lib.cgvae_segment_reduce_fwd(_p(X), _p(seg.rowptr), _p(seg.atoms), seg.n_beads, W, int(bool(mean)), _p(out),
                                            _stream()), "segment_reduce_fwd")
    return out


def segment_reduce_bwd(g_out, seg, mean):
    _need_cuda(g_out)
    lib = _lib.load()
    g_out = _f32(g_out)
    W = int(np.prod(g_out.shape[1:]))
    g_X = torch.empty((seg.n,) + tuple(g_out.shape[1:]), dtype=torch.float32, device=g_out.device)
    _lib.check(lib.cgvae_segment_reduce_bwd(_p(g_out), _p(seg.mapping), _p(seg.rowptr), seg.n, W, int(bool(mean)), _p(g_X),
                                            _stream()), "segment_reduce_bwd")
    return g_X


def gather_rows(table, idx):
    _need_cuda(table, idx)
    lib = _lib.load()
    idx = idx.to(torch.int64).contiguous()
    W = table.shape[1]
    out = torch.empty((idx.shape[0], W), dtype=torch.float32, device=table.device)
    error_flags(table.device)
    _lib.check(lib.cgvae_gather_rows(_p(table), _p(idx), idx.shape[0], W, table.shape[0], _p(out), _stream()), "gather_rows")
    return out


def lift_fwd(V, cg_xyz, seg, mode, pin):
    _need_cuda(V, cg_xyz)
    lib = _lib.load()
    F = V.shape[-1]
    out = torch.empty((seg.n, 3), dtype=torch.float32, device=V.device)
    error_flags(V.device)
    _lib.check(lib.cgvae_lift_fwd(_p(V), _p(_f32(cg_xyz)), _p(seg.mapping), _p(seg.rank), _p(seg.rowptr), _p(seg.atoms), _p(pin),
                                  seg.n, seg.n_beads, F, mode, _p(out), _stream()), "lift_fwd")
    return out


def lift_bwd(g_xyz, seg, F, mode, pin):
    _need_cuda(g_xyz)
    lib = _lib.load()
    g_V = torch.empty((seg.n_beads, 3, F), dtype=torch.float32, device=g_xyz.device)
    _lib.check(lib.cgvae_lift_bwd(_p(_f32(g_xyz)), _p(seg.mapping), _p(seg.rank), _p(seg.rowptr), _p(seg.atoms), _p(pin), seg.n,
                                  seg.n_beads, F, mode, _p(g_V), _stream()), "lift_bwd")
    return g_V


def vec_to_planar(v_nf3):
    _need_cuda(v_nf3)
    lib = _lib.load()
    v_nf3 = _f32(v_nf3)
    N, F, _ = v_nf3.shape
    out = torch.empty((N, 3, F), dtype=torch.float32, device=v_nf3.device)
    _lib.check(lib.cgvae_vec_to_planar(_p(v_nf3), N, F, _p(out), _stream()), "vec_to_planar")
    return out


def vec_from_planar(v_n3f):
    _need_cuda(v_n3f)
    lib = _lib.load()
    v_n3f = _f32(v_n3f)
    N, _, F = v_n3f.shape
    out = torch.empty((N, F, 3), dtype=torch.float32, device=v_n3f.device)
    _lib.check(lib.cgvae_vec_from_planar(_p(v_n3f), N, F, _p(out), _stream()), "vec_from_planar")
    return out


def adam_clip_step(p, g, m, v, step, max_norm, lr, betas=(0.9, 0.999), eps=1e-8, norm_out=None, grad_scale=1.0,
                   loss=None, loss_scale=1.0, loss_limit=float("inf"), skipped=None):
    """fused clip_grad_norm_ + Adam on flat buffers (cgvae_adam_clip_step); all tensors flat fp32 CUDA, `step` float [1];
    the gradients are taken as grad_scale * g (1/world after an all-reduce(sum)).  loss (device float [1], optional):
    the reference's skip guard (scripts/utils.py:145-148) -- the step is a no-op when loss*loss_scale is NaN or >=
    loss_limit (or the gradient norm is not finite); skipped (device float [1], optional) counts such steps."""
    _need_cuda(p, g, m, v, step)
    lib = _lib.load()
    ws_bytes = int(lib.cgvae_adam_ws_bytes())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    t0 = TIMER.begin("adam_clip") if TIMER is not None else None
    _lib.check(lib.cgvae_adam_clip_step(_p(p), _p(g), _p(m), _p(v), p.numel(), float(max_norm), float(grad_scale), float(lr), float(betas[0]),
                                        float(betas[1]), float(eps), _p(step), _p(norm_out), _p(loss), float(loss_scale),
                                        float(min(loss_limit, 3.0e38)), _p(skipped), _p(ws), ws_bytes, _stream()),
               "adam_clip_step")
    if t0 is not None:
        TIMER.end("adam_clip", t0, dict(n=p.numel()))


def set_pdl(on):
    """programmatic dependent launch on / off for subsequent launches; returns the previous setting."""
    return bool(_lib.load().cgvae_set_pdl(int(bool(on))))


MATMUL_PRECISIONS = ("highest", "high")


def set_matmul_precision(mode):
    """precision of the tensor-core contractions for every launch from now on; returns the previous mode.

    "highest" (the default): 3xTF32, fp32 parity.  "high": 1xTF32, operands rounded to nearest TF32 with fp32
    accumulation, within 4 * 2^-11 scale-relative per contraction.  It covers the tcgen05 GEMMs (>= 64 rows) and the
    filter of the tensor-core message forward; every other kernel stays fp32 in both modes.  Independent of
    torch.get_float32_matmul_precision().  CUDA graphs replay the kernels they were captured with."""
    if mode not in MATMUL_PRECISIONS:
        raise ValueError("matmul precision must be one of %s, got %r" % (MATMUL_PRECISIONS, mode))
    rc = _lib.load().cgvae_set_matmul_precision(MATMUL_PRECISIONS.index(mode))
    if rc < 0:
        _lib.check(rc, "set_matmul_precision")
    return MATMUL_PRECISIONS[rc]


def get_matmul_precision():
    """the current mode of set_matmul_precision: "highest" or "high"."""
    return MATMUL_PRECISIONS[_lib.load().cgvae_get_matmul_precision()]


@_contextlib.contextmanager
def matmul_precision(mode):
    """``with matmul_precision("high"): ...`` -- the mode inside the block, the previous one restored on exit (also on an
    exception)."""
    prev = set_matmul_precision(mode)
    try:
        yield
    finally:
        set_matmul_precision(prev)


def register_const_range(t):
    """declare a parameter buffer constant between optimiser steps (weight prefetch before the PDL dependency wait);
    None clears the table."""
    lib = _lib.load()
    if t is None:
        _lib.check(lib.cgvae_register_const_range(None, 0), "register_const_range")
    else:
        _lib.check(lib.cgvae_register_const_range(_p(t), t.numel() * t.element_size()), "register_const_range")


def register_const_params(module):
    """every CUDA parameter of a module whose weights are frozen (sampling)."""
    for p in module.parameters():
        if p.is_cuda:
            register_const_range(p.data)


def adam_ws(device):
    """workspace of the two-phase (sharded) optimiser: float [1028] = 1024 norm partials | loss | ticket | pad."""
    lib = _lib.load()
    return torch.zeros(int(lib.cgvae_adam_ws_bytes()) // 4, dtype=torch.float32, device=device)


def grad_sumsq(g, loss, ws):
    _need_cuda(g, ws)
    lib = _lib.load()
    _lib.check(lib.cgvae_grad_sumsq(_p(g), g.numel(), _p(loss), _p(ws), ws.numel() * 4, _stream()), "grad_sumsq")


def adam_apply(p, g, m, v, step, max_norm, lr, ws, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0, use_ws_loss=False, loss_scale=1.0,
               loss_limit=float("inf"), skipped=None):
    """phase 2 of the sharded optimiser: ws holds the all-reduced norm partials (and loss); p / g / m / v are this rank's slices."""
    _need_cuda(p, g, m, v, step, ws)
    lib = _lib.load()
    _lib.check(lib.cgvae_adam_apply(_p(p), _p(g), _p(m), _p(v), p.numel(), float(max_norm), float(grad_scale), float(lr), float(betas[0]),
                                    float(betas[1]), float(eps), _p(step), None, int(bool(use_ws_loss)), float(loss_scale),
                                    float(min(loss_limit, 3.0e38)), _p(skipped), _p(ws), ws.numel() * 4, _stream()), "adam_apply")


# --------------------------------------------------------------------------------------------------
# VAE latent, prior std, fused training loss (csrc/loss.cu)
# --------------------------------------------------------------------------------------------------

def fill(shape, value, like):
    """torch.full(shape, value) on ``like``'s device through the library's own fill kernel (initial decoder state, cgvae.py:90-95)."""
    lib = _lib.load()
    _f32(like)
    out = torch.empty(shape, dtype=torch.float32, device=like.device)
    _need_cuda(out)
    _lib.check(lib.cgvae_fill(_p(out), out.numel(), float(value), _stream()), "fill")
    return out


def vae_latent_fwd(mu, logvar, eps):
    """(z, sigma): sigma = 1e-12 + exp(logvar/2), z = eps*sigma + mu (cgvae.py:445-449,500-507); eps None: sigma only."""
    _need_cuda(logvar)
    lib = _lib.load()
    logvar = _f32(logvar)
    sigma = torch.empty_like(logvar)
    z = torch.empty_like(logvar) if eps is not None else None
    _lib.check(lib.cgvae_vae_latent_fwd(_p(_f32(mu)) if eps is not None else None, _p(logvar), _p(_f32(eps)) if eps is not None else None,
                                        logvar.numel(), _p(sigma), _p(z), _stream()), "vae_latent_fwd")
    return z, sigma


def vae_latent_bwd(g_z, g_sigma, eps, sigma):
    lib = _lib.load()
    g_mu = torch.empty_like(sigma) if g_z is not None else None
    g_logvar = torch.empty_like(sigma)
    _lib.check(lib.cgvae_vae_latent_bwd(_p(g_z), _p(g_sigma), _p(eps), _p(sigma), sigma.numel(), _p(g_mu), _p(g_logvar), _stream()),
               "vae_latent_bwd")
    return g_mu, g_logvar


def std_logvar_fwd(x, c):
    _need_cuda(x)
    lib = _lib.load()
    x = _f32(x)
    y = torch.empty_like(x)
    _lib.check(lib.cgvae_std_logvar_fwd(_p(x), x.numel(), float(c), _p(y), _stream()), "std_logvar_fwd")
    return y


def std_logvar_bwd(gy, y, c):
    lib = _lib.load()
    gx = torch.empty_like(y)
    _lib.check(lib.cgvae_std_logvar_bwd(_p(_f32(gy)), _p(y), y.numel(), float(c), _p(gx), _stream()), "std_logvar_bwd")
    return gx


def loss_fwd(xyz, xyz_rec, bond_graph, mu, sigma, pmu, pstd, norms, beta, gamma, out=None):
    """(loss, recon, kl, graph) as one float[4] tensor: scripts/utils.py:117-141 in two launches."""
    _need_cuda(xyz_rec)
    lib = _lib.load()
    dev = xyz_rec.device
    out4 = out if out is not None else torch.empty(4, dtype=torch.float32, device=dev)
    ws_bytes = int(lib.cgvae_loss_ws_bytes())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    n_beads, F = (mu.shape[0], mu.shape[1]) if mu is not None else (0, 0)
    _lib.check(lib.cgvae_loss_fwd(_p(xyz), _p(xyz_rec), xyz_rec.shape[0], _p(bond_graph.rowptr) if bond_graph is not None else None,
                                  _p(bond_graph.col) if bond_graph is not None else None, _p(mu), _p(sigma), _p(pmu), _p(pstd),
                                  n_beads, F, _p(norms), float(beta), float(gamma), _p(out4), _p(ws), ws_bytes, _stream()), "loss_fwd")
    return out4


def loss_bwd(g_loss, xyz, xyz_rec, bond_graph, mu, sigma, pmu, pstd, norms, beta, gamma):
    lib = _lib.load()
    g_rec = torch.empty_like(xyz_rec)
    g_mu = torch.empty_like(mu) if mu is not None else None
    g_sigma = torch.empty_like(mu) if mu is not None else None
    g_pmu = torch.empty_like(pmu) if pmu is not None else None
    g_pstd = torch.empty_like(pmu) if pmu is not None else None
    n_beads, F = (mu.shape[0], mu.shape[1]) if mu is not None else (0, 0)
    _lib.check(lib.cgvae_loss_bwd(_p(g_loss), _p(xyz), _p(xyz_rec), xyz_rec.shape[0], _p(bond_graph.rowptr) if bond_graph is not None else None,
                                  _p(bond_graph.col) if bond_graph is not None else None, _p(mu), _p(sigma), _p(pmu), _p(pstd), n_beads,
                                  F, _p(norms), float(beta), float(gamma), _p(g_rec), _p(g_mu), _p(g_sigma), _p(g_pmu), _p(g_pstd),
                                  _stream()), "loss_bwd")
    return g_rec, g_mu, g_sigma, g_pmu, g_pstd


def loss_bwd_target(g_loss, xyz, xyz_rec, bond_graph, norms, gamma):
    """gradient of the training loss to its target coordinates xyz [n_atoms,3]"""
    lib = _lib.load()
    g_xyz = torch.empty_like(xyz)
    _lib.check(lib.cgvae_loss_bwd_target(_p(g_loss), _p(xyz), _p(xyz_rec), xyz.shape[0],
                                         _p(bond_graph.rowptr) if bond_graph is not None else None,
                                         _p(bond_graph.col) if bond_graph is not None else None, _p(norms), float(gamma), _p(g_xyz),
                                         _stream()), "loss_bwd_target")
    return g_xyz


def pin_mask(idx, n_atoms, count=None):
    """uint8 [n_atoms] mask of the PCN C-alpha re-anchoring (cgvae.py:569-571), predicate evaluated on the device."""
    _need_cuda(idx)
    lib = _lib.load()
    idx = idx.to(torch.int64).contiguous()
    nbytes = (n_atoms + 3) // 4 * 4
    buf = torch.empty(max(nbytes, 4), dtype=torch.uint8, device=idx.device)
    error_flags(idx.device)
    _lib.check(lib.cgvae_pin_mask(_p(idx), idx.numel(), _p(count), n_atoms, _p(buf), buf.numel(), _stream()), "pin_mask")
    return buf[:n_atoms]


def dihedral_loss_fwd(xyz, xyz_rec, idx, count=None, norm=None):
    """(loss [1], contrib [D,4,3]): scripts/pcn_utils.py:114-132,178-180."""
    _need_cuda(xyz_rec)
    lib = _lib.load()
    idx = idx.to(torch.int64).contiguous()
    D = idx.shape[0]
    dev = xyz_rec.device
    contrib = torch.empty((D, 4, 3), dtype=torch.float32, device=dev)
    out = torch.empty(1, dtype=torch.float32, device=dev)
    ws = torch.empty(256, dtype=torch.float32, device=dev)
    _lib.check(lib.cgvae_dihedral_loss_fwd(_p(_f32(xyz)), _p(_f32(xyz_rec)), _p(idx), D, _p(count), _p(norm), _p(contrib), _p(out),
                                           _p(ws), 1024, _stream()), "dihedral_loss_fwd")
    return out, contrib


def dihedral_loss_bwd(g_loss, contrib, graph, n_atoms, count=None, norm=None):
    lib = _lib.load()
    g = torch.empty((n_atoms, 3), dtype=torch.float32, device=contrib.device)
    _lib.check(lib.cgvae_dihedral_loss_bwd(_p(g_loss), _p(contrib), _p(graph.rowptr), _p(graph.col), n_atoms, contrib.shape[0],
                                           _p(count), _p(norm), _p(g), _stream()), "dihedral_loss_bwd")
    return g


# --------------------------------------------------------------------------------------------------
# ragged batch collation (csrc/collate.cu)
# --------------------------------------------------------------------------------------------------

COLLATE_KINDS = 6          # atoms, residues, bonds, C-alpha edges, dihedrals, C-alpha indices (CGVAE_COLLATE_*)
COLLATE_MAX_OUT = 8


class _CollateOut(ctypes.Structure):
    _fields_ = [("dst", ctypes.c_void_p), ("src", ctypes.c_void_p), ("rows", ctypes.c_int64), ("width", ctypes.c_int32),
                ("elem_bytes", ctypes.c_int32), ("kind", ctypes.c_int32), ("add_kind", ctypes.c_int32),
                ("pad_beads", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class CollatePlan(ctypes.Structure):
    """struct cgvae_collate_plan of include/cgvae_b200.h."""
    _fields_ = [("idx", ctypes.c_void_p), ("item_ptr", ctypes.c_void_p), ("slot_off", ctypes.c_void_p),
                ("counts", ctypes.c_void_p), ("count_out", ctypes.c_void_p * COLLATE_KINDS), ("norms", ctypes.c_void_p),
                ("n_slots", ctypes.c_int64), ("n_items", ctypes.c_int64), ("atoms_per_bead", ctypes.c_int64),
                ("n_beads", ctypes.c_int64), ("live_cap", ctypes.c_int64 * COLLATE_KINDS), ("n_out", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("out", _CollateOut * COLLATE_MAX_OUT)]


def collate(idx, item_ptr, outputs, live_cap, atoms_per_bead=1, n_beads=0, count_out=None, norms=None):
    """cgvae_collate: gather the rows of the items ``idx`` (int64 [B] CUDA, -1 = empty slot) from ragged stores into
    fixed-size outputs.  item_ptr: int64 [KINDS, n_items+1] CUDA row offsets of every item in every kind's store.
    outputs: list of (dst, src, kind, add_kind or None, pad_beads) with dst [rows] / [rows, width] and src the kind's store
    of the same dtype and width.  live_cap: KINDS ints.  count_out: KINDS int64 [1] tensors or None; norms: float [3] or None.
    Returns the live counts (int64 [KINDS], CUDA).  Two launches, no host synchronisation."""
    _need_cuda(idx, item_ptr)
    lib = _lib.load()
    dev = idx.device
    if idx.dtype != torch.int64 or not idx.is_contiguous() or not item_ptr.is_contiguous():
        raise ValueError("collate: idx / item_ptr must be contiguous int64")
    B = idx.shape[0]
    slot_off = torch.empty(COLLATE_KINDS * (B + 1), dtype=torch.int64, device=dev)
    counts = torch.empty(COLLATE_KINDS, dtype=torch.int64, device=dev)
    plan = CollatePlan()
    plan.idx, plan.item_ptr, plan.slot_off, plan.counts = _p(idx), _p(item_ptr), _p(slot_off), _p(counts)
    for k, t in enumerate(count_out or ()):
        plan.count_out[k] = _p(t)
    plan.norms = _p(norms)
    plan.n_slots, plan.n_items = B, item_ptr.shape[1] - 1
    plan.atoms_per_bead, plan.n_beads = int(atoms_per_bead), int(n_beads)
    for k, c in enumerate(live_cap):
        plan.live_cap[k] = int(c)
    if len(outputs) > COLLATE_MAX_OUT:
        raise ValueError("collate: at most %d outputs" % COLLATE_MAX_OUT)
    plan.n_out = len(outputs)
    for i, (dst, src, kind, add_kind, pad_beads) in enumerate(outputs):
        _need_cuda(dst, src)
        width = dst.shape[1] if dst.dim() == 2 else 1
        if not (dst.is_contiguous() and src.is_contiguous()) or dst.dtype != src.dtype or \
                (src.shape[1] if src.dim() == 2 else 1) != width or dst.dtype not in (torch.float32, torch.int64):
            raise ValueError("collate: output %d: dst / src must be contiguous float32 or int64 of the same width" % i)
        o = plan.out[i]
        o.dst, o.src, o.rows, o.width, o.elem_bytes = _p(dst), _p(src), dst.shape[0], width, dst.element_size()
        o.kind, o.add_kind, o.pad_beads = int(kind), -1 if add_kind is None else int(add_kind), int(bool(pad_beads))
    error_flags(dev)
    _lib.check(lib.cgvae_collate(ctypes.byref(plan), _stream()), "collate")
    return counts
