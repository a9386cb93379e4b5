"""Training / sampling steps around the hot path: the loss assembly and optimiser step of
scripts/utils.py:81-157 and the ensemble loop of scripts/sampling.py:252-284 of the reference, kept on
the device with no host round trips except the loss read the reference also does.

The model forward / backward runs in the sm_100a kernels; the loss terms, gradient clipping and Adam
are small element-wise / reduction passes (SURVEY.md section 8f lists their fusion as the next step) and use
torch device ops on a single flat gradient buffer.
"""
import torch

EPS = 1e-6          # scripts/utils.py:27


def kl_divergence(mu1, std1, mu2, std2):
    """scripts/utils.py:81-86 -- note the reference divides (mu1-mu2)^2 by std2, not std2^2; kept.  Without a prior
    network (``mu2 is None``) the reference falls back to the KL against the standard normal (:82-83)."""
    if mu2 is None:
        return -0.5 * torch.sum(1 + torch.log(std1.pow(2)) - mu1.pow(2) - std1.pow(2), dim=-1).mean()
    return 0.5 * ((std1.pow(2) / std2.pow(2)).sum(-1) + ((mu1 - mu2).pow(2) / std2).sum(-1)
                  + torch.log(std2.pow(2)).sum(-1) - torch.log(std1.pow(2)).sum(-1) - std1.shape[-1]).mean()


def training_loss(outputs, xyz, bond_edge_list, beta, gamma, bond_count=None, norms=None):
    """scripts/utils.py:117-141: MSE + beta*KL + gamma*bond-graph loss, all on the device (the reference moves the
    edge list and the target coordinates to the CPU first: utils.py:127-128).  ``bond_count`` (device scalar): number of
    live rows of a zero-padded static-capacity ``bond_edge_list`` -- padded (0, 0) rows contribute exactly 0 to the sum.
    ``norms`` (device float [3], data-parallel training): the denominators (atoms, beads, bonds) of the three means as
    GLOBAL count / world, so that the mean over ranks of the local losses (and gradients) equals the single-process
    ``mean()`` over the global batch even when the ranks hold different numbers of atoms / bonds (SURVEY.md section 8e)."""
    mu, sigma, pmu, pstd, _, xyz_recon = outputs
    if xyz_recon.is_cuda and FUSED_LOSS:
        return _training_loss_fused(outputs, xyz, bond_edge_list, beta, gamma, bond_count, norms)
    if norms is None:
        recon = (xyz_recon - xyz).pow(2).mean()
    else:
        recon = (xyz_recon - xyz).pow(2).sum() / (3.0 * norms[0])
    loss = recon
    kl = graph = None
    if mu is not None:
        kl = kl_divergence(mu, sigma, pmu, pstd)
        if norms is not None:
            kl = kl * (mu.shape[0] / norms[1])
        loss = loss + kl * beta
    if gamma != 0.0:
        a, b = bond_edge_list[:, 0], bond_edge_list[:, 1]
        gen = ((xyz_recon[a] - xyz_recon[b]).pow(2).sum(-1) + EPS).sqrt()
        dat = ((xyz[a] - xyz[b]).pow(2).sum(-1) + EPS).sqrt()
        if norms is not None:
            graph = (gen - dat).pow(2).sum() / norms[2]
        elif bond_count is None:
            graph = (gen - dat).pow(2).mean()
        else:
            graph = (gen - dat).pow(2).sum() / bond_count.to(gen.dtype).reshape(())
        loss = loss + graph * gamma
    return loss, recon, kl, graph


FUSED_LOSS = True   # CUDA tensors: csrc/loss.cu (2 launches forward, 2 backward); False keeps the torch expression above


def _training_loss_fused(outputs, xyz, bond_edge_list, beta, gamma, bond_count, norms):
    """The same loss through functions.TrainingLoss: the bond term walks the receiver CSR of the symmetrised bond list
    (built with the graph kernels, live count taken from ``bond_count`` in static-capacity mode), so neither direction
    needs an index_put or a host-visible size."""
    from . import functions, ops
    mu, sigma, pmu, pstd, _, xyz_recon = outputs
    n_atoms = xyz_recon.shape[0]
    bond_graph = None
    if gamma != 0.0:
        bond_graph = ops.build_graph(bond_edge_list, n_atoms, symmetrize=True, n_edges_dev=bond_count)
    loss, comps = functions.TrainingLoss.apply(bond_graph, float(beta), float(gamma), norms, xyz, xyz_recon, mu, sigma, pmu, pstd)
    return loss, comps[1], (comps[2] if mu is not None else None), (comps[3] if gamma != 0.0 else None)


class FlatGrads(object):
    """One contiguous fp32 buffer holding the gradients of the parameters that actually receive one
    (two thirds of the reference's parameters are constructed and never used: SURVEY.md section 5).  On CUDA the
    buffer is registered as the gradient SINK of those parameters (ops.GRAD_SINK): the weight / bias / filter gradient
    kernels write straight into it and autograd adopts the views as ``p.grad`` -- no accumulate kernels, no zero fill,
    no flatten copy; the data-parallel all-reduce is ONE collective on ONE tensor and clipping is two passes over it.
    On CPU (tests) ``p.grad`` is pre-set to views and autograd accumulates in place."""

    def __init__(self, params, align=4):
        self.params = [p for p in params]
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device if self.params else "cpu"
        dtype = self.params[0].dtype if self.params else torch.float32
        # storage = [ gradients (n) | pad to 16 bytes | loss slot ]: the loss of the step rides at the tail so that the
        # data-parallel all-reduce of ``buffer`` also sums the per-rank losses -- the skip guard of the reference loop
        # (scripts/utils.py:145-148) is then decided on the SAME all-reduced value on every rank (SURVEY.md section 5)
        # align: 4 floats (16 bytes), or 4 * world for the sharded optimiser (equal 16-byte aligned slices per rank)
        pad = (-n) % align
        self.n_padded = n + pad
        self.buffer = torch.zeros(n + pad + 4, dtype=dtype, device=dev)
        self.flat = self.buffer[:n]
        self.loss_slot = self.buffer[n + pad:n + pad + 1]
        self.sink = self.flat.is_cuda
        self.views = []
        off = 0
        for p in self.params:
            self.views.append((off, p.numel()))
            if self.sink:
                from . import ops
                ops.GRAD_SINK[p.data_ptr()] = (self.flat, off)
                p.grad = None
            else:
                p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def zero_(self):
        if self.sink:
            for p in self.params:          # every region is fully overwritten by its kernel: nothing to clear
                p.grad = None
        else:
            self.flat.zero_()

    def check_adopted(self):
        """after a backward: every parameter's .grad must alias its region of the flat buffer."""
        base = self.flat.data_ptr()
        for p, (off, n) in zip(self.params, self.views):
            if p.grad is None or p.grad.data_ptr() != base + 4 * off:
                return False
        return True

    def release(self):
        if self.sink:
            from . import ops
            # the flat parameter buffer of this step may be freed next: forget every "constant weights" range (conservative:
            # a stale range would let a streaming GEMM prefetch an operand that IS written by the preceding kernel)
            ops.register_const_range(None)
            for p in self.params:
                ops.GRAD_SINK.pop(p.data_ptr(), None)

    def allreduce_mean_(self, group=None, scale_in_optimizer=False):
        """gradient exchange of data-parallel training: one all-reduce(sum) over NVLink, then 1/world -- applied here, or
        (scale_in_optimizer) left to the fused optimiser kernel, which takes the factor as an argument."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return
        world = dist.get_world_size(group)
        if world == 1:
            return
        dist.all_reduce(self.buffer, op=dist.ReduceOp.SUM, group=group)      # gradients + the loss slot
        if not scale_in_optimizer:
            self.buffer.mul_(1.0 / world)

    def clip_(self, max_norm):
        """torch.nn.utils.clip_grad_norm_ semantics (scripts/utils.py:156) on the flat buffer; returns the norm."""
        norm = torch.linalg.vector_norm(self.flat)
        coef = torch.clamp(max_norm / (norm + 1e-6), max=1.0)
        self.flat.mul_(coef)
        return norm


def used_parameters(model, run_backward):
    """names and parameters that receive a gradient in one backward pass (``run_backward()`` must do one)."""
    for p in model.parameters():
        p.grad = None
    run_backward()
    return [(k, p) for k, p in model.named_parameters() if p.grad is not None]


class TrainStep(object):
    """one optimisation step of scripts/utils.py::loop (train=True branch): forward, loss, backward, [all-reduce],
    clip_grad_norm_(0.01), Adam."""

    def __init__(self, model, beta, gamma, lr=1e-4, max_norm=0.01, group=None, capturable=False, optimizer="fused",
                 loss_limit="reference"):
        """optimizer: "fused" = cgvae_adam_clip_step on flat parameter / gradient / moment buffers (CUDA only; the used
        parameters are re-pointed at views of one contiguous buffer), "torch" = clip on the flat gradients +
        torch.optim.Adam (always used for CPU tensors).
        loss_limit: the skip guard of the reference loop -- a batch whose loss is NaN or >= loss_limit takes no optimiser
        step (scripts/utils.py:145-148); "reference" = gamma * 200, None disables it.  With the fused optimiser the
        decision is taken on the device (no host read, graph-capturable); ``skipped`` counts such steps."""
        self.model, self.beta, self.gamma = model, beta, gamma
        self.loss_limit = (gamma * 200.0) if loss_limit == "reference" else loss_limit
        self.skipped = None
        self.max_norm, self.group = max_norm, group
        self.lr = lr
        self.capturable = capturable
        self.optimizer = optimizer
        self.flat = None
        self.opt = None
        self.flat_p = self.exp_avg = self.exp_avg_sq = self.step_count = None
        import os
        self.defer_grads = os.environ.get("CGVAE_DEFER_WGRAD", "1") != "0"
        # data parallel: exchange the FACTORS of the deferred weight gradients (all-gather of ~20 MB) instead of the
        # gradients themselves (all-reduce of 222 MB at chignolin): dW = sum_r gy_r^T x_r is one contraction over the
        # rows of all ranks.  Needs the fused optimiser layout (deferred parameters at the end of the flat buffers).
        # Measured on 2 x B200 (tools/check_ddp.py): all-reduce 24 MB + all-gather 32 MB per rank instead of an all-reduce
        # of 270 MB, 3.99 vs 4.16 ms per step.  The gathered volume grows with the world size (8 ranks: 258 MB received,
        # 8x the rows in the grouped kernel) while a ring all-reduce does not, so "auto" enables it for 2 ranks only;
        # CGVAE_GATHER_FACTORS=1 / 0 forces / disables it.
        self.gather_factors = os.environ.get("CGVAE_GATHER_FACTORS", "auto")
        # data parallel, overlap: the decoder's parameters (83 % of the gradient bytes at chignolin) are laid out FIRST in the
        # flat buffers; a hook on the latent's gradient fires when the backward pass leaves the decoder, and their
        # all-reduce runs on a side stream while the encoder's backward (message + atom-level GEMM kernels) proceeds.
        # Measured on 2 x B200 (chignolin, graph replay, final build): plain all-reduce 3.39 ms per step, factor exchange
        # 3.24-3.32 ms (default for 2 ranks), sharded optimiser 3.40 ms; overlapped exchange 3.64 ms on an earlier build (the
        # NCCL kernel holds its SMs for the whole transfer and the encoder's backward slows down by more than the transfer
        # takes) -> overlap is opt-in (CGVAE_DP_OVERLAP=1).
        self.dp_overlap = os.environ.get("CGVAE_DP_OVERLAP", "0") == "1"
        # sharded optimiser: reduce-scatter of the flat gradient buffer, clip + Adam on this rank's 1/world slice (global norm
        # and loss from a 1025-float all-reduce), all-gather of the parameters: the 0.35 ms HBM-bound optimiser pass (28 B per
        # parameter) shrinks world-fold.  Measured (tools/nccl_micro.py, 270 MB): 2 x B200 all-reduce 543 us vs reduce-scatter
        # 347 + all-gather 321 us -> the pair costs what half an Adam pass saves (3.40 vs 3.39 ms per step); 8 x B200
        # all-reduce 723 us vs 407 + 406 us -> 3.58 vs 3.72 ms per step.  "auto" = from 4 ranks; CGVAE_SHARD_OPT=0 / 1 forces.
        self.shard_opt = os.environ.get("CGVAE_SHARD_OPT", "auto")
        self._adam_ws = None
        self.n_overlap = 0
        self._comm_stream = None
        self._scope = None
        self.n_reduce = None            # floats at the head of the flat gradient buffer that still need the all-reduce
        self._arena = self._gathered = self._factor_table = None
        self._factor_layout = None

    def _loss(self, batch, eps):
        out = self.model(batch, eps=eps) if eps is not None else self.model(batch)
        xyz = out[4]
        return training_loss(out, xyz, batch["bond_edge_list"], self.beta, self.gamma, batch.get("bond_count"),
                             batch.get("dp_norms"))[0]

    def update_dp_norms(self, batch):
        """data parallel: (atoms, beads, bonds) of the GLOBAL batch divided by the world size, all-reduced into
        ``batch['dp_norms']`` (a device float [3], updated in place when present so that a captured graph sees it)."""
        import torch.distributed as dist
        world = self._world()
        if world == 1:
            return batch
        if "atom_count" in batch:
            return self._update_dp_norms_live(batch, world)
        xyz = batch["nxyz"] if "nxyz" in batch else batch["xyz"]
        beads = batch["CG_nxyz"] if "CG_nxyz" in batch else batch["ca_xyz"]
        dev = xyz.device
        bonds = batch["bond_count"].to(torch.float32).reshape(1) if "bond_count" in batch else \
            torch.full((1,), float(batch["bond_edge_list"].shape[0]), device=dev)
        counts = torch.cat([torch.tensor([float(xyz.shape[0]), float(beads.shape[0])], device=dev), bonds.to(dev)])
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=self.group)
        counts = (counts / world).clamp_min(1.0)
        if "dp_norms" in batch:
            batch["dp_norms"].copy_(counts)
        else:
            batch["dp_norms"] = counts
        return batch

    def _update_dp_norms_live(self, batch, world):
        """capacity-padded batches (data.DeviceProteinDataset.collate(static=True)): all-reduce the LIVE counts (atoms,
        residues, bonds, dihedrals) on the device; ``dihe_norm`` (device float [1]) gets the global dihedral count / world,
        so that the dihedral term too is the mean over the global batch and not a mean of per-rank means."""
        import torch.distributed as dist
        dihe = batch["dihe_count"] if "dihe_count" in batch else torch.zeros_like(batch["atom_count"])
        counts = torch.cat([batch["atom_count"], batch["res_count"], batch["bond_count"], dihe]).to(torch.float32)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=self.group)
        counts = (counts / world).clamp_min(1.0)
        for key, val in (("dp_norms", counts[:3]), ("dihe_norm", counts[3:])):
            if key in batch:
                batch[key].copy_(val)
            else:
                batch[key] = val.clone()
        return batch

    def prepare(self, batch, eps=None):
        """discover the used parameters with one dry backward and lay their gradients out in one flat buffer."""
        used = used_parameters(self.model, lambda: self._loss(batch, eps).backward())
        params = [p for _, p in used]
        on_cuda = bool(params) and params[0].is_cuda
        want = self.gather_factors
        overlap_ok = (self.dp_overlap and on_cuda and self.optimizer == "fused" and self._world() > 1
                      and any(k.startswith("equivaraintconv.") for k, _ in used)
                      and any(not k.startswith("equivaraintconv.") for k, _ in used))
        want = (self._world() == 2 and not overlap_ok) if want == "auto" else (want not in ("0", False, None))
        self.gather_factors = bool(want and on_cuda and self.optimizer == "fused" and self.defer_grads and self._world() > 1)
        if self.gather_factors:
            params = self._deferred_last(params, batch, eps)
        elif overlap_ok:
            dec = [p for k, p in used if k.startswith("equivaraintconv.")]
            params = dec + [p for k, p in used if not k.startswith("equivaraintconv.")]
            self.n_overlap = sum(p.numel() for p in dec)
        world = self._world()
        want_shard = (world >= 4) if self.shard_opt == "auto" else (self.shard_opt not in ("0", False, None))
        self.shard_opt = bool(want_shard and on_cuda and self.optimizer == "fused" and world > 1
                              and not self.gather_factors and not self.n_overlap)
        align = 4 * world if self.shard_opt else 4
        if on_cuda and self.optimizer == "fused":
            # parameters of the used set become views of ONE buffer (same order as the gradient buffer): the optimiser
            # is then a single streaming pass.  Must happen before FlatGrads registers the sinks (keyed by data_ptr).
            n = sum(p.numel() for p in params)
            self.flat_p = torch.zeros(n + ((-n) % align if self.shard_opt else 0), dtype=torch.float32, device=params[0].device)
            off = 0
            for p in params:
                view = self.flat_p[off:off + p.numel()].view_as(p)
                view.copy_(p.data)
                p.data = view
                off += p.numel()
            n_moment = self.flat_p.numel() // world if self.shard_opt else self.flat_p.numel()    # sharded: this rank's slice
            self.exp_avg = torch.zeros(n_moment, dtype=torch.float32, device=params[0].device)
            self.exp_avg_sq = torch.zeros(n_moment, dtype=torch.float32, device=params[0].device)
            from . import ops
            ops.register_const_range(self.flat_p)      # weights are only written by the optimiser kernel (see gemm_stream.cu)
            self.step_count = torch.zeros(1, dtype=torch.float32, device=params[0].device)
            self.skipped = torch.zeros(1, dtype=torch.float32, device=params[0].device)
        self.flat = FlatGrads(params, align=align)
        fused = self.flat.flat.is_cuda
        if self.flat_p is None:
            self.opt = torch.optim.Adam(self.flat.params, lr=self.lr, fused=fused, capturable=bool(self.capturable and fused))
        if self.flat.sink:                 # verify once that autograd adopts the sink views (else fall back to copies)
            self.forward_backward(batch, eps)
            if not self.flat.check_adopted():
                raise RuntimeError("gradient sink views were not adopted by autograd")
        return [k for k, _ in used]

    def _deferred_last(self, params, batch, eps):
        """order the used parameters so that those whose gradients come from the deferred grouped launch sit at the END of
        the flat buffers: the head [0, n_reduce) is what the data-parallel all-reduce still has to cover."""
        from . import ops
        probe = FlatGrads(params)
        try:
            loss = self._loss(batch, eps)
            with ops.DeferredGrads(flush=False) as scope:
                loss.backward()
            base = probe.flat.data_ptr()
            deferred_offsets = set()
            for _, _, dW, db in scope.pending:
                for t in (dW, db):
                    if t is not None:
                        deferred_offsets.add((t.data_ptr() - base) // 4)
            head, tail = [], []
            for p, (off, _) in zip(probe.params, probe.views):
                (tail if off in deferred_offsets else head).append(p)
        finally:
            probe.release()
            for p in params:
                p.grad = None
        self.n_reduce = sum(p.numel() for p in head)
        return head + tail

    def forward_backward(self, batch, eps=None):
        self.flat.zero_()
        loss = self._loss(batch, eps)
        if self.flat.sink and self.defer_grads:
            from . import ops
            if self.gather_factors:        # recorded only: the factors are packed for the all-gather, the grouped
                with ops.DeferredGrads(flush=False) as scope:      # launch follows the exchange (apply_gradients)
                    loss.backward()
                self._pack_factors(scope.pending)
            else:
                with ops.DeferredGrads() as scope:  # small-graph weight / bias gradients: recorded, then ONE grouped launch
                    self._scope = scope
                    self._arm_overlap()
                    try:
                        loss.backward()
                    finally:
                        self._scope = None
                        self.model._latent_grad_hook = None
        else:
            loss.backward()
        with torch.no_grad():
            self.flat.loss_slot.copy_(loss.detach().reshape(1))     # read by the skip guard (after the all-reduce)
        return loss

    def _arm_overlap(self):
        self._overlapped = False
        if self.n_overlap and self._world() > 1 and getattr(self, "_exchange_follows", False):
            self.model._latent_grad_hook = self._on_decoder_done

    def _on_decoder_done(self, grad):
        """autograd hook on the latent's gradient: every decoder node has run (they were created after the latent, so the
        engine schedules them first).  Flush the deferred decoder weight gradients, then all-reduce the decoder block of
        the flat buffer on the communication stream; the encoder's backward continues on the compute stream."""
        import torch.distributed as dist
        if self._overlapped or self._scope is None:
            return None
        self._overlapped = True
        self._scope.flush_now()
        cur = torch.cuda.current_stream()
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream()
        self._comm_stream.wait_stream(cur)
        with torch.cuda.stream(self._comm_stream):
            dist.all_reduce(self.flat.buffer[:self.n_overlap], op=dist.ReduceOp.SUM, group=self.group)
        return None

    def _pack_factors(self, pending):
        """copy gy / x of every deferred problem into one contiguous arena (one torch.cat) in a fixed layout; on the first
        call allocate the arena, the all-gather destination and the problem table over the gathered rows."""
        import numpy as np
        from . import ops
        world = self._world()
        dev = self.flat.flat.device
        if getattr(self, "_pad", None) is None:
            self._pad = torch.zeros(4, dtype=torch.float32, device=dev)
        pieces, layout, off = [], [], 0

        def add(t):
            nonlocal off
            start = off
            pieces.append(t.detach().contiguous().view(-1))  # strided views (basis columns) are compacted here
            off += t.numel()
            if off % 4:                                      # keep every piece 16-byte aligned inside the arena
                pieces.append(self._pad[:4 - off % 4])
                off += 4 - off % 4
            return start

        for gy, x, dW, db in pending:
            rows, n_out = gy.shape
            n_in = x.shape[1] if x is not None else 0
            g_off = add(gy)
            x_off = add(x) if x is not None else 0
            layout.append((rows, n_out, n_in, g_off, x_off, dW.data_ptr() if dW is not None else 0,
                           db.data_ptr() if db is not None else 0))
        if self._factor_layout is None:
            self._factor_layout = layout
            L = off
            self._arena = torch.zeros(L, dtype=torch.float32, device=dev)
            self._gathered = torch.zeros(world * L, dtype=torch.float32, device=dev)
            table = np.zeros(len(layout), dtype=ops._wgrad_dtype())
            base = self._gathered.data_ptr()
            for i, (rows, n_out, n_in, g_off, x_off, dW_ptr, db_ptr) in enumerate(layout):
                table[i] = (base + 4 * g_off, (base + 4 * x_off) if n_in else 0, dW_ptr, db_ptr, rows * world, n_out, n_in,
                            n_out, n_in, rows, L, L)
            self._factor_table = table
            self._factor_out_floats = sum(n_out * n_in + n_out for _, n_out, n_in, _, _, _, _ in layout)
        elif layout != self._factor_layout:
            raise RuntimeError("deferred-gradient layout changed between steps (shapes must be static for data-parallel "
                               "factor exchange; set CGVAE_GATHER_FACTORS=0)")
        if pieces:
            with torch.no_grad():
                torch.cat(pieces, out=self._arena)           # one batched copy kernel per 128 pieces

    def _world(self):
        import torch.distributed as dist
        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def exchange_gradients(self):
        """data-parallel gradient mean; with the fused optimiser the 1/world factor is applied inside its kernel.  With
        factor exchange: all-reduce of the head of the gradient buffer + all-gather of the packed factors."""
        if self.gather_factors:
            import torch.distributed as dist
            if self.n_reduce:
                dist.all_reduce(self.flat.flat[:self.n_reduce], op=dist.ReduceOp.SUM, group=self.group)
            dist.all_reduce(self.flat.loss_slot, op=dist.ReduceOp.SUM, group=self.group)
            dist.all_gather_into_tensor(self._gathered, self._arena, group=self.group)
            return
        if self.shard_opt:
            import torch.distributed as dist
            cnt = self.flat.n_padded // self._world()
            r = dist.get_rank(self.group)
            dist.reduce_scatter_tensor(self.flat.buffer[r * cnt:(r + 1) * cnt], self.flat.buffer[:self.flat.n_padded],
                                       op=dist.ReduceOp.SUM, group=self.group)
            return
        if getattr(self, "_overlapped", False):
            # the decoder block is already in flight on the communication stream: reduce the rest (+ the loss slot), join
            import torch.distributed as dist
            self._overlapped = False
            dist.all_reduce(self.flat.buffer[self.n_overlap:], op=dist.ReduceOp.SUM, group=self.group)
            torch.cuda.current_stream().wait_stream(self._comm_stream)
            return
        self.flat.allreduce_mean_(self.group, scale_in_optimizer=self.flat_p is not None)

    def apply_gradients(self):
        if self.flat_p is not None:
            from . import ops
            if self.gather_factors:        # every rank forms the SUM over ranks of the deferred gradients itself
                ops.wgrad_grouped_table(self._factor_table, self._factor_out_floats)
            guard = self.loss_limit is not None
            if self.shard_opt:
                import torch.distributed as dist
                world, r = self._world(), dist.get_rank(self.group)
                cnt = self.flat.n_padded // world
                g_sl, p_sl = self.flat.buffer[r * cnt:(r + 1) * cnt], self.flat_p[r * cnt:(r + 1) * cnt]
                if self._adam_ws is None:
                    self._adam_ws = ops.adam_ws(self.flat_p.device)
                ops.grad_sumsq(g_sl, self.flat.loss_slot if guard else None, self._adam_ws)
                dist.all_reduce(self._adam_ws[:1025], op=dist.ReduceOp.SUM, group=self.group)     # global norm^2 partials + loss
                ops.adam_apply(p_sl, g_sl, self.exp_avg, self.exp_avg_sq, self.step_count, self.max_norm, self.lr, self._adam_ws,
                               grad_scale=1.0 / world, use_ws_loss=guard, loss_scale=1.0 / world,
                               loss_limit=self.loss_limit if guard else float("inf"), skipped=self.skipped)
                dist.all_gather_into_tensor(self.flat_p, p_sl, group=self.group)
                return
            ops.adam_clip_step(self.flat_p, self.flat.flat, self.exp_avg, self.exp_avg_sq, self.step_count, self.max_norm, self.lr,
                               grad_scale=1.0 / self._world(), loss=self.flat.loss_slot if guard else None,
                               loss_scale=1.0 / self._world(), loss_limit=self.loss_limit if guard else float("inf"),
                               skipped=self.skipped)
        else:
            # torch optimiser path (CPU tensors / optimizer="torch"): the guard is the reference's host read
            # (allreduce_mean_ has already turned the slot into the mean over ranks)
            if self.loss_limit is not None:
                l = float(self.flat.loss_slot.item())
                if l != l or l >= self.loss_limit:
                    self.n_skipped_host = getattr(self, "n_skipped_host", 0) + 1
                    return
            self.flat.clip_(self.max_norm)
            self.opt.step()

    def skipped_steps(self):
        """number of optimiser steps the skip guard suppressed so far (one host read)."""
        n = getattr(self, "n_skipped_host", 0)
        if self.skipped is not None:
            n += int(self.skipped.item())
        return n

    def step(self, batch, eps=None, train=True):
        """train=False: the validation branch of the reference loop (scripts/utils.py:159-160) -- forward, loss and
        backward (the reference calls loss.backward() there too), no gradient exchange and no optimiser step."""
        if self._world() > 1 and "dp_norms" not in batch and not torch.cuda.is_current_stream_capturing():
            batch = self.update_dp_norms(dict(batch))
        self._exchange_follows = bool(train)      # arms the overlapped all-reduce of the decoder block (data parallel)
        try:
            loss = self.forward_backward(batch, eps)
        finally:
            self._exchange_follows = False
        if train:
            self.exchange_gradients()
            self.apply_gradients()
        return loss


STATIC_LISTS = (("nbr_list", "nbr_count"), ("CG_nbr_list", "CG_nbr_count"), ("bond_edge_list", "bond_count"))


def compute_dihe(xyz, indices):
    """scripts/pcn_utils.py:114-132 (torch expression; CPU tensors and the float64 checks)."""
    b1 = xyz[indices[:, 1]] - xyz[indices[:, 0]]
    b2 = xyz[indices[:, 2]] - xyz[indices[:, 1]]
    b3 = xyz[indices[:, 3]] - xyz[indices[:, 2]]
    c1 = torch.linalg.cross(b2, b3)
    c2 = torch.linalg.cross(b1, b2)
    p1 = (b1 * c1).sum(-1) * ((b2 * b2).sum(-1) + EPS) ** 0.5
    p2 = (c1 * c2).sum(-1)
    return torch.arctan(p1 / (p2 + EPS))


def dihedral_loss(xyz_recon, xyz, dihe_idxs, count=None, norm=None):
    """loss_dihe of the PCN loop (scripts/pcn_utils.py:178-180): mean squared difference of the generated and the data
    dihedrals.  CUDA tensors: two launches forward, one backward (csrc/loss.cu)."""
    if xyz_recon.is_cuda and FUSED_LOSS:
        from . import functions
        return functions.DihedralLoss.apply(xyz, xyz_recon, dihe_idxs, count, norm)
    n = dihe_idxs.shape[0] if count is None else int(count)
    idx = dihe_idxs[:n]
    sq = (compute_dihe(xyz_recon, idx) - compute_dihe(xyz.detach(), idx)).pow(2)
    return sq.sum() / norm if norm is not None else sq.mean()


def to_static_pcn_batch(batch, capacities):
    """``to_static_batch`` for the PCN (run_pdb) batches: ``CG_nbr_list`` / ``bond_edge_list`` / ``dihe_idxs`` / ``ca_idx``
    zero-padded to fixed capacities with their live counts (``CG_nbr_count``, ``bond_count``, ``dihe_count``, ``ca_count``);
    python lists (``seq``) are dropped -- the decoder does not read them."""
    out = {k: v for k, v in batch.items() if torch.is_tensor(v)}
    for key, count_key, width in (("CG_nbr_list", "CG_nbr_count", 2), ("bond_edge_list", "bond_count", 2),
                                  ("dihe_idxs", "dihe_count", 4), ("ca_idx", "ca_count", 0)):
        if key not in batch:
            continue
        t = batch[key]
        cap, n = int(capacities[key]), int(t.shape[0])
        if n > cap:
            raise ValueError("%s has %d rows, capacity %d" % (key, n, cap))
        padded = torch.zeros((cap, width) if width else (cap,), dtype=torch.int64)
        padded[:n] = t
        out[key] = padded
        out[count_key] = torch.tensor([n], dtype=torch.int64)
        if key == "CG_nbr_list":
            up = bool((t[:, 0] > t[:, 1]).any()) if n else False
            down = bool((t[:, 1] > t[:, 0]).any()) if n else False
            out["CG_nbr_symmetrize"] = not (up and down)
    return out


class PCNTrainStep(TrainStep):
    """one optimisation step of the PCN loop (scripts/pcn_utils.py::loop): MSE + gamma * bond-graph loss + kappa *
    dihedral loss (the KL term is absent: PCN returns no latent), skip guard at gamma * 300 (pcn_utils.py:191), then
    clip_grad_norm_(0.01) + Adam as in the CGVAE loop.  Batches from ``to_static_pcn_batch`` make the step
    CUDA-graph-capturable (``GraphedTrainStep(PCNTrainStep(..., capturable=True), batch, None)``)."""

    def __init__(self, model, gamma, kappa=0.0, loss_limit="reference", **kw):
        TrainStep.__init__(self, model, 0.0, gamma, loss_limit=None, **kw)
        self.kappa = kappa
        self.loss_limit = (gamma * 300.0) if loss_limit == "reference" else loss_limit

    def _loss(self, batch, eps):
        out = self.model(batch)
        norms = batch.get("dp_norms")
        if norms is None and "atom_count" in batch:
            norms = batch["loss_norms"]          # capacity-padded batch: live (atoms, residues, bonds), not the padded shapes
        loss = training_loss(out, out[4], batch["bond_edge_list"], 0.0, self.gamma, batch.get("bond_count"), norms)[0]
        if self.kappa != 0.0 and "dihe_idxs" in batch:
            loss = loss + self.kappa * dihedral_loss(out[5], out[4], batch["dihe_idxs"], batch.get("dihe_count"),
                                                     batch.get("dihe_norm"))
        return loss


def to_static_batch(batch, capacities):
    """Pad the variable-length index lists of a collated batch to fixed capacities and add their live row counts
    (``nbr_count``, ``CG_nbr_count``, ``bond_count``: int64 [1]).  Host-side, once per batch at dataset-preparation time
    (the reference precomputes the lists themselves once per dataset: scripts/run_ala.py:64-67).  Every tensor of the
    result has a shape that depends only on (atoms, beads, capacities), which is what CUDA-graph replay needs."""
    out = dict(batch)
    for key, count_key in STATIC_LISTS:
        t = batch[key]
        cap = int(capacities[key])
        n = int(t.shape[0])
        if n > cap:
            raise ValueError("%s has %d rows, capacity %d" % (key, n, cap))
        padded = torch.zeros((cap, 2), dtype=torch.int64)
        padded[:n] = t
        out[key] = padded
        out[count_key] = torch.tensor([n], dtype=torch.int64)
        if key != "bond_edge_list":
            # the two host reads of make_directed (conv.py:12-13), taken here once per batch: the flipped half is only
            # generated for one-directional lists
            up = bool((t[:, 0] > t[:, 1]).any()) if n else False
            down = bool((t[:, 1] > t[:, 0]).any()) if n else False
            out[key.replace("_list", "_symmetrize")] = not (up and down)
    return out


def validate_batch(batch, n_basis=None):
    """Host-side index validation of a (static) batch -- what the device kernels would flag (ops.check_device_errors)
    and the reference raises as IndexError: mapping / edge-list ranges, atomic numbers inside the embedding table, and
    no bead with more atoms than feature channels (cgvae.py:473)."""
    def _cpu(t):
        return t.detach().cpu() if torch.is_tensor(t) else torch.as_tensor(t)
    if "CG_mapping" in batch:
        mapping = _cpu(batch["CG_mapping"]).long()
        n_beads = int(batch["CG_nxyz"].shape[0])
        n_atoms = int(batch["nxyz"].shape[0])
        if mapping.numel() and (int(mapping.min()) < 0 or int(mapping.max()) >= n_beads):
            raise IndexError("CG_mapping entry outside [0, %d)" % n_beads)
        if n_basis is not None and mapping.numel() and int(torch.bincount(mapping, minlength=n_beads).max()) > n_basis:
            raise IndexError("a bead holds more atoms than feature channels (%d) -- cg_v[mapping, CG2atomChannel], "
                             "cgvae.py:473" % n_basis)
        z = _cpu(batch["nxyz"])[:, 0]
        if z.numel() and (float(z.min()) < 0 or float(z.max()) >= 100):
            raise IndexError("atomic number outside the embedding table (nn.Embedding(100, F), cgvae.py:273)")
        for key, count_key, n in (("nbr_list", "nbr_count", n_atoms), ("CG_nbr_list", "CG_nbr_count", n_beads),
                                  ("bond_edge_list", "bond_count", n_atoms)):
            if key in batch:
                t = _cpu(batch[key])
                if count_key in batch:
                    t = t[:int(_cpu(batch[count_key]).reshape(-1)[0])]
                if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n):
                    raise IndexError("%s entry outside [0, %d)" % (key, n))


class GraphedTrainStep(object):
    """The whole optimisation step (CSR build, geometry, forward, loss, backward, [NCCL all-reduce], clip, Adam:
    ~550 kernel launches at the chignolin config) captured ONCE as a CUDA graph over static-capacity input buffers and
    replayed per batch -- the step is launch-bound on the host otherwise.  Batches must come from ``to_static_batch``
    with the capacities used at capture time."""

    def __init__(self, trainer, example_batch, eps):
        if not trainer.capturable:
            raise ValueError("TrainStep(capturable=True) required")
        self.trainer = trainer
        if trainer._world() > 1 and "dp_norms" not in example_batch:
            example_batch = trainer.update_dp_norms(dict(example_batch))
        # all input tensors live in ONE byte buffer (256-byte aligned slots): a batch packed on the host the same way
        # (``pack``) is loaded with a single copy instead of one launch per key (11 copies, ~10 us of host latency each)
        self.layout, off = [], 0
        for k, v in example_batch.items():
            if torch.is_tensor(v):
                nbytes = v.numel() * v.element_size()
                self.layout.append((k, off, nbytes, v.dtype, tuple(v.shape)))
                off += (nbytes + 255) // 256 * 256
        dev = next(v.device for v in example_batch.values() if torch.is_tensor(v))
        self.packed = torch.zeros(max(off, 256), dtype=torch.uint8, device=dev)
        self.static = dict(example_batch)
        for k, o, nbytes, dtype, shape in self.layout:
            view = self.packed[o:o + nbytes].view(dtype).view(shape)
            view.copy_(example_batch[k])
            self.static[k] = view
        self.eps = eps.clone() if eps is not None else None
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):                 # warm-up on a side stream, as graph capture requires
            for _ in range(3):
                trainer.step(self.static, self.eps)
        torch.cuda.synchronize()
        from . import ops
        import torch.distributed as dist
        self.distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size(trainer.group) > 1
        before = ops.launch_count()
        # the precision mode the kernels were captured with: a replay runs those kernels whatever the mode is later
        self.matmul_precision = ops.get_matmul_precision()
        self.graph = torch.cuda.CUDAGraph()
        self.opt_graph = None
        if not self.distributed or trainer.n_overlap:
            # one graph for the whole step.  Data parallel with overlap: the NCCL all-reduces are captured too -- the
            # decoder block on the communication stream (forked and joined inside the capture), the rest on the compute
            # stream (CGVAE_DP_OVERLAP=0: the two-graph form below with an eager all-reduce in between)
            with torch.cuda.graph(self.graph, stream=side):   # same stream as the warm-up: autograd's accumulate nodes match
                self.loss = trainer.step(self.static, self.eps)
        else:
            # data parallel: the NCCL all-reduce stays an ordinary stream operation between two graphs
            # (forward+backward | clip+Adam); collectives inside a capture depend on process-group internals
            with torch.cuda.graph(self.graph, stream=side):
                self.loss = trainer.forward_backward(self.static, self.eps)
            if not trainer.shard_opt:
                self.opt_graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.opt_graph, stream=side, pool=self.graph.pool()):
                    trainer.apply_gradients()
            # sharded optimiser: its three launches (norm partials, loss copy, update) sit between three collectives and
            # stay ordinary stream work; the host enqueues them while the forward/backward graph is still running
        cur.wait_stream(side)
        self.launches_per_step = ops.launch_count() - before

    def pack(self, batch, pin=False, device=None):
        """the batch as one uint8 tensor in the layout of the static input buffer (host-side, once per batch)."""
        for k, v in batch.items():
            if k.endswith("_symmetrize") and bool(v) != bool(self.static.get(k, True)):
                raise ValueError("%s differs from the captured graph (one-directional vs bidirectional edge list)" % k)
        out = torch.zeros(self.packed.numel(), dtype=torch.uint8, pin_memory=pin) if device is None else \
            torch.zeros(self.packed.numel(), dtype=torch.uint8, device=device)
        for k, o, nbytes, dtype, shape in self.layout:
            if k in ("dp_norms", "dihe_norm") and k not in batch:    # filled on the device by update_dp_norms before every replay
                continue
            v = batch[k]
            if tuple(v.shape) != shape or v.dtype != dtype:
                raise ValueError("%s: expected %s %s, got %s %s" % (k, dtype, shape, v.dtype, tuple(v.shape)))
            out[o:o + nbytes].view(dtype).view(shape).copy_(v)
        return out

    def load(self, batch):
        if torch.is_tensor(batch):                 # packed: one copy (H2D from pinned memory or D2D)
            self.packed.copy_(batch, non_blocking=True)
            return
        for k, v in batch.items():
            if torch.is_tensor(v):
                self.static[k].copy_(v, non_blocking=True)

    def step(self, batch):
        """batch: a dict from ``to_static_batch`` (one copy per key) or its ``pack``ed form (one copy)."""
        self.load(batch)
        if self.distributed:
            self.trainer.update_dp_norms(self.static)          # tiny all-reduce of the (atoms, beads, bonds) counts
        self.graph.replay()
        if self.opt_graph is not None:
            self.trainer.exchange_gradients()
            self.opt_graph.replay()
        elif self.distributed and not self.trainer.n_overlap:
            self.trainer.exchange_gradients()
            self.trainer.apply_gradients()
        return self.loss


@torch.no_grad()
def sample_ensemble_member(model, cg_xyz, CG_nbr_list, mapping, num_CGs, H_prior_mu, H_prior_sigma, eps, graphs=None):
    """scripts/sampling.py:276-279: H = mu + eps*sigma, then the decoder."""
    H = H_prior_mu + eps * H_prior_sigma
    return model.decoder(cg_xyz, CG_nbr_list, H, H, mapping, num_CGs, graphs=graphs)


@torch.no_grad()
def sample_single(model, batch, n_ensemble, eps_members=None, eps_recon=None, reconstruct=True):
    """``sample_single`` scripts/sampling.py:252-293 without its ASE bookkeeping: the prior once (:268), ``n_ensemble``
    members ``H = eps*sigma + mu`` -> ``model.decoder`` (:276-279), then one reconstruction forward ``model(batch)`` (:293).
    The noise is drawn with ``torch.randn_like`` in the reference's call order unless given (``eps_members
    [n_ensemble, Nc, F]``, ``eps_recon [Nc, F]``).  Returns (members [n_ensemble, N, 3], xyz_recon or None, mu, sigma)."""
    from .cgvae import BatchGraphs
    z, cg_z, xyz, cg_xyz, nbr, cg_nbr, mapping, num = model.get_inputs(batch)
    cg_xyz = cg_xyz.contiguous()
    graphs = BatchGraphs.for_batch(batch)
    mu, sigma = model.prior_net(cg_z, cg_xyz, cg_nbr, graphs=graphs)
    members = []
    for m in range(int(n_ensemble)):
        eps = torch.randn_like(sigma) if eps_members is None else eps_members[m]
        members.append(sample_ensemble_member(model, cg_xyz, cg_nbr, mapping, num, mu, sigma, eps, graphs=graphs))
    xyz_recon = None
    if reconstruct:
        batch2 = dict(batch)
        batch2["_graphs"] = graphs
        xyz_recon = model(batch2, eps=eps_recon)[5]
    return torch.stack(members), xyz_recon, mu, sigma


def sample_ensemble_sharded(model, batch, n_ensemble, eps_members, group=None):
    """Ensemble members sharded over the ranks of a process group (SURVEY.md section 8e; BASELINE config 3: 8 members on 8
    GPUs): member m runs on rank m % world, the prior is recomputed on every rank (cheaper than a broadcast), and the
    geometries ``[n_atoms, 3]`` are exchanged with ONE all_gather.  ``eps_members [n_ensemble, Nc, F]`` must be the same on
    every rank (rank 0's generator, replayed or broadcast by the caller): the result is then identical to
    ``sample_single`` on one device, member by member.  Returns xyz [n_ensemble, N, 3] on every rank."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return sample_single(model, batch, n_ensemble, eps_members, reconstruct=False)[0]
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n_ensemble = int(n_ensemble)
    per = (n_ensemble + world - 1) // world
    mine = [m for m in range(n_ensemble) if m % world == rank]
    n_atoms = int(batch["nxyz"].shape[0])
    local = torch.zeros((per, n_atoms, 3), dtype=torch.float32, device=batch["nxyz"].device)
    if mine:
        out = sample_single(model, batch, len(mine), eps_members[mine], reconstruct=False)[0]
        local[:len(mine)] = out
    gathered = torch.empty((world, per, n_atoms, 3), dtype=torch.float32, device=local.device)
    dist.all_gather_into_tensor(gathered, local, group=group)
    # member m = slot m // world of rank m % world
    idx_rank = torch.arange(n_ensemble, device=local.device) % world
    idx_slot = torch.arange(n_ensemble, device=local.device) // world
    return gathered[idx_rank, idx_slot]


class GraphedSampler(object):
    """Ensemble sampling of scripts/sampling.py:265-284 for one conformation shape as ONE CUDA graph: the prior once,
    then ``n_ensemble`` decoder passes H_m = mu + eps_m * sigma -> decoder.  Sampling is host-launch-bound when issued
    eagerly (~125 launches of a few microseconds per member); a replay costs one launch per conformation.  Inputs are
    static-capacity batches from ``to_static_batch`` (CG_nbr_list padded, live count on the device); the noise
    ``eps [n_ensemble, n_beads, F]`` is an input, so a fixed seed reproduces the reference's geometries member by member.
    Ensemble members of different conformations are independent: under torchrun each rank samples its own conformations
    (or members) with no exchange step."""

    def __del__(self):
        try:                                   # the model may be freed next: forget the "constant weights" ranges
            from . import ops
            ops.register_const_range(None)
        except Exception:
            pass

    def __init__(self, model, example_batch, n_ensemble):
        self.model, self.n_ensemble = model, int(n_ensemble)
        self.static = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in example_batch.items()}
        n_beads = self.static["CG_nxyz"].shape[0]
        F = model.atom_munet[0].weight.shape[1]
        dev = self.static["CG_nxyz"].device
        self.eps = torch.zeros((self.n_ensemble, n_beads, F), dtype=torch.float32, device=dev)
        # sampling never writes the weights: the streaming GEMMs may fetch them before their dependency wait (gemm_stream.cu).
        # A caller that updates the parameters afterwards (fine-tuning) clears the table with ops.register_const_range(None).
        from . import ops
        ops.register_const_params(model)
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(2):
                self._run()
        torch.cuda.synchronize()
        self.matmul_precision = ops.get_matmul_precision()      # replays keep the kernels of this mode
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self.out = self._run()
        cur.wait_stream(side)

    @torch.no_grad()
    def _run(self):
        from .cgvae import BatchGraphs
        m = self.model
        z, cg_z, xyz, cg_xyz, nbr, cg_nbr, mapping, num = m.get_inputs(self.static)
        cg_xyz = cg_xyz.contiguous()
        graphs = BatchGraphs(None, self.static.get("CG_nbr_count"), True, self.static.get("CG_nbr_symmetrize", True))
        mu, sigma = m.prior_net(cg_z, cg_xyz, cg_nbr, graphs=graphs)
        outs = [sample_ensemble_member(m, cg_xyz, cg_nbr, mapping, num, mu, sigma, self.eps[k], graphs=graphs)
                for k in range(self.n_ensemble)]
        return torch.stack(outs)

    def sample(self, batch, eps):
        """batch: static-capacity dict of one conformation batch; eps [n_ensemble, n_beads, F].  Returns the static output
        buffer xyz [n_ensemble, n_atoms, 3] (overwritten by the next call)."""
        for k, v in batch.items():
            if torch.is_tensor(v):
                self.static[k].copy_(v, non_blocking=True)
        self.eps.copy_(eps, non_blocking=True)
        self.graph.replay()
        return self.out



class ShardedGraphedSampler(object):
    """``GraphedSampler`` with the ensemble members sharded over the ranks of a process group (SURVEY.md section 8e, BASELINE
    config 3): member m runs on rank m % world, every rank replays ONE CUDA graph (the prior + its ceil(n_ensemble / world)
    members) per conformation, and the geometries are exchanged with one ``all_gather``.  ``eps [n_ensemble, n_beads, F]`` must be
    the same on every rank; the result equals ``GraphedSampler`` / ``sample_single`` on one device member by member."""

    def __init__(self, model, example_batch, n_ensemble, group=None):
        import torch.distributed as dist
        self.group = group
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.n_ensemble = int(n_ensemble)
        self.per = (self.n_ensemble + self.world - 1) // self.world
        self.mine = [m for m in range(self.n_ensemble) if m % self.world == self.rank]
        self.local = GraphedSampler(model, example_batch, self.per)
        self.matmul_precision = self.local.matmul_precision
        dev = self.local.eps.device
        self._eps_local = torch.zeros_like(self.local.eps)
        self._mine_idx = torch.tensor(self.mine, dtype=torch.int64, device=dev)
        n_atoms = int(self.local.out.shape[1])
        self._gathered = torch.empty((self.world, self.per, n_atoms, 3), dtype=torch.float32, device=dev)
        members = torch.arange(self.n_ensemble, device=dev)
        self._idx_rank, self._idx_slot = members % self.world, members // self.world

    def sample(self, batch, eps):
        import torch.distributed as dist
        if self.mine:
            self._eps_local[:len(self.mine)].copy_(eps.index_select(0, self._mine_idx))
        out = self.local.sample(batch, self._eps_local)
        if self.world == 1:
            return out[:self.n_ensemble]
        dist.all_gather_into_tensor(self._gathered, out.contiguous(), group=self.group)
        return self._gathered[self._idx_rank, self._idx_slot]          # member m = slot m // world of rank m % world
