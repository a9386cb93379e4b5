"""GPU (B200): the kernels every training step ends in, against float64 at the sizes the steps run.

  * clip + Adam (csrc/optim.cu): ``sumsq_partial_kernel`` + ``adam_clip_kernel`` in the one-launch form
    (``ops.adam_clip_step``) and in the sharded two-phase form of ``TrainStep.apply_gradients`` (``ops.grad_sumsq``, an
    all-reduce of the 1025-float workspace, ``ops.adam_apply`` on each rank's slice), emulated on one GPU;
  * the skip guard of both forms with 1184 blocks racing for the ticket;
  * the fused training loss (``loss_partial_kernel`` / ``loss_final_kernel`` / ``loss_bwd_*``) and the dihedral loss
    (csrc/loss.cu) at the c4 PCN batch and at KL / dihedral sizes where their loops run more than once.

``adam_clip_kernel`` caps its grid at 148 * 8 blocks of 256 threads with 4 elements each: one pass covers STRIDE
elements, and the c2 parameter count takes 128 passes.  ``loss_partial_kernel`` gives each of its 256 blocks
ceil(n / 256) atoms (500 at c4) and strides by 256 inside the slice.  ``test_step_tail_grids`` pins these grids, so that a
change of grid cap cannot quietly turn these tests back into single-pass tests.

The float64 references are the plain expressions written out below, evaluated on the device; the kernel's fp32 scalar
arguments (betas, lr, eps, max_norm) enter them at their fp32 values.  Run with ``-s`` to see the worst error of every
comparison.  Metric: max|a - b| / max|b| (tests.test_gpu_dense_paths._rel_err)."""
import functools
import math

import numpy as np
import pytest
import torch

from coarsegrainingvae_b200 import ops, synthetic, train
from coarsegrainingvae_b200.factory import build_cgvae
from tests.test_gpu_dense_paths import _probe, _rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
LOSS_TOL = 1e-5                        # the fused-loss rule of test_gpu_round2.py
# the update's error is mostly the kernel's fp32 bias correction: 1 - powf(0.999, t) rounded at t = 2..4 is off by
# up to 6.7e-6 relative, 3.3e-6 after the square root (5.3e-6 in all on a B200)
NORM_TOL, MOMENT_TOL, UPDATE_TOL = 1e-5, 1e-6, 1e-5
STRIDE = 148 * 8 * 256 * 4             # elements one pass of adam_clip_kernel's capped grid covers
LR, MAX_NORM, ADAM_EPS, BETAS = 1e-3, 0.01, 1e-8, (0.9, 0.999)
LOSS_LIMIT = 50.0 * 200.0              # the reference skip limit gamma * 200 at c2

# Adam steps: (clipped, grad_scale, step counter preset before the step)
SCHEDULE = [(True, 1.0, None), (False, 1.0, None), (True, 0.25, None), (False, 0.25, None), (True, 0.25, 10000.0)]

_WORST = {}


def _record(name, err):
    _WORST[name] = max(err, _WORST.get(name, 0.0))
    return err


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print()
    for name in sorted(_WORST):
        print("worst %-40s %.2e" % (name, _WORST[name]))


@functools.lru_cache(maxsize=None)
def _n(size):
    if size == "c2":           # every parameter build_cgvae constructs at the c2 widths (the step updates 67.5 M of them)
        cfg = synthetic.CONFIGS["c2_chignolin"]
        with torch.device("meta"):
            model = build_cgvae(cfg["n_basis"], cfg["n_rbf"], cfg["enc_nconv"], cfg["dec_nconv"], cfg["atom_cutoff"],
                                cfg["cg_cutoff"], cfg["n_cgs"])
        return sum(p.numel() for p in model.parameters())
    assert size == "2_strides_tail_3"          # a partial last pass, and a tail that is not a whole float4
    return 2 * STRIDE + 3


SIZES = ["c2", "2_strides_tail_3"]


def _f32(x):
    return float(np.float32(x))


def _cdiv(a, b):
    return -(-a // b)


def _grad(n, clipped, grad_scale, gen):
    """random gradients; unclipped: norm = grad_scale * |g| = max_norm / 2, so the clip coefficient is grad_scale.
    Clipped: |g| ~ sqrt(n), so every clipped element is ~ max_norm / sqrt(n) (1e-6 at c2) and eps stays visible."""
    g = torch.randn(n, device=DEV, generator=gen)
    if not clipped:
        g *= 0.5 * MAX_NORM / (grad_scale * float(g.double().norm()))
    return g


def _adam64(p, g, m, v, step, grad_scale):
    """clip_grad_norm_(max_norm) of grad_scale * g, then one Adam step, in float64 from the fp32 state before the step:
    (norm, m, v, p_new - p)."""
    b1, b2, lr, eps, max_norm, gs = map(_f32, (*BETAS, LR, ADAM_EPS, MAX_NORM, grad_scale))
    g64 = g.double()
    norm = gs * math.sqrt(float(g64.square().sum()))
    gg = g64 * (gs * min(max_norm / (norm + _f32(1e-6)), 1.0))
    m1 = b1 * m.double() + (1.0 - b1) * gg
    v1 = b2 * v.double() + (1.0 - b2) * gg.square()
    t = float(step) + 1.0
    upd = -(lr / (1.0 - b1 ** t)) * m1 / (v1.sqrt() / math.sqrt(1.0 - b2 ** t) + eps)
    return norm, m1, v1, upd


def _check_adam(tag, norm, m, v, p_new, p_old, ref):
    want_norm, m1, v1, upd = ref
    errs = {"norm": abs(norm - want_norm) / want_norm, "m": _rel_err(m, m1), "v": _rel_err(v, v1),
            "update": _rel_err(p_new.double() - p_old.double(), upd)}
    for k, e in errs.items():
        _record("%s %s" % (tag, k), e)
    assert errs["norm"] <= NORM_TOL and errs["m"] <= MOMENT_TOL and errs["v"] <= MOMENT_TOL and errs["update"] <= UPDATE_TOL, \
        (tag, errs)


class _Shards(object):
    """The sharded optimiser of TrainStep.apply_gradients on one GPU: rank r owns slice r of the padded flat buffers and
    has its own workspace, step counter and skip counter; the all-reduce of ws[:1025] (norm partials + loss) is a torch
    sum written back to every rank."""

    def __init__(self, world, n_pad):
        assert n_pad % (4 * world) == 0
        self.world, self.cnt = world, n_pad // world
        self.ws = [ops.adam_ws(DEV) for _ in range(world)]
        self.step = [torch.zeros(1, device=DEV) for _ in range(world)]
        self.skipped = [torch.zeros(1, device=DEV) for _ in range(world)]

    def apply(self, p, g, m, v, losses, grad_scale):
        """losses: device float [world], the per-rank loss slots; returns the all-reduced workspace head."""
        sl = [slice(r * self.cnt, (r + 1) * self.cnt) for r in range(self.world)]
        for r in range(self.world):
            ops.grad_sumsq(g[sl[r]], losses[r:r + 1], self.ws[r])
        total = torch.stack([w[:1025] for w in self.ws]).sum(0)
        for w in self.ws:
            w[:1025].copy_(total)
        for r in range(self.world):
            ops.adam_apply(p[sl[r]], g[sl[r]], m[sl[r]], v[sl[r]], self.step[r], MAX_NORM, LR, self.ws[r],
                           grad_scale=grad_scale, use_ws_loss=True, loss_scale=1.0 / self.world, loss_limit=LOSS_LIMIT,
                           skipped=self.skipped[r])
        return total


def _padded(n, world):
    return n + (-n) % (4 * world)


# ------------------------------------------------------------------------------------------ clip + Adam

@pytest.mark.parametrize("size", SIZES)
def test_clip_adam_matches_float64(size):
    """ops.adam_clip_step over SCHEDULE (clipped / unclipped, grad_scale 1 and 0.25, the step counter preset to 10 000):
    norm, m, v and the update against float64, and two runs from the same state bitwise identical."""
    n = _n(size)
    gen = torch.Generator(device=DEV).manual_seed(11)
    p0 = 1e-2 * torch.randn(n, device=DEV, generator=gen)
    runs = [[p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV), torch.zeros(1, device=DEV),
             torch.zeros(1, device=DEV)] for _ in range(2)]                         # p, m, v, step, norm
    for k, (clipped, gs, preset) in enumerate(SCHEDULE):
        g = _grad(n, clipped, gs, gen)
        if preset is not None:
            for r in runs:
                r[3].fill_(preset)
        p, m, v, step, norm = runs[0]
        t_want = float(step) + 1.0
        ref = _adam64(p, g, m, v, step, gs)
        p_old = p.clone()
        for r in runs:
            ops.adam_clip_step(r[0], g, r[1], r[2], r[3], MAX_NORM, LR, norm_out=r[4], grad_scale=gs)
        assert all(torch.equal(a, b) for a, b in zip(*runs)), (size, k)
        assert float(step) == t_want, (size, k)
        _check_adam("one-launch %s" % size, float(norm), m, v, p, p_old, ref)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("size", SIZES)
def test_sharded_clip_adam_matches_float64_and_one_launch(size, world):
    """grad_sumsq -> all-reduce -> adam_apply on world equal slices of one padded buffer: within the float64 tolerances,
    within the same tolerances of adam_clip_step on the same data, every rank's step counter the same."""
    n = _n(size)
    n_pad = _padded(n, world)
    gen = torch.Generator(device=DEV).manual_seed(world)
    p = torch.zeros(n_pad, device=DEV)
    p[:n] = 1e-2 * torch.randn(n, device=DEV, generator=gen)
    m, v, g = torch.zeros(n_pad, device=DEV), torch.zeros(n_pad, device=DEV), torch.zeros(n_pad, device=DEV)
    shards = _Shards(world, n_pad)
    losses = torch.full((world,), 1.5, device=DEV)
    for k, (clipped, gs, preset) in enumerate(SCHEDULE):
        g[:n] = _grad(n, clipped, gs, gen)
        if preset is not None:
            for s in shards.step:
                s.fill_(preset)
        ref = _adam64(p, g, m, v, shards.step[0], gs)
        p_old = p.clone()
        q, mq, vq, sq = (t.clone() for t in (p, m, v, shards.step[0]))
        total = shards.apply(p, g, m, v, losses, gs)
        norm = gs * math.sqrt(float(total[:1024].double().sum()))
        _check_adam("sharded %s" % size, norm, m, v, p, p_old, ref)
        # the one-launch form from the same state with the same gradients
        nq = torch.zeros(1, device=DEV)
        ops.adam_clip_step(q, g, mq, vq, sq, MAX_NORM, LR, norm_out=nq, grad_scale=gs)
        errs = {"norm": abs(norm - float(nq)) / float(nq), "m": _rel_err(m, mq), "v": _rel_err(v, vq),
                "update": _rel_err(p.double() - p_old.double(), q.double() - p_old.double())}
        for key, e in errs.items():
            _record("sharded vs one-launch %s" % key, e)
        assert errs["norm"] <= NORM_TOL and errs["m"] <= MOMENT_TOL and errs["v"] <= MOMENT_TOL and \
            errs["update"] <= UPDATE_TOL, (size, world, k, errs)
        assert all(torch.equal(s, sq) for s in shards.step), (size, world, k)
        assert all(float(s) == 0.0 for s in shards.skipped)
    assert float(shards.step[0]) == 10001.0


# ------------------------------------------------------------------------------------------ skip guard

@pytest.mark.parametrize("form", ["one_launch", "sharded"])
def test_skip_guard_at_size(form):
    """NaN loss, loss at the limit (after loss_scale = 1/world), one inf and one NaN gradient entry: p / m / v / step
    bitwise unchanged, skipped +1.0 per launch (per rank); the next good step equals the same step without the skipped
    launches before it, bit for bit."""
    world, n = 4, _n("2_strides_tail_3")
    n_pad = _padded(n, world)
    gen = torch.Generator(device=DEV).manual_seed(7)
    p0 = torch.zeros(n_pad, device=DEV)
    p0[:n] = 1e-2 * torch.randn(n, device=DEV, generator=gen)
    warm = [torch.zeros(n_pad, device=DEV) for _ in range(2)]
    for k in range(2):
        warm[k][:n] = _grad(n, k == 0, 1.0 / world, gen)
    good = torch.zeros(n_pad, device=DEV)
    good[:n] = _grad(n, True, 1.0 / world, gen)
    L = np.float32(LOSS_LIMIT)
    below = np.float32(2 * L) - np.spacing(np.float32(4 * L))   # rank sums stay exact: 4L - ulp(4L), below the limit
    rank_losses = {"ok": [L / 2] * world, "good": [below, 2 * L, 0, 0], "nan_loss": [np.nan, L, L, L],
                   "loss_at_limit": [L / 2, 3 * L / 2, L, L]}

    class Run(object):
        def __init__(self):
            self.p, self.m, self.v = p0.clone(), torch.zeros(n_pad, device=DEV), torch.zeros(n_pad, device=DEV)
            if form == "sharded":
                self.shards = _Shards(world, n_pad)
                self.steps, self.skips = self.shards.step, self.shards.skipped
            else:
                self.steps, self.skips = [torch.zeros(1, device=DEV)], [torch.zeros(1, device=DEV)]

        def apply(self, g, key):
            losses = torch.tensor(rank_losses[key], dtype=torch.float32, device=DEV)
            if form == "sharded":
                self.shards.apply(self.p, g, self.m, self.v, losses, 1.0 / world)
            else:
                ops.adam_clip_step(self.p, g, self.m, self.v, self.steps[0], MAX_NORM, LR, grad_scale=1.0 / world,
                                   loss=losses.sum().reshape(1), loss_scale=1.0 / world, loss_limit=LOSS_LIMIT,
                                   skipped=self.skips[0])

        def state(self):
            return [self.p, self.m, self.v] + self.steps

    a, b = Run(), Run()
    for r in (a, b):
        for g in warm:
            r.apply(g, "ok")
    assert all(torch.equal(x, y) for x, y in zip(a.state(), b.state()))
    assert float(a.m.abs().max()) > 0 and all(float(s) == 2.0 for s in a.steps)
    before = [t.clone() for t in a.state()]
    bad_inf, bad_nan = good.clone(), good.clone()
    bad_inf[n - 1] = float("inf")              # the last element: the last rank's slice
    bad_nan[STRIDE + 5] = float("nan")         # the second pass of the one-launch grid, rank 2's slice
    cases = [("nan_loss", good, "nan_loss"), ("loss_at_limit", good, "loss_at_limit"), ("inf_grad", bad_inf, "ok"),
             ("nan_grad", bad_nan, "ok")]
    for k, (name, g, loss_key) in enumerate(cases):
        a.apply(g, loss_key)
        assert all(torch.equal(x, y) for x, y in zip(a.state(), before)), (form, name)
        assert all(float(s) == k + 1.0 for s in a.skips), (form, name, [float(s) for s in a.skips])
    for r in (a, b):
        r.apply(good, "good")
    assert all(torch.equal(x, y) for x, y in zip(a.state(), b.state())), form
    assert all(float(s) == 3.0 for s in a.steps) and all(float(s) == 0.0 for s in b.skips)
    assert not torch.equal(a.p, before[0])


# ------------------------------------------------------------------------------------------ fused training loss

@pytest.fixture(scope="module")
def c4():
    """the c4 PCN batch: 64 proteins, 128 000 atoms, 255 744 bonds, 31 872 dihedral quadruples (its bead graph is not
    used here)."""
    b = synthetic.pcn_batch(synthetic.CONFIGS["c4_protein"], 0, lambda xyz, cutoff: np.zeros((0, 2), np.int64))
    xyz, bonds, dihe = b["xyz"].to(DEV), b["bond_edge_list"].to(DEV), b["dihe_idxs"].to(DEV)
    assert (xyz.shape[0], bonds.shape[0], dihe.shape[0]) == (128000, 255744, 31872)
    rec = xyz + 0.3 * torch.randn(xyz.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    return xyz, rec, bonds, dihe


def _training_loss(fused, dtype, xyz, rec, bonds, mu, sigma, pmu, pstd, beta, gamma, bond_count=None):
    """train.training_loss, fused (csrc/loss.cu) or the torch expression, and the gradients of (1.7 * loss) to
    rec, mu, sigma and the prior mean / std."""
    old = train.FUSED_LOSS
    train.FUSED_LOSS = fused
    try:
        leaves = [t.detach().to(dtype).requires_grad_(True) if t is not None else None for t in (rec, mu, sigma, pmu, pstd)]
        out = (leaves[1], leaves[2], leaves[3], leaves[4], None, leaves[0])
        values = train.training_loss(out, xyz.to(dtype), bonds, beta, gamma, bond_count=bond_count)
        (values[0] * 1.7).backward()
        return [t.detach() if t is not None else None for t in values], [t.grad if t is not None else None for t in leaves]
    finally:
        train.FUSED_LOSS = old


def _check_loss(tag, got, want):
    (got_v, got_g), (want_v, want_g) = got, want
    for name, a, b in zip(("loss", "recon", "kl", "graph", "g_rec", "g_mu", "g_sigma", "g_pmu", "g_pstd"), got_v + got_g,
                          want_v + want_g):
        assert (a is None) == (b is None), (tag, name)
        if a is not None:
            e = _record("%s %s" % (tag, name), _rel_err(a.reshape(-1), b.reshape(-1)))
            assert e <= LOSS_TOL, (tag, name, e)


def _assert_bitwise(tag, first, again):
    for a, b in zip(first[0] + first[1], again[0] + again[1]):
        assert (a is None and b is None) or torch.equal(a, b), tag


@pytest.mark.parametrize("bond_list", ["plain", "static_capacity"])
def test_fused_loss_at_c4_batch(c4, bond_list):
    """value and g_rec of the fused loss (no KL) at the c4 batch: 500 atoms per loss_partial block, two passes each; the
    static-capacity list is zero-padded with a device count."""
    xyz, rec, bonds, _ = c4
    beta, gamma = 0.0, 2.0
    bonds_in, count = bonds, None
    if bond_list == "static_capacity":
        bonds_in = torch.cat([bonds, torch.zeros(1000, 2, dtype=torch.int64, device=DEV)])
        count = torch.tensor(bonds.shape[0], dtype=torch.int64, device=DEV)
    got = _training_loss(True, torch.float32, xyz, rec, bonds_in, None, None, None, None, beta, gamma, count)
    want = _training_loss(False, torch.float64, xyz, rec, bonds, None, None, None, None, beta, gamma)
    _check_loss("c4 loss", got, want)
    _assert_bitwise(bond_list, got, _training_loss(True, torch.float32, xyz, rec, bonds_in, None, None, None, None, beta,
                                                   gamma, count))


@pytest.mark.parametrize("prior", [True, False])
def test_fused_loss_kl_beyond_one_pass(prior):
    """KL over n_beads * F = 384 * 600 = 230 400 latent entries (c1 at batch 128): 900 per loss_partial block, four
    passes; with a prior and against the standard normal, value and every gradient."""
    n_atoms, n_beads, F = 22 * 128, 3 * 128, 600
    g = torch.Generator(device=DEV).manual_seed(9)
    xyz = 2.0 * torch.randn(n_atoms, 3, device=DEV, generator=g)
    rec = xyz + 0.3 * torch.randn(n_atoms, 3, device=DEV, generator=g)
    a = torch.randint(0, n_atoms, (2 * n_atoms,), device=DEV, generator=g)
    bonds = torch.stack([a, (a + 1 + torch.randint(0, n_atoms - 1, a.shape, device=DEV, generator=g)) % n_atoms], 1)
    mu = torch.randn(n_beads, F, device=DEV, generator=g)
    sigma = 0.2 + torch.rand(n_beads, F, device=DEV, generator=g)
    pmu = torch.randn(n_beads, F, device=DEV, generator=g) if prior else None
    pstd = 0.2 + torch.rand(n_beads, F, device=DEV, generator=g) if prior else None
    args = (xyz, rec, bonds, mu, sigma, pmu, pstd, 0.05, 25.0)
    got = _training_loss(True, torch.float32, *args)
    _check_loss("kl loss", got, _training_loss(False, torch.float64, *args))
    _assert_bitwise(prior, got, _training_loss(True, torch.float32, *args))


def _dihedral_case(c4, form):
    """(idx given to the kernel, live quadruples, count, norm); "c4": 31 872 quadruples in a zero-padded list with a live
    count and a norm (125 blocks, one pass); "c4x3": the list three times (95 616 > 256 * 256: the grid-stride loop)."""
    _, _, _, q = c4
    if form == "c4":
        idx = torch.cat([q, torch.zeros(77, 4, dtype=torch.int64, device=DEV)])
        return idx, q, torch.tensor([q.shape[0]], dtype=torch.int64, device=DEV), torch.tensor([1.5 * q.shape[0]], device=DEV)
    q3 = q.repeat(3, 1)
    return q3, q3, None, None


@pytest.mark.parametrize("form", ["c4", "c4x3"])
def test_dihedral_loss_at_c4(c4, form):
    """train.dihedral_loss == the float64 compute_dihe expression: value and the gradient to the reconstruction."""
    xyz, rec, _, _ = c4
    idx, q, count, norm = _dihedral_case(c4, form)

    def run():
        r = rec.clone().requires_grad_(True)
        loss = train.dihedral_loss(r, xyz, idx, count=count, norm=norm)
        loss.backward()
        return [loss.detach()], [r.grad]

    got = run()
    r64 = rec.double().requires_grad_(True)
    sq = (train.compute_dihe(r64, q) - train.compute_dihe(xyz.double(), q)).pow(2)
    l64 = sq.sum() / float(norm) if norm is not None else sq.mean()
    l64.backward()
    for name, a, b in (("loss", got[0][0], l64.detach()), ("g_rec", got[1][0], r64.grad)):
        e = _record("dihedral %s" % name, _rel_err(a.reshape(-1), b.reshape(-1)))
        assert e <= LOSS_TOL, (form, name, e)
    _assert_bitwise(form, got, run())


# ------------------------------------------------------------------------------------------ which kernel ran

def test_step_tail_grids(c4):
    """In one profile: adam_clip_kernel at c2 size (one-launch, and one rank of 8 in the sharded form) with the capped
    1184-block grid, sumsq_partial_kernel with 1024 blocks, loss_partial_kernel with 256, dihedral_fwd_kernel with the
    grid cgvae_dihedral_loss_fwd computes; every loop the tests above rely on runs more than once at these grids."""
    n = _n("c2")
    world = 8
    n_pad = _padded(n, world)
    p, g, m, v = (torch.zeros(n_pad, device=DEV) for _ in range(4))
    step, ws = torch.zeros(2, device=DEV), ops.adam_ws(DEV)
    xyz, rec, bonds, _ = c4
    dihedral = [_dihedral_case(c4, form) for form in ("c4", "c4x3")]

    def run():
        ops.adam_clip_step(p, g, m, v, step[:1], MAX_NORM, LR)
        sl = slice(0, n_pad // world)
        ops.grad_sumsq(g[sl], None, ws)
        ops.adam_apply(p[sl], g[sl], m[sl], v[sl], step[1:], MAX_NORM, LR, ws, grad_scale=1.0 / world)
        train.training_loss((None, None, None, None, None, rec), xyz, bonds, 0.0, 2.0)
        for idx, _, count, norm in dihedral:
            train.dihedral_loss(rec, xyz, idx, count=count, norm=norm)

    def run_twice():
        run()
        torch.cuda.synchronize()
        run()

    # the profiler can miss the first launches of a session (seen after many earlier profiles in one process): the
    # sequence runs twice and its second pass must be complete
    _, launched = _probe(run_twice)
    names = ("sumsq_partial_kernel", "adam_clip_kernel", "loss_partial_kernel", "dihedral_fwd_kernel")
    got = [(k, grid) for k, grid, _ in launched if k in names]
    dihe_grids = [max(1, min(256, _cdiv(idx.shape[0], 256))) for idx, _, _, _ in dihedral]
    want = [("sumsq_partial_kernel", (1024, 1, 1)), ("adam_clip_kernel", (1184, 1, 1)),
            ("sumsq_partial_kernel", (1024, 1, 1)), ("adam_clip_kernel", (1184, 1, 1)),
            ("loss_partial_kernel", (256, 1, 1))] + [("dihedral_fwd_kernel", (b, 1, 1)) for b in dihe_grids]
    head = got[:len(got) - len(want)]                             # what the profile kept of the first pass
    assert len(want) <= len(got) <= 2 * len(want) and got[len(head):] == want, (got, launched)
    assert head == want[len(want) - len(head):], (got, launched)
    assert dihe_grids == [125, 256]
    # passes of each loop at these grids and the sizes the tests above use
    assert STRIDE == 1184 * 256 * 4
    assert _cdiv(n, STRIDE) == 128 and _cdiv(n_pad // world, STRIDE) == 16 and _cdiv(_n("2_strides_tail_3"), STRIDE) == 3
    assert _cdiv(_cdiv(xyz.shape[0], 256), 256) == 2              # loss_partial: atoms per block, 256 threads
    assert _cdiv(_cdiv(384 * 600, 256), 256) == 4                 # loss_partial: KL entries per block
    assert _cdiv(3 * c4[3].shape[0], 256 * 256) == 2              # dihedral_fwd: grid-stride passes of the c4x3 list
