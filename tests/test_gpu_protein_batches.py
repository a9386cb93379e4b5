"""GPU (B200): data.DeviceProteinDataset -- on-device collation of variable-length proteins (csrc/collate.cu) into the
unpadded batch of the host pipeline and into capacity-padded batches that one CUDA graph of the PCN step replays."""
import numpy as np
import pytest
import torch

from coarsegrainingvae_b200 import data, ops, train
from coarsegrainingvae_b200.factory import build_pcn
from oracle import cgvae_oracle as orc
from tests.golden_util import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
CUTOFF = 10.0
GAMMA, KAPPA = 2.0, 0.5
LIST_KEYS = ("bond_edge_list", "CG_nbr_list", "dihe_idxs", "ca_idx")
TENSOR_KEYS = ("xyz", "ca_xyz", "res", "cg_map") + LIST_KEYS
COUNT_KEYS = ("atom_count", "res_count", "bond_count", "CG_nbr_count", "dihe_count", "ca_count")


def make_protein(rng, n_res, min_per=1, max_per=14):
    """a chain of n_res residues with min_per..max_per atoms each; the C-alpha is a random atom of its residue"""
    per = rng.integers(min_per, max_per + 1, size=n_res)
    per[rng.integers(n_res)] = max_per
    start = np.concatenate([[0], np.cumsum(per)[:-1]])
    n_at = int(per.sum())
    from coarsegrainingvae_b200 import synthetic
    ca = synthetic.lattice_points(n_res, 3.8, rng)
    cg_map = np.repeat(np.arange(n_res), per)
    xyz = (ca[cg_map] + rng.normal(scale=1.2, size=(n_at, 3))).astype(np.float32)
    ca_idx = start + rng.integers(0, per)
    xyz[ca_idx] = ca
    chain = np.arange(n_at - 2)
    bonds = np.concatenate([np.stack([chain, chain + 1], 1), np.stack([chain[::3], chain[::3] + 2], 1)], 0)
    first = np.arange(0, n_at - 3, 2)
    dihe = np.stack([first, first + 1, first + 2, first + 3], 1)
    return {"xyz": xyz, "ca_xyz": ca, "res": rng.integers(1, 21, size=n_res), "cg_map": cg_map, "bond_edge_list": bonds,
            "dihe_idxs": dihe, "ca_idx": ca_idx, "seq": "".join(rng.choice(list("ACDEFGHIKLMNPQRSTVWY"), size=n_res))}


def protein_set(n, lo, hi, seed, min_per=1, max_per=14):
    rng = np.random.default_rng(seed)
    return [make_protein(rng, int(rng.integers(lo, hi + 1)), min_per, max_per) for _ in range(n)]


_SMALL = {}


def small_set():
    if "ds" not in _SMALL:
        prots = protein_set(8, 20, 90, seed=7)
        _SMALL["prots"], _SMALL["ds"] = prots, data.DeviceProteinDataset(prots, CUTOFF)
    return _SMALL["prots"], _SMALL["ds"]


def host_collate(prots, idx):
    """SCNCG_collate on the host: per-protein dicts concatenated, indices offset by the running atom / residue counts; the
    C-alpha lists from data.get_neighbor_list per protein (data.py:357)."""
    cols = {k: [] for k in TENSOR_KEYS}
    seqs, a_off, r_off = [], 0, 0
    for i in idx:
        if i < 0:
            continue
        p = prots[i]
        nbr = data.get_neighbor_list(p["ca_xyz"], DEV, CUTOFF, True).cpu()
        t = lambda k, dt: torch.as_tensor(np.asarray(p[k])).to(dt)
        cols["xyz"].append(t("xyz", torch.float32)); cols["ca_xyz"].append(t("ca_xyz", torch.float32))
        cols["res"].append(t("res", torch.int64)); cols["cg_map"].append(t("cg_map", torch.int64) + r_off)
        cols["bond_edge_list"].append(t("bond_edge_list", torch.int64) + a_off); cols["CG_nbr_list"].append(nbr + r_off)
        cols["dihe_idxs"].append(t("dihe_idxs", torch.int64) + a_off); cols["ca_idx"].append(t("ca_idx", torch.int64) + a_off)
        seqs.append(p["seq"])
        a_off += p["xyz"].shape[0]
        r_off += p["ca_xyz"].shape[0]
    out = {k: torch.cat(v, 0) for k, v in cols.items()}
    out["seq"] = seqs
    return out


def check_static(ds, got, want):
    """live region == the unpadded batch, pad region inert (section 3 of the design), counts exact"""
    n_at, n_res = want["xyz"].shape[0], want["ca_xyz"].shape[0]
    live = {"xyz": n_at, "cg_map": n_at, "ca_xyz": n_res, "res": n_res}
    live.update({k: want[k].shape[0] for k in LIST_KEYS})
    for k in TENSOR_KEYS:
        g = got[k].cpu()
        assert g.dtype == want[k].dtype and torch.equal(g[:live[k]], want[k].cpu()), k
        if k != "cg_map":
            assert (g[live[k]:] == 0).all(), k
    pad_map = got["cg_map"].cpu()[n_at:]
    A = ds.atoms_per_bead
    assert torch.equal(pad_map, n_res + torch.arange(pad_map.shape[0]) // A)
    assert int(torch.bincount(got["cg_map"].cpu()).max()) <= A
    assert pad_map.numel() == 0 or int(pad_map.max()) < got["ca_xyz"].shape[0]
    counts = [int(got[k]) for k in COUNT_KEYS]
    assert counts == [n_at, n_res, live["bond_edge_list"], live["CG_nbr_list"], live["dihe_idxs"], live["ca_idx"]]
    assert got["loss_norms"].tolist() == [float(n_at), float(n_res), float(live["bond_edge_list"])]
    assert got["CG_nbr_symmetrize"] is True


@pytest.mark.parametrize("idx", [[3, 1, 3, 0], [5], list(range(8)), [7, 6, 2]])
def test_eager_collate_matches_host_concatenation(idx):
    prots, ds = small_set()
    want = host_collate(prots, idx)
    got = ds.collate(idx)
    assert list(got) == ["xyz", "ca_xyz", "res", "cg_map", "bond_edge_list", "CG_nbr_list", "seq", "ca_idx", "dihe_idxs"]
    assert got["seq"] == want["seq"]
    for k in TENSOR_KEYS:
        assert got[k].device.type == "cuda" and got[k].dtype == want[k].dtype, k
        assert torch.equal(got[k].cpu(), want[k]), k
    on_device = ds.collate(torch.tensor(idx, device=DEV))      # device idx: same tensors, no seq
    assert "seq" not in on_device and all(torch.equal(on_device[k], got[k]) for k in TENSOR_KEYS)


def test_stored_ca_graph_equals_per_protein_neighbor_lists():
    prots, ds = small_set()
    ptr = ds.item_ptr[3].cpu()
    for i, p in enumerate(prots):
        assert torch.equal(ds.store["CG_nbr_list"][ptr[i]:ptr[i + 1]].cpu(),
                           data.get_neighbor_list(p["ca_xyz"], DEV, CUTOFF, True).cpu()), i


def test_static_collate_pads_inertly_and_ignores_empty_slots():
    prots, ds = small_set()
    batches = [[3, 1, 3, 0], [5, 2, 6, 4], [1, -1, 7, -1]]
    caps = ds.capacities(batches=batches)
    caps = {k: v + 11 for k, v in caps.items()}
    for idx in batches:
        got = ds.collate(torch.tensor(idx, device=DEV), static=True, capacities=caps)
        check_static(ds, got, ds.collate([i for i in idx if i >= 0]))
        dense = ds.collate([i for i in idx if i >= 0], static=True, capacities=caps)    # host idx, no empty slots
        for k in TENSOR_KEYS + COUNT_KEYS + ("loss_norms",):
            assert torch.equal(got[k], dense[k]), k
    ops.check_device_errors(torch.device(DEV), force=True)


def _graph_collate_case(ds, batches, caps):
    B = max(len(b) for b in batches)
    pad = lambda b: torch.tensor(list(b) + [-1] * (B - len(b)), dtype=torch.int64)
    static_idx = pad(batches[0]).to(DEV)
    out = ds.collate(static_idx, static=True, capacities=caps)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")                   # no host synchronisation in the static collate
    try:
        ds.collate(static_idx, static=True, out=out)
        ds.collate(static_idx, static=True, capacities=caps)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ds.collate(static_idx, static=True, out=out)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        ds.collate(static_idx, static=True, out=out)
    totals = set()
    for b in batches:
        static_idx.copy_(pad(b))
        graph.replay()
        want = ds.collate(pad(b).to(DEV), static=True, capacities=caps)
        torch.cuda.synchronize()
        totals.add(int(out["atom_count"]))
        for k in TENSOR_KEYS + COUNT_KEYS + ("loss_norms",):
            assert torch.equal(out[k], want[k]), k
    assert len(totals) == len(batches)                           # different total lengths
    ops.check_device_errors(torch.device(DEV), force=True)


def test_static_collate_is_sync_free_and_replays_in_a_graph():
    _, ds = small_set()
    batches = [[0, 1, 2, 3], [7, 5], [6, 6, 4, -1]]
    _graph_collate_case(ds, batches, ds.capacities(batches=batches))


def test_static_collate_graph_replay_at_bench_size():
    """64 proteins of 120..400 residues with 6..14 atoms each (the c4 protein scale)"""
    ds = data.DeviceProteinDataset(protein_set(96, 120, 400, seed=11), 15.5)
    rng = np.random.default_rng(5)
    batches = [rng.permutation(96)[:64].tolist(), rng.permutation(96)[:64].tolist(), rng.permutation(96)[:40].tolist()]
    caps = ds.capacities(batch_size=64)
    _graph_collate_case(ds, batches, caps)
    got = ds.collate(torch.tensor(batches[1], device=DEV), static=True, capacities=caps)
    check_static(ds, got, ds.collate(batches[1]))


def _make_model():
    torch.manual_seed(3)
    return build_pcn(128, 8, CUTOFF, 3).to(DEV)


def test_padding_is_exact_for_the_pcn():
    """PCN (F = 128, 3 layers) on the padded vs the unpadded batch: the same reconstruction, loss and parameter gradients to
    rounding; pad atoms reconstruct to exactly 0 and receive exactly 0 gradient; loss == the float64 oracle."""
    _, ds = small_set()
    idx = [0, 2, 5, 1]
    raw = ds.collate(idx)
    caps = {k: v + 37 for k, v in ds.capacities(batch_size=len(idx)).items()}
    pad = ds.collate(torch.tensor(idx, device=DEV), static=True, capacities=caps)
    assert pad["xyz"].shape[0] > raw["xyz"].shape[0]
    model = _make_model()
    tr = train.PCNTrainStep(model, GAMMA, KAPPA)
    kept = []

    def keep_recon(module, inputs, out):
        out[5].retain_grad()
        kept.append(out[5])

    hook = model.register_forward_hook(keep_recon)
    results = []
    for batch in (raw, pad):
        for p in model.parameters():
            p.grad = None
        kept.clear()
        loss = tr._loss(batch, None)
        loss.backward()
        results.append((loss.detach(), kept[0].detach(), kept[0].grad.detach(),
                        {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}))
    hook.remove()
    (lu, ru, gru, pu), (lp, rp, grp, pp) = results
    n = raw["xyz"].shape[0]
    assert rel_err(lp, lu) <= 1e-6 and rel_err(rp[:n], ru) <= 1e-6
    assert (rp[n:] == 0).all() and (grp[n:] == 0).all()
    assert set(pu) == set(pp) and "embedding.weight" in pu
    for k in pu:
        assert rel_err(pp[k], pu[k]) <= 1e-5, k
    assert (pp["embedding.weight"][0] == 0).all()           # pad residues use the padding row: no gradient reaches it
    want = orc.pcn_loss(ru.double().cpu(), raw["xyz"].double().cpu(), raw["bond_edge_list"].cpu(), raw["dihe_idxs"].cpu(),
                        GAMMA, KAPPA)[0]
    assert rel_err(lu, want) <= 1e-5 and rel_err(lp, want) <= 1e-5


def test_one_graph_trains_on_ragged_batches():
    """GraphedTrainStep captured once; every step re-collates into its static buffers.  Losses and parameters equal an
    eager PCNTrainStep on the same padded batches bit for bit, and the losses equal eager steps on the unpadded batches."""
    _, ds = small_set()
    batches = [[0, 1, 2, 3], [4, 5, 6, 7], [2, 7, -1, -1], [1, 3, 5, -1]]
    caps = ds.capacities(batches=batches)
    idx_t = [torch.tensor(b, device=DEV) for b in batches]
    statics = [ds.collate(t, static=True, capacities=caps) for t in idx_t]
    raws = [ds.collate([i for i in b if i >= 0]) for b in batches]
    assert len({int(s["atom_count"]) for s in statics}) == len(batches)
    ma, mb, mc = _make_model(), _make_model(), _make_model()
    ta = train.PCNTrainStep(ma, GAMMA, KAPPA, capturable=True)
    ta.prepare(statics[0], None)
    tb = train.PCNTrainStep(mb, GAMMA, KAPPA, capturable=True)
    tb.prepare(statics[0], None)
    graphed = train.GraphedTrainStep(tb, statics[0], None)
    tc = train.PCNTrainStep(mc, GAMMA, KAPPA)
    tc.prepare(raws[0], None)
    # the warm-up steps of the capture advanced tb: reset it (parameters are views of the flat buffers)
    for name in ("exp_avg", "exp_avg_sq", "step_count"):
        getattr(tb, name).zero_()
    tb.flat_p.copy_(ta.flat_p)
    assert torch.equal(tc.flat_p, ta.flat_p)
    for i in range(len(batches)):
        la = float(ta.step(statics[i], None))
        ds.collate(idx_t[i], static=True, out=graphed.static)
        lb = float(graphed.step({}))
        lc = float(tc.step(raws[i], None))
        assert la == lb, (i, la, lb)
        assert abs(lb - lc) <= 1e-5 * abs(lc), (i, lb, lc)
    assert torch.equal(ta.flat_p, tb.flat_p)
    ops.check_device_errors(torch.device(DEV), force=True)


def test_capacity_overflow_writes_nothing_past_capacity_and_raises():
    _, ds = small_set()
    idx = torch.tensor([3, 1, 6], device=DEV)
    exact = ds.capacities(batches=[[3, 1, 6]])
    dev = torch.device(DEV)
    ops.check_device_errors(dev, force=True)
    for short in data._PROTEIN_CAP_KEYS:
        caps = dict(exact)
        caps[short] -= 3
        big = ds._outputs({k: v + 50 for k, v in caps.items()})
        for t in big.values():
            t.fill_(-7)
        canary = {k: t.clone() for k, t in big.items()}
        out = {k: big[k][:caps[data._PROTEIN_CAP_KEYS[kind]]] for k, kind, *_ in data._PROTEIN_KEYS}
        out.update({k: torch.zeros(1, dtype=torch.int64, device=DEV) for k in COUNT_KEYS})
        out["loss_norms"] = torch.zeros(3, device=DEV)
        ds.collate(idx, static=True, out=out)
        with pytest.raises(IndexError, match="capacities"):
            ops.check_device_errors(dev, force=True)
        for k, kind, *_ in data._PROTEIN_KEYS:
            rows = caps[data._PROTEIN_CAP_KEYS[kind]]
            assert torch.equal(big[k][rows:], canary[k][rows:]), (short, k)
        kind = data._PROTEIN_CAP_KEYS.index(short)
        live_cap = caps[short] - (-(-caps["xyz"] // ds.atoms_per_bead) if short == "ca_xyz" else 0)
        assert int(out[COUNT_KEYS[kind]]) == live_cap, short          # truncated to the capacity
    ds.collate(torch.tensor([3, 99], device=DEV), static=True)      # an item outside the set
    with pytest.raises(IndexError, match="outside the dataset"):
        ops.check_device_errors(dev, force=True)
    with pytest.raises(IndexError):
        ds.collate([3, 99])
