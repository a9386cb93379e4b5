"""Graph builders and batch assembly with the reference's names (data.py of the reference):
``get_neighbor_list``, ``CGDataset.generate_neighbor_list``, ``CG_collate``, ``batch_to``.
The radius search runs on the GPU (cell lists for large frames) and returns the reference's edge set
bit for bit, in the reference's order.
"""
import numpy as np
import torch
from torch.utils.data import Dataset as TorchDataset

from . import ops


def batch_to(batch, device):
    """data.py:16-20."""
    return {key: (val.to(device) if hasattr(val, 'to') else val) for key, val in batch.items()}


def get_neighbor_list(xyz, device='cuda', cutoff=5, undirected=True):
    """data.py:65-82.  ``device`` must be a CUDA device: the search is an sm_100a kernel.  Returns an int64
    [E,2] tensor on that device, sorted like ``torch.nonzero`` (i ascending, then j ascending)."""
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise RuntimeError("get_neighbor_list runs on the GPU only (device=%r); no CPU fallback" % (device,))
    xyz = torch.as_tensor(np.asarray(xyz) if not torch.is_tensor(xyz) else xyz, dtype=torch.float32).to(dev)
    return ops.radius_graph(xyz, cutoff, undirected=undirected)


def get_neighbor_list_batch(xyz, num_atoms, cutoff, undirected=True):
    """All frames of a batch in one launch: equals the per-frame lists of data.py:207-225 after the
    CG_collate offsets (data.py:255-270).  xyz [sum(num_atoms),3] CUDA, num_atoms [B]."""
    counts = torch.as_tensor(num_atoms, dtype=torch.int64)
    frame_ptr = torch.zeros(counts.numel() + 1, dtype=torch.int64)
    frame_ptr[1:] = torch.cumsum(counts.cpu(), 0)
    use_cells = bool(counts.max().item() > 1024) if counts.numel() else False
    return ops.radius_graph(xyz, cutoff, undirected=undirected, frame_ptr=frame_ptr.to(xyz.device), use_cells=use_cells)


def bond_cg_graph(bond_edge_list, mapping, n_cgs):
    """CG graph derived from the bond graph (data.py:227-248): beads I != J are neighbours iff some bond joins an atom of
    I to an atom of J.  The reference forms assign^T . adj . assign as dense float matrices and takes ``nonzero()``; this
    is the same set in the same (row-major, both directions) order from integer keys -- dataset-preparation time, on the
    device the lists live on (the reference keeps them on the CPU)."""
    bond = torch.as_tensor(bond_edge_list, dtype=torch.int64)
    mapping = torch.as_tensor(mapping, dtype=torch.int64)
    a, b = mapping[bond[:, 0]], mapping[bond[:, 1]]
    keys = torch.cat([a * n_cgs + b, b * n_cgs + a])
    keys = torch.unique(keys[torch.cat([a != b, a != b])])          # sorted: row-major order of nonzero()
    return torch.stack([keys // n_cgs, keys % n_cgs], 1)


class CGDataset(TorchDataset):
    """data.py:186-252."""

    def __init__(self, props, check_props=True):
        self.props = props

    def __len__(self):
        return len(self.props['nxyz'])

    def __getitem__(self, idx):
        return {key: val[idx] for key, val in self.props.items()}

    def generate_neighbor_list(self, atom_cutoff, cg_cutoff, device='cuda', undirected=True, use_bond=False):
        """Builds props['nbr_list'] / props['CG_nbr_list'] for every frame.  All frames go through ONE batched
        kernel call per graph kind instead of the reference's python loop (data.py:215-225); results are split
        back into per-frame CPU tensors with frame-local indices, as the reference stores them."""
        if use_bond:
            nbr_list = self.props['bond_edge_list']
        else:
            nbr_list = self._batched(self.props['nxyz'], atom_cutoff, device, undirected)
        if cg_cutoff is None:
            cg_nbr_list = [bond_cg_graph(bond, self.props['CG_mapping'][i], int(self.props['num_CGs'][i]))
                           for i, bond in enumerate(self.props['bond_edge_list'])]
        else:
            cg_nbr_list = self._batched(self.props['CG_nxyz'], cg_cutoff, device, undirected)
        self.props['nbr_list'] = nbr_list
        self.props['CG_nbr_list'] = cg_nbr_list

    @staticmethod
    def _batched(frames, cutoff, device, undirected):
        counts = [int(f.shape[0]) for f in frames]
        xyz = torch.cat([torch.as_tensor(f)[:, 1:4].float() for f in frames], 0).to(device)
        pairs = get_neighbor_list_batch(xyz, counts, cutoff, undirected).cpu()
        offsets = np.cumsum([0] + counts)
        first = torch.searchsorted(pairs[:, 0].contiguous(), torch.as_tensor(offsets, dtype=torch.int64))
        return [pairs[first[k]:first[k + 1]] - int(offsets[k]) for k in range(len(counts))]


class DeviceCGDataset(object):
    """On-GPU batch assembly (SURVEY.md section 8f, rank 2) for the trajectory datasets of the reference: every frame is the
    same molecule (datasets.py:434-500: one atomic-number vector, one CG mapping, one bond list; only the coordinates
    differ), so the whole trajectory stays resident in HBM as ``xyz [T, n, 3]`` and a batch is assembled ON THE DEVICE from
    a vector of frame indices:

    * ``nxyz`` / ``CG_nxyz`` rows gathered, ``CG_mapping`` / ``bond_edge_list`` offset by the running atom / bead counts
      (``CG_collate``, data.py:255-289);
    * ``CG_xyz = scatter_mean(xyz, mapping)`` (datasets.py:487) by the bead-pooling kernel when no CG trajectory is given;
    * ``nbr_list`` / ``CG_nbr_list`` built on the fly by ONE batched radius-graph launch each (``get_neighbor_list`` per
      frame in ``generate_neighbor_list``, data.py:207-225) -- no stored edge lists, no per-frame CPU pre-pass, no H2D of
      index tensors; ``cg_cutoff=None`` takes the bond-derived CG graph (data.py:227-248), identical in every frame.

    ``collate(idx)`` returns the dict ``CG_collate([dataset[i] for i in idx])`` would (same keys, dtypes, order: bit-exact
    index tensors); ``collate(idx, static=True)`` returns the static-capacity form of ``train.to_static_batch`` (padded lists
    + device-side live counts) with NO host synchronisation, ready for ``GraphedTrainStep.step``."""

    def __init__(self, atomic_nums, xyz, mapping, bond_edge_list, atom_cutoff, cg_cutoff, device='cuda', undirected=True,
                 cg_xyz=None):
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError("DeviceCGDataset lives on a CUDA device (device=%r); no CPU fallback" % (device,))
        self.device = dev
        self.xyz = torch.as_tensor(np.asarray(xyz) if not torch.is_tensor(xyz) else xyz, dtype=torch.float32).to(dev).contiguous()
        self.n_frames, self.n_atoms = int(self.xyz.shape[0]), int(self.xyz.shape[1])
        self.z = torch.as_tensor(atomic_nums, dtype=torch.float32).to(dev)
        self.mapping = torch.as_tensor(mapping, dtype=torch.int64).to(dev)
        self.n_cgs = int(self.mapping.max().item()) + 1
        self.bonds = torch.as_tensor(bond_edge_list, dtype=torch.int64).to(dev)
        self.atom_cutoff, self.cg_cutoff, self.undirected = atom_cutoff, cg_cutoff, undirected
        self.seg = ops.build_segments(self.mapping, self.n_cgs)
        self.cg_xyz = None if cg_xyz is None else torch.as_tensor(cg_xyz, dtype=torch.float32).to(dev).contiguous()
        self.cg_bond_graph = bond_cg_graph(self.bonds, self.mapping, self.n_cgs) if cg_cutoff is None else None

    def __len__(self):
        return self.n_frames

    def capacities(self, batch_size):
        """worst-case list capacities of a static batch of ``batch_size`` frames."""
        n, nb, div = self.n_atoms, self.n_cgs, (2 if self.undirected else 1)
        cg = batch_size * nb * (nb - 1) // div if self.cg_cutoff is not None else batch_size * int(self.cg_bond_graph.shape[0])
        return {"nbr_list": batch_size * n * (n - 1) // div, "CG_nbr_list": cg, "bond_edge_list": batch_size * int(self.bonds.shape[0])}

    def collate(self, idx, static=False):
        dev, n, nb = self.device, self.n_atoms, self.n_cgs
        idx = torch.as_tensor(idx, dtype=torch.int64, device=dev)
        B = int(idx.shape[0])
        xyz = self.xyz.index_select(0, idx)                                        # [B, n, 3]
        flat = xyz.reshape(B * n, 3)
        nxyz = torch.cat([self.z.repeat(B)[:, None], flat], 1)
        if self.cg_xyz is not None:
            cg_flat = self.cg_xyz.index_select(0, idx).reshape(B * nb, 3)
        else:
            # scatter_mean per frame == bead pooling over the block-diagonal batch mapping
            cg_flat = ops.segment_reduce_fwd(flat.contiguous(), self._batch_segments(B), True)
        frame = torch.arange(B, dtype=torch.int64, device=dev)
        CG_nxyz = torch.cat([torch.arange(nb, dtype=torch.float32, device=dev).repeat(B)[:, None], cg_flat], 1)
        CG_mapping = (self.mapping[None, :] + frame[:, None] * nb).reshape(-1)
        bond = (self.bonds[None, :, :] + (frame * n)[:, None, None]).reshape(-1, 2)
        atom_ptr = torch.arange(B + 1, dtype=torch.int64, device=dev) * n
        bead_ptr = torch.arange(B + 1, dtype=torch.int64, device=dev) * nb
        batch = {'nxyz': nxyz, 'CG_nxyz': CG_nxyz, 'num_atoms': torch.full((B,), n, dtype=torch.int64, device=dev),
                 'num_CGs': torch.full((B,), nb, dtype=torch.int64, device=dev), 'CG_mapping': CG_mapping,
                 'bond_edge_list': bond}
        cap = self.capacities(B) if static else None
        kw = lambda key, mf: dict(capacity=cap[key], max_frame=mf) if static else dict(max_frame=mf)
        nbr = ops.radius_graph(flat, self.atom_cutoff, self.undirected, frame_ptr=atom_ptr, use_cells=n > 1024, **kw("nbr_list", n))
        if self.cg_cutoff is not None:
            cg_nbr = ops.radius_graph(cg_flat.contiguous(), self.cg_cutoff, self.undirected, frame_ptr=bead_ptr, use_cells=nb > 1024,
                                      **kw("CG_nbr_list", nb))
        else:
            lst = (self.cg_bond_graph[None, :, :] + (frame * nb)[:, None, None]).reshape(-1, 2)
            cg_nbr = (lst, torch.full((1,), int(lst.shape[0]), dtype=torch.int64, device=dev)) if static else lst
        if static:
            batch['nbr_list'], batch['nbr_count'] = nbr
            batch['CG_nbr_list'], batch['CG_nbr_count'] = cg_nbr
            batch['bond_count'] = torch.full((1,), int(bond.shape[0]), dtype=torch.int64, device=dev)
            # radius graphs are one-directional (j > i) when undirected: the flipped half is generated by the CSR kernels;
            # the bond-derived CG graph already holds both directions (nonzero() of a symmetric matrix)
            batch['nbr_symmetrize'] = bool(self.undirected)
            batch['CG_nbr_symmetrize'] = bool(self.undirected) if self.cg_cutoff is not None else False
        else:
            batch['nbr_list'], batch['CG_nbr_list'] = nbr, cg_nbr
        return batch

    def _batch_segments(self, B):
        cache = getattr(self, "_seg_cache", None)
        if cache is None or cache[0] != B:
            frame = torch.arange(B, dtype=torch.int64, device=self.device)
            mapping = (self.mapping[None, :] + frame[:, None] * self.n_cgs).reshape(-1)
            self._seg_cache = (B, ops.build_segments(mapping, B * self.n_cgs))
        return self._seg_cache[1]


def CG_collate(dicts):
    """data.py:255-289: offset the index tensors of every sample by the running atom / bead counts, then
    concatenate (tensors with a shape) or stack (0-d tensors); strings are gathered in lists."""
    atom_off = np.cumsum([0] + [int(d['num_atoms']) for d in dicts])[:-1]
    bead_off = np.cumsum([0] + [int(d['num_CGs']) for d in dicts])[:-1]
    shifted = []
    for d, a, b in zip(dicts, atom_off, bead_off):
        e = dict(d)
        e['nbr_list'] = d['nbr_list'] + int(a)
        e['bond_edge_list'] = d['bond_edge_list'] + int(a)
        e['CG_mapping'] = d['CG_mapping'] + int(b)
        e['CG_nbr_list'] = d['CG_nbr_list'] + int(b)
        shifted.append(e)
    batch = {}
    for key, val in shifted[0].items():
        if hasattr(val, 'shape') and len(val.shape) > 0:
            batch[key] = torch.cat([s[key] for s in shifted], dim=0)
        elif isinstance(val, str):
            batch[key] = [s[key] for s in shifted]
        else:
            batch[key] = torch.stack([torch.as_tensor(s[key]) for s in shifted], dim=0)
    return batch


# Kinds of rows of a protein item (CGVAE_COLLATE_* of the C ABI) and the per-protein arrays they count.
PROTEIN_KINDS = ("atoms", "residues", "bonds", "ca_edges", "dihedrals", "ca_idx")
# batch key -> (kind, row width (0: a vector), dtype, kind whose running count the collate adds, or None)
_PROTEIN_KEYS = (("xyz", 0, 3, torch.float32, None), ("ca_xyz", 1, 3, torch.float32, None), ("res", 1, 0, torch.int64, None),
                 ("cg_map", 0, 0, torch.int64, 1), ("bond_edge_list", 2, 2, torch.int64, 0),
                 ("CG_nbr_list", 3, 2, torch.int64, 1), ("ca_idx", 5, 0, torch.int64, 0), ("dihe_idxs", 4, 4, torch.int64, 0))
# live-count key of every kind in a static batch (train.to_static_pcn_batch names, plus atom_count / res_count)
_PROTEIN_COUNT_KEYS = ("atom_count", "res_count", "bond_count", "CG_nbr_count", "dihe_count", "ca_count")
# the capacity of a kind is the row count of this key ("ca_xyz" rows include the pad beads)
_PROTEIN_CAP_KEYS = ("xyz", "ca_xyz", "bond_edge_list", "CG_nbr_list", "dihe_idxs", "ca_idx")


def protein_capacities(sizes, atoms_per_bead, batch_size=None, batches=None):
    """Static capacities of a protein batch from a size table ``sizes [P, 6]`` (columns in ``PROTEIN_KINDS`` order),
    keyed like the batch tensors whose row count they fix.  Default: per kind, the sum of the ``batch_size`` largest
    entries.  ``batches`` (planned lists of item indices, -1 = empty slot): per kind, the largest total over those batches.
    ``ca_xyz`` adds ceil(atoms / atoms_per_bead) pad beads, so the pad atoms of a batch can be spread over beads of at most
    ``atoms_per_bead`` atoms each."""
    sizes = np.asarray(sizes, dtype=np.int64).reshape(-1, len(PROTEIN_KINDS))
    if batches is not None:
        tot = np.zeros(len(PROTEIN_KINDS), dtype=np.int64)
        for b in batches:
            b = np.asarray(b, dtype=np.int64).reshape(-1)
            tot = np.maximum(tot, sizes[b[b >= 0]].sum(0))
    elif batch_size is not None:
        tot = -np.sort(-sizes, axis=0)[:int(batch_size)].sum(0)
    else:
        raise ValueError("protein_capacities needs batch_size or batches")
    caps = {key: int(t) for key, t in zip(_PROTEIN_CAP_KEYS, tot)}
    caps["ca_xyz"] += -(-caps["xyz"] // int(atoms_per_bead))
    return caps


class DeviceProteinDataset(object):
    """HBM-resident protein set of the protein-completion path (``SCNCGDataset`` + ``SCNCG_collate``, data.py:292-398 of the
    reference) for proteins of different lengths.

    ``proteins``: a list of per-protein dicts in the reference's item layout with frame-local indices -- ``xyz [n_at,3]``,
    ``ca_xyz [n_res,3]``, ``res [n_res]``, ``cg_map [n_at]`` (residue of each atom), ``bond_edge_list [n_b,2]``,
    ``dihe_idxs [n_d,4]`` and ``ca_idx [n_c]`` (atom indices), optional ``seq``.  Every array goes into one concatenated
    device store per kind of row with an int64 row-offset table.  The C-alpha graph (``get_neighbor_list(ca_xyz, cg_cutoff,
    True)`` of data.py:357) is built once, for all proteins in one batched launch, and stored the same way: the coordinates
    never change, so the collate is a pure gather.

    ``collate(idx)`` returns the dict the host pipeline builds (per-protein dicts concatenated, indices offset by the
    running atom / residue counts).  ``collate(idx, static=True)`` returns capacity-padded tensors with device live counts
    for ``GraphedTrainStep``: two launches, no host synchronisation, graph-capturable.  Pads are inert for the PCN: pad
    atoms have zero coordinates and map, at most ``atoms_per_bead`` to a bead, to pad residues with ``res = 0`` (the
    embedding's padding row), zero coordinates and no edges, bonds, dihedrals or C-alpha entries."""

    def __init__(self, proteins, cg_cutoff, device='cuda'):
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError("DeviceProteinDataset lives on a CUDA device (device=%r); no CPU fallback" % (device,))
        self.device, self.cg_cutoff = dev, cg_cutoff
        P = len(proteins)
        host = {key: [] for key, *_ in _PROTEIN_KEYS if key != "CG_nbr_list"}
        sizes = np.zeros((P, len(PROTEIN_KINDS)), dtype=np.int64)
        self.atoms_per_bead = 1
        for p, item in enumerate(proteins):
            arr = {}
            for key, kind, width, dtype, _ in _PROTEIN_KEYS:
                if key == "CG_nbr_list":
                    continue
                shape = (-1, width) if width else (-1,)
                val = item.get(key)
                t = torch.zeros((0, width) if width else (0,), dtype=dtype) if val is None else \
                    torch.as_tensor(np.asarray(val) if not torch.is_tensor(val) else val).detach().cpu().to(dtype)
                if t.numel() == 0:
                    t = t.reshape((0, width) if width else (0,))
                if tuple(t.shape[1:]) != tuple(shape[1:]) or t.dim() != len(shape):
                    raise ValueError("protein %d: %s has shape %s, expected [n%s]" % (p, key, tuple(t.shape),
                                                                                       ", %d" % width if width else ""))
                arr[key] = t.contiguous()
            n_at, n_res = int(arr["xyz"].shape[0]), int(arr["ca_xyz"].shape[0])
            if arr["cg_map"].shape[0] != n_at or arr["res"].shape[0] != n_res:
                raise ValueError("protein %d: cg_map must have one entry per atom and res one per residue" % p)
            # every index inside its own protein: a ca_idx entry >= n_atoms would make the pin predicate of cgvae.py:569-571
            # depend on which proteins share a batch
            for key, n in (("cg_map", n_res), ("bond_edge_list", n_at), ("dihe_idxs", n_at), ("ca_idx", n_at)):
                t = arr[key]
                if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n):
                    raise IndexError("protein %d: %s entry outside [0, %d)" % (p, key, n))
            if n_at:
                self.atoms_per_bead = max(self.atoms_per_bead, int(torch.bincount(arr["cg_map"], minlength=1).max()))
            for key in host:
                host[key].append(arr[key])
            sizes[p] = (n_at, n_res, arr["bond_edge_list"].shape[0], 0, arr["dihe_idxs"].shape[0], arr["ca_idx"].shape[0])
        self.seq = [item.get("seq") for item in proteins]
        self.store = {key: torch.cat(v, 0).to(dev).contiguous() if v else None for key, v in host.items()}
        # C-alpha graph of every protein: one batched launch, split by the residue offsets into frame-local lists
        res_ptr = torch.zeros(P + 1, dtype=torch.int64)
        res_ptr[1:] = torch.cumsum(torch.as_tensor(sizes[:, 1]), 0)
        if P and int(res_ptr[-1]) > 0:
            pairs = get_neighbor_list_batch(self.store["ca_xyz"], sizes[:, 1], cg_cutoff, True)
            res_ptr_d = res_ptr.to(dev)
            owner = torch.searchsorted(res_ptr_d, pairs[:, 0].contiguous(), right=True) - 1
            self.store["CG_nbr_list"] = (pairs - res_ptr_d[owner][:, None]).contiguous()
            sizes[:, 3] = torch.bincount(owner, minlength=P).cpu().numpy()
        else:
            self.store["CG_nbr_list"] = torch.zeros((0, 2), dtype=torch.int64, device=dev)
        self.sizes = sizes
        ptr = np.zeros((len(PROTEIN_KINDS), P + 1), dtype=np.int64)
        ptr[:, 1:] = np.cumsum(sizes, 0).T
        self.item_ptr = torch.from_numpy(ptr).to(dev)

    def __len__(self):
        return len(self.sizes)

    def capacities(self, batch_size=None, batches=None):
        """``protein_capacities`` of this set's size table (see there)."""
        return protein_capacities(self.sizes, self.atoms_per_bead, batch_size, batches)

    def _outputs(self, caps):
        out = {}
        for key, kind, width, dtype, _ in _PROTEIN_KEYS:
            rows = caps[_PROTEIN_CAP_KEYS[kind]]
            out[key] = torch.empty((rows, width) if width else (rows,), dtype=dtype, device=self.device)
        return out

    def _run(self, idx, out, n_pad_beads, count_out=None, norms=None):
        outputs, live = [], [0] * len(PROTEIN_KINDS)
        for key, kind, width, dtype, add in _PROTEIN_KEYS:
            t = out[key]
            if t.dtype != dtype or tuple(t.shape[1:]) != ((width,) if width else ()):
                raise ValueError("%s: expected %s [rows%s], got %s %s" % (key, dtype, ", %d" % width if width else "", t.dtype,
                                                                        tuple(t.shape)))
            outputs.append((t, self.store[key], kind, add, key == "cg_map" and n_pad_beads > 0))
            live[kind] = int(t.shape[0])
        if out["cg_map"].shape[0] != out["xyz"].shape[0] or out["res"].shape[0] != out["ca_xyz"].shape[0]:
            raise ValueError("cg_map / xyz and res / ca_xyz must have the same number of rows")
        live[1] -= n_pad_beads
        if live[1] < 0:
            raise ValueError("ca_xyz has fewer rows than the %d pad beads of %d atom rows" % (n_pad_beads, live[0]))
        return ops.collate(idx, self.item_ptr, outputs, live, self.atoms_per_bead, out["ca_xyz"].shape[0], count_out, norms)

    def _device_idx(self, idx):
        if torch.is_tensor(idx) and idx.is_cuda:
            return idx.to(torch.int64).contiguous()
        t = torch.as_tensor(np.asarray(idx, dtype=np.int64).reshape(-1))
        return t.pin_memory().to(self.device, non_blocking=True)

    def collate(self, idx, static=False, out=None, capacities=None):
        """``idx``: item indices (host list / array or int64 tensor on host or device; -1 = empty slot).

        static=False: the unpadded batch of the host pipeline (keys and dtypes of ``synthetic.pcn_batch``; ``seq`` is a
        list when ``idx`` is on the host).  One host read of the batch size when ``idx`` is on the device.

        static=True: fixed shapes from ``capacities`` (default ``self.capacities(len(idx))``) or from the tensors of ``out``
        (written in place, e.g. ``GraphedTrainStep.static``), live counts ``atom_count``, ``res_count``, ``bond_count``,
        ``CG_nbr_count``, ``dihe_count``, ``ca_count`` (int64 [1]) and the loss denominators ``loss_norms`` (float [3]:
        atoms, residues, bonds) on the device; no host synchronisation.  Inside a CUDA graph capture ``idx`` must be a
        device tensor.  A batch larger than the capacities is truncated and flagged: ``ops.check_device_errors`` raises."""
        if not static:
            idx_h = np.asarray(idx.cpu() if torch.is_tensor(idx) else idx, dtype=np.int64).reshape(-1)
            if idx_h.size and (idx_h.min() < -1 or idx_h.max() >= len(self)):
                raise IndexError("protein index outside [-1, %d)" % len(self))
            tot = self.sizes[idx_h[idx_h >= 0]].sum(0)
            batch = self._outputs(dict(zip(_PROTEIN_CAP_KEYS, (int(t) for t in tot))))
            self._run(self._device_idx(idx), batch, 0)
            if not (torch.is_tensor(idx) and idx.is_cuda):
                batch = {k: batch[k] for k in ("xyz", "ca_xyz", "res", "cg_map", "bond_edge_list", "CG_nbr_list")} | \
                    {"seq": [self.seq[i] for i in idx_h if i >= 0], "ca_idx": batch["ca_idx"], "dihe_idxs": batch["dihe_idxs"]}
            return batch
        if out is None:
            n = int(idx.shape[0]) if torch.is_tensor(idx) else len(np.asarray(idx).reshape(-1))
            out = self._outputs(capacities if capacities is not None else self.capacities(n))
            for key in _PROTEIN_COUNT_KEYS:
                out[key] = torch.empty(1, dtype=torch.int64, device=self.device)
            out["loss_norms"] = torch.empty(3, dtype=torch.float32, device=self.device)
        n_pad = -(-int(out["xyz"].shape[0]) // self.atoms_per_bead)
        self._run(self._device_idx(idx), out, n_pad, [out[k] for k in _PROTEIN_COUNT_KEYS], out["loss_norms"])
        batch = dict(out)
        batch["CG_nbr_symmetrize"] = True            # one-directional (j > i) C-alpha lists: the CSR kernels add the flip
        return batch
