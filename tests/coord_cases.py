"""Coordinate-gradient cases shared by the CPU tests (kernel emulator, float64) and the GPU tests (sm_100a kernels,
float32).  Each case runs the product with its coordinate inputs requiring grad and returns
(got {name: gradient}, oracle) where ``oracle(dtype)`` evaluates the same gradients with the oracle's autograd on CPU
(the oracle's edge_geometry restates the reference's expressions line for line)."""
import torch

import coarsegrainingvae_b200 as cg
from coarsegrainingvae_b200 import train
from oracle import cgvae_oracle as orc
from tests.golden_util import load, section, rel_err
from tests.parity_cases import _load_params, build_vae, _batch_to


def _oracle_P(module, dtype):
    return {k: v.detach().cpu().to(dtype if v.dtype.is_floating_point else v.dtype).clone() for k, v in module.state_dict().items()}


def _leaf(t, dtype, dev):
    return t.to(dtype).to(dev).clone().requires_grad_()


def _cotangents(shapes, dtype, seed=7):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(s, generator=g, dtype=torch.float64).to(dtype) for s in shapes]


def check(got, oracle, tol, fp32_rule=False):
    """got vs oracle(float64).  fp32_rule: per tensor, error <= max(tol, 10 x the fp32 oracle's own error), and the
    relative L2 error over all coordinate gradients together <= tol (parity_cases._check_grads with P64).
    Returns {name: error vs float64}."""
    o64 = oracle(torch.float64)
    o32 = oracle(torch.float32) if fp32_rule else None
    errs, num, den = {}, 0.0, 0.0
    for k, g in got.items():
        assert g is not None, k
        truth = o64[k]
        e = rel_err(g, truth)
        errs[k] = e
        if o32 is None:
            assert e < tol, (k, e)
        else:
            e_ref = rel_err(o32[k], truth)
            assert e < max(tol, 10.0 * e_ref), (k, e, e_ref)
        num += float((g.detach().cpu().double() - truth).pow(2).sum())
        den += float(truth.pow(2).sum())
    if o32 is not None:
        assert (num / den) ** 0.5 < tol, ("global relative L2", (num / den) ** 0.5)
    return errs


BLOCKS = {"k3": ("EquiMessageBlock", orc.equi_message), "k4": ("EquiMessageCross", orc.equi_message_cross),
          "k9": ("EquiMessagePsuedo", orc.equi_message_pseudo), "k3w": ("EquiMessageBlock", orc.equi_message)}


def block_r(dev, tag, dtype):
    """d loss / d r_ij of the block API on the blocks_small.npz inputs (k3w: with edge_wgt)."""
    z = load("blocks_small.npz")
    sec = section(z, tag)
    F, R, cutoff = int(z["meta/F"]), int(z["meta/R"]), float(z["meta/cutoff"])
    cls, ofn = BLOCKS[tag]
    blk = getattr(cg, cls)(feat_dim=F, activation="swish", n_rbf=R, cutoff=cutoff, dropout=0.0)
    _load_params(blk, sec, dtype, dev)
    nbrs = torch.from_numpy(z["in/nbrs"])
    r0 = torch.from_numpy(z["in/r"])
    names = ("s", "sbar", "v", "vbar") if tag == "k9" else ("s", "v")
    ins0 = [sec[k] for k in names]
    w0 = sec.get("w")

    def run(P, dtype_, dev_):
        r = _leaf(r0, dtype_, dev_)
        ins = [t.to(dtype_).to(dev_) for t in ins0]
        w = w0.to(dtype_).to(dev_) if w0 is not None else None
        if P is None:
            kw = dict(edge_wgt=w) if w is not None else {}
            outs = blk(*ins, r, nbrs.to(dev_), **kw)
        else:
            kw = dict(edge_wgt=w) if w is not None else {}
            outs = ofn(P, "blk", *ins, r, nbrs, R, cutoff, **kw)
        gs = _cotangents([o.shape for o in outs], dtype_)
        sum((o * g.to(dev_)).sum() for o, g in zip(outs, gs)).backward()
        return {"r": r.grad}

    got = run(None, dtype, dev)
    return got, lambda dt: run({"blk." + k: v for k, v in _oracle_P(blk, dt).items()}, dt, "cpu")


def contraction_r(dev, dtype):
    z = load("blocks_small.npz")
    F, R = int(z["meta/F"]), int(z["meta/R"])
    sec = section(z, "con")
    blk = cg.ContractiveMessageBlock(feat_dim=F, activation="swish", n_rbf=R, cutoff=20.0, dropout=0.0)
    _load_params(blk, sec, dtype, dev)

    def run(P, dtype_, dev_):
        r = _leaf(sec["r_iI"], dtype_, dev_)
        s, v = sec["s"].to(dtype_).to(dev_), sec["v"].to(dtype_).to(dev_)
        if P is None:
            outs = blk(s, v, r, sec["mapping"].to(dev_))
        else:
            outs = orc.contractive_message(P, "blk", s, v, r, sec["mapping"], R)
        gs = _cotangents([o.shape for o in outs], dtype_)
        sum((o * g.to(dev_)).sum() for o, g in zip(outs, gs)).backward()
        return {"r_iI": r.grad}

    got = run(None, dtype, dev)
    return got, lambda dt: run({"blk." + k: v for k, v in _oracle_P(blk, dt).items()}, dt, "cpu")


def cgvae_coords(dev, tag, dtype, fused_loss=False):
    """CGequiVAE training loss -> d / d nxyz, d / d CG_nxyz (xyz is the encoder input AND the loss target)."""
    equivariant = tag != "vae_noneq"
    sec = section(load("cgvae_small.npz" if equivariant else "cgvae_noneq.npz"), tag)
    F, R, enc, dec, acut, ccut, breaksym, beta, gamma = [float(x) for x in sec["meta"]]
    model = build_vae(int(F), int(R), int(enc), int(dec), acut, ccut, bool(breaksym), equivariant=equivariant)
    _load_params(model, sec, dtype, dev)
    batch = {k[len("batch/"):]: v for k, v in sec.items() if k.startswith("batch/")}
    spec = dict(n_basis=int(F), n_rbf=int(R), enc_nconv=int(enc), dec_nconv=int(dec), atom_cutoff=acut, cg_cutoff=ccut,
                decoder="pseudo", breaksym=bool(breaksym), activation="swish", equivariant=equivariant)

    def run(P, dtype_, dev_):
        b = _batch_to(batch, dtype_, dev_)
        b["nxyz"], b["CG_nxyz"] = b["nxyz"].clone().requires_grad_(), b["CG_nxyz"].clone().requires_grad_()
        eps = sec["eps"].to(dtype_).to(dev_)
        if P is None:
            out = model(b, eps=eps)
            if fused_loss:
                loss = train.training_loss(out, out[4], b["bond_edge_list"], beta, gamma)[0]
            else:
                loss = orc.training_loss(out, b, beta, gamma)[0]
        else:
            loss = orc.training_loss(orc.cgvae_forward(P, spec, b, eps=eps), b, beta, gamma)[0]
        loss.backward()
        return {"nxyz": b["nxyz"].grad, "CG_nxyz": b["CG_nxyz"].grad}

    got = run(None, dtype, dev)
    return got, lambda dt: run(_oracle_P(model, dt), dt, "cpu")


def pcn_coords(dev, tag, dtype, ca_pin=True):
    """PCN -> d / d ca_xyz (ca_pin: the C-alpha atoms pinned to their bead, lifting mode 2; else plain mode 0)."""
    sec = section(load("pcn_small.npz"), tag)
    F, R, dec, cutoff, cross_flag = [float(x) for x in sec["meta"]]
    net = cg.EquivariantDecoder(n_atom_basis=int(F), n_rbf=int(R), cutoff=cutoff, num_conv=int(dec), activation="swish",
                                cross_flag=bool(cross_flag))
    model = cg.PCN(net, feature_dim=int(F), offset=False)
    _load_params(model, sec, dtype, dev)
    batch = {k[len("batch/"):]: v for k, v in sec.items() if k.startswith("batch/")}
    batch["seq"] = ["A" * batch["ca_xyz"].shape[0]]
    if not ca_pin:
        batch["ca_idx"] = batch["ca_idx"][:0]
    spec = dict(n_basis=int(F), n_rbf=int(R), dec_nconv=int(dec), atom_cutoff=cutoff,
                decoder="cross" if cross_flag else "plain", activation="swish")

    def run(P, dtype_, dev_):
        b = _batch_to(batch, dtype_, dev_)
        b["ca_xyz"] = b["ca_xyz"].clone().requires_grad_()
        if P is None:
            out = model(b)
        elif ca_pin:
            out = orc.pcn_forward(P, spec, b)
        else:                        # pcn_forward with no C-alpha list: lifting without re-anchoring
            S = torch.nn.functional.embedding(b["res"].long(), P["embedding.weight"], padding_idx=0)
            _, V = orc.decoder_stack_forward(P, "equivaraintconv", spec, b["ca_xyz"], b["CG_nbr_list"], S)
            out = (None, None, None, None, b["xyz"], orc.lift(V, b["ca_xyz"], b["cg_map"], offset=False))
        (out[5] - out[4]).pow(2).mean().backward()
        return {"ca_xyz": b["ca_xyz"].grad}

    got = run(None, dtype, dev)
    return got, lambda dt: run(_oracle_P(model, dt), dt, "cpu")
