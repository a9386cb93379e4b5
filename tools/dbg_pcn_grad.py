"""worst weight-gradient tensors of the reduced c4 PCN step: kernel and fp32 oracle vs the float64 oracle."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import coarsegrainingvae_b200 as cg
from coarsegrainingvae_b200 import ops, synthetic
from oracle import cgvae_oracle as orc
from tests import parity_cases as pc
from tests.golden_util import rel_err
DEV = "cuda"
rad = lambda xyz, c: ops.radius_graph(torch.as_tensor(xyz, dtype=torch.float32, device=DEV), c).cpu().numpy()
cfg = dict(synthetic.CONFIGS["c4_protein"]); cfg["n_res"] = 60
batch = synthetic.pcn_batch(cfg, 0, rad, n_proteins=2)
torch.manual_seed(123)
net = cg.EquivariantDecoder(n_atom_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], cutoff=cfg["cg_cutoff"], num_conv=cfg["dec_nconv"], activation="swish", cross_flag=True)
model = cg.PCN(net, feature_dim=cfg["n_basis"], offset=False).to(DEV)
out = model({k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in batch.items()})
((out[5] - out[4]).pow(2).mean()).backward()
spec = dict(n_basis=cfg["n_basis"], n_rbf=cfg["n_rbf"], dec_nconv=cfg["dec_nconv"], atom_cutoff=cfg["cg_cutoff"], decoder="cross", activation="swish")
P = pc._oracle_params(model)
o = orc.pcn_forward(P, spec, batch); ((o[5] - o[4]).pow(2).mean()).backward()
P64 = {k: v.detach().double().requires_grad_(v.dtype.is_floating_point) for k, v in P.items()}
b64 = {k: (v.double() if torch.is_tensor(v) and v.dtype.is_floating_point else v) for k, v in batch.items()}
o64 = orc.pcn_forward(P64, spec, b64); ((o64[5] - o64[4]).pow(2).mean()).backward()
rows = []
for k, p in model.named_parameters():
    if P[k].grad is None or p.grad is None or float(P[k].grad.abs().max()) == 0: continue
    rows.append((rel_err(p.grad, P[k].grad), rel_err(p.grad, P64[k].grad), rel_err(P[k].grad, P64[k].grad), k))
rows.sort(reverse=True)
print("%-12s %-12s %-12s %s" % ("kern-vs-f32", "kern-vs-f64", "f32-vs-f64", "tensor"))
for r in rows[:6]: print("%-12.3e %-12.3e %-12.3e %s" % r)
