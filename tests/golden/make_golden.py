"""Generates the committed fixtures under tests/golden/.

  python tests/golden/make_golden.py REFERENCE_CHECKOUT

* ``gat_ckpt.npz`` / ``tgn_ckpt.npz``: the reference's own trained weights
  (REFERENCE_CHECKOUT/results/gat_model.pt, tgn_model.pt of aum2606/GNN-Fraud-Detection -- the only golden artefacts
  the reference ships for this path), converted to numpy with the ``lin_dst.weight`` alias dropped (it is bit-identical
  to ``lin_src.weight``; asserted below).
* ``golden_small.npz``: a seeded small Elliptic-shaped input and the outputs of the ORACLE
  (oracle/pyg_gatconv.py) on it with those weights: layer-0 GATConv output + attention, full GAT and
  TemporalGNN eval-mode logits, and the CSR of the graph.  PyG itself is not installable here, so these
  are oracle outputs, not outputs of the reference running -- they pin the oracle against regressions
  and give the GPU tests a fixed target that does not need the reference at run time.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import pyg_gatconv as O  # noqa: E402
from gnn_fraud_detection_b200 import synth  # noqa: E402

def convert(name):
    sd = torch.load(os.path.join(sys.argv[1], "results", name), map_location="cpu", weights_only=False)
    out = {}
    for k, v in sd.items():
        if k.endswith("lin_dst.weight"):
            assert torch.equal(v, sd[k.replace("lin_dst", "lin_src")]), "lin_dst is expected to alias lin_src"
            continue
        out[k] = v.numpy()
    return out


def load_into(model, npz):
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in npz.items()}
    for k in list(sd):
        if k.endswith("lin_src.weight"):
            sd[k.replace("lin_src", "lin_dst")] = sd[k]
    model.load_state_dict(sd, strict=True)
    return model


def main():
    gat = convert("gat_model.pt")
    tgn = convert("tgn_model.pt")
    np.savez(os.path.join(HERE, "gat_ckpt.npz"), **gat)
    np.savez(os.path.join(HERE, "tgn_ckpt.npz"), **tgn)

    K = gat["gat_layers.0.lin_src.weight"].shape[1]          # 165 in the shipped checkpoints
    x, ei, ts = synth.elliptic_synth(num_nodes=600, num_edges=1400, num_feats=K, num_steps=7, seed=11)
    # make the edge cases part of the fixture: a few pre-existing self-loops and duplicate edges
    ei = torch.cat([ei, torch.tensor([[5, 17, 17, 300], [5, 17, 17, 301]]), ei[:, :6]], dim=1).contiguous()
    torch.manual_seed(0)
    m_gat = load_into(O.OracleGAT(K, 64, 1, num_layers=3), gat).eval()
    m_tgn = load_into(O.OracleTemporalGNN(K, 64, 1, num_layers=3), tgn).eval()
    with torch.no_grad():
        l0 = m_gat.gat_layers[0]
        out0, (ei2, alpha0) = l0(x, ei, return_attention_weights=True)
        logits_gat = m_gat(x, ei)
        logits_tgn, hid_tgn = m_tgn(x, ei)
        rowptr, col, perm, _ = O.csr_oracle(ei, x.size(0))
    np.savez(os.path.join(HERE, "golden_small.npz"), x=x.numpy(), edge_index=ei.numpy(), time_steps=ts.numpy(),
             layer0_out=out0.numpy(), layer0_alpha=alpha0.numpy(), edge_index_rewritten=ei2.numpy(),
             gat_logits=logits_gat.numpy(), tgn_logits=logits_tgn.numpy(), tgn_hidden=hid_tgn.numpy(),
             rowptr=rowptr.numpy(), col=col.numpy(), perm=perm.numpy())
    for f in ("gat_ckpt.npz", "tgn_ckpt.npz", "golden_small.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")


if __name__ == "__main__":
    main()
