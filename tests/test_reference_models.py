"""The reference's OWN model classes (src/models/gat.py, src/models/tgn.py) as stored in the committed fixture, against the
oracle's restatement of those classes and against the drop-in layer -- CPU side.

* ``tests/golden/reference_models_golden.npz`` holds the outputs of the reference's classes, run unmodified with
  ``torch_geometric.nn.GATConv`` stubbed to the CPU oracle layer (``tests/golden/make_reference_goldens.py``).  The
  oracle's restated wrappers (``OracleGAT`` / ``OracleTemporalGNN``) must reproduce it, so the fixture the GPU tests use
  and the oracle they compare with are the same function.
* With the layer swapped for THIS repo's ``GATConv`` (the one-line import swap of INTEGRATION.md), the classes construct,
  expose the same state_dict keys as the reference's checkpoints and load them with ``strict=True``."""
import os

import numpy as np
import pytest
import torch

from oracle import pyg_gatconv as O
from util import load_ckpt, oracle_model_outputs, relerr

HERE = os.path.dirname(os.path.abspath(__file__))


def test_fixture_is_the_reference_wrappers_output():
    gold = np.load(os.path.join(HERE, "golden", "reference_models_golden.npz"))
    small = np.load(os.path.join(HERE, "golden", "golden_small.npz"))
    x, ei = torch.from_numpy(small["x"]), torch.from_numpy(small["edge_index"])
    y = torch.from_numpy(gold["train_y"])
    assert torch.equal(y, torch.clamp(torch.from_numpy(small["time_steps"]) % 5 - 1, max=1))
    fresh = oracle_model_outputs(x, ei, y, os.path.join(HERE, "golden"))
    stored = sorted(k for k in gold.files if not k.endswith(".rows"))
    assert stored == sorted([k for k in fresh if not k.endswith("_f32")] + ["train_y"])
    for k in stored:
        if k == "train_y":
            continue
        ours = fresh[k]
        if k + ".rows" in gold.files:                   # a fixed sample of the rows of this gradient is stored
            ours = ours[torch.from_numpy(gold[k + ".rows"])]
        ref = torch.from_numpy(gold[k])
        assert ours.shape == ref.shape, k
        # the fixture stores float32 roundings of the fp64 values: one float32 ulp is 6e-8 relative
        if float(ref.double().norm()) > 1e-12:
            assert relerr(ours, ref) <= 1e-6, (k, relerr(ours, ref))
        else:
            assert float(ours.abs().max()) <= 1e-12, k
    # the reference's fp32 eval outputs are those of golden_small.npz (the oracle's restated wrappers made that file)
    for k, s in (("gat_logits_f32", "gat_logits"), ("tgn_logits_f32", "tgn_logits"), ("tgn_hidden_f32", "tgn_hidden")):
        assert relerr(fresh[k], torch.from_numpy(small[s])) <= 1e-6, k


def test_reference_classes_accept_the_drop_in_layer(monkeypatch):
    from gnn_fraud_detection_b200 import GATConv
    monkeypatch.setattr(O, "OracleGATConv", GATConv)     # the restated classes build their layers from this name
    for cls, ck in ((O.OracleGAT, "gat_ckpt.npz"), (O.OracleTemporalGNN, "tgn_ckpt.npz")):
        npz = np.load(os.path.join(HERE, "golden", ck))
        keys = set(npz.files) | {k.replace("lin_src", "lin_dst") for k in npz.files if k.endswith("lin_src.weight")}
        m = cls(165, 64, 1, num_layers=3)
        assert all(type(l) is GATConv for l in m.gat_layers)
        assert sorted(m.state_dict().keys()) == sorted(keys)
        load_ckpt(m, os.path.join(HERE, "golden", ck))
        for l in m.gat_layers:                      # the reference's ctor call: heads=8, concat=False, dropout=p
            assert (l.heads, l.concat, l.dropout) == (8, False, 0.2) and l.lin_dst is l.lin_src
        with pytest.raises(RuntimeError):           # the layer has no CPU path: the model must be moved to the GPU
            m(torch.randn(4, 165), torch.zeros(2, 0, dtype=torch.long))
