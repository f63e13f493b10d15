"""Golden vectors produced by the reference's OWN model code.

  python tests/golden/make_reference_goldens.py REFERENCE_CHECKOUT

``REFERENCE_CHECKOUT/src/models/gat.py`` and ``tgn.py`` (a checkout of aum2606/GNN-Fraud-Detection) are imported
UNMODIFIED (importlib, from where they lie).  Their
only missing import is third-party ``torch_geometric.nn.GATConv`` (not installable here), which is satisfied by a stub
module exposing the CPU oracle layer (``oracle.pyg_gatconv.OracleGATConv``).  The reference's classes -- constructor
logic, layer loop, BatchNorm / ReLU / dropout / residual, GRUCell head, ``predict`` -- then run exactly as shipped, load the
reference's own checkpoints (``results/gat_model.pt`` / ``tgn_model.pt``) with ``strict=True``, and their outputs are
stored in ``reference_models_golden.npz``:

  * eval-mode logits of GAT / TemporalGNN (+ hidden state) on the ``golden_small.npz`` inputs, fp32 and fp64;
  * one TRAIN-mode step (BatchNorm batch statistics; dropout 0 so it is deterministic) of each reference model with the
    reference's loss (masked ``BCEWithLogitsLoss(pos_weight=50)``, ``src/train.py:108-139,360-361``) in fp64: loss, logits
    and the gradient of every parameter.

To keep the file under 1 MB, ``shrink`` stores every float array as float32 (its rounding is three orders of magnitude
below the tolerances of the tests that read it) and, of each weight gradient with more than 64 rows, a fixed seeded half
of its rows (their indices under ``<name>.rows``).  The fp32 eval outputs are not stored: they are bit-identical to
``golden_small.npz``'s ``gat_logits`` / ``tgn_logits`` / ``tgn_hidden``.

The reference is not part of this repository, so the tests compare with THIS file: the GPU tests the CUDA models, and
``tests/test_reference_models.py`` the oracle's restated wrappers (which reproduced it bit for bit in fp64).
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
ROW_SAMPLE_MIN_ROWS = 64


def load_reference_models(gatconv_cls, ref):
    """The reference's ``GAT`` / ``TemporalGNN`` classes with ``torch_geometric.nn.GATConv`` := ``gatconv_cls``."""
    saved = {k: sys.modules.get(k) for k in ("torch_geometric", "torch_geometric.nn", "src", "src.config")}
    tg, tgnn = types.ModuleType("torch_geometric"), types.ModuleType("torch_geometric.nn")
    tgnn.GATConv = gatconv_cls
    tg.nn = tgnn
    sys.modules["torch_geometric"], sys.modules["torch_geometric.nn"] = tg, tgnn
    # tgn.py does `from src.config import MODEL_CONFIG` (never used): load the reference's config the same way
    src_pkg = types.ModuleType("src")
    src_pkg.__path__ = [os.path.join(ref, "src")]
    sys.modules["src"] = src_pkg
    mods = {}
    try:
        for name, rel in (("src.config", "src/config.py"), ("_ref_gat", "src/models/gat.py"), ("_ref_tgn", "src/models/tgn.py")):
            spec = importlib.util.spec_from_file_location(name, os.path.join(ref, rel))
            m = importlib.util.module_from_spec(spec)
            sys.modules[name] = m
            spec.loader.exec_module(m)
            mods[name] = m
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mods["_ref_gat"].GAT, mods["_ref_tgn"].TemporalGNN


def reference_outputs(ref):
    from oracle import pyg_gatconv as O
    RefGAT, RefTGN = load_reference_models(O.OracleGATConv, ref)
    gold = np.load(os.path.join(HERE, "golden_small.npz"))
    x, ei = torch.from_numpy(gold["x"]), torch.from_numpy(gold["edge_index"])
    K = x.size(1)
    out = {}
    sds = {}
    for name, cls, ck in (("gat", RefGAT, "gat_model.pt"), ("tgn", RefTGN, "tgn_model.pt")):
        sd = torch.load(os.path.join(ref, "results", ck), map_location="cpu", weights_only=False)
        sds[name] = sd
        m = cls(K, 64, 1, num_layers=3)                         # compare_gnn_models.py:35-54
        m.load_state_dict(sd, strict=True)                      # src/evaluate.py:173-176
        m.eval()
        with torch.no_grad():
            r32 = m(x, ei)
            # (tgn.py:88-89 creates its zero state in fp32: the fp64 run passes the same zero state explicitly)
            kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if name == "tgn" else {}
            r64 = m.double()(x.double(), ei, **kw)
        if name == "tgn":
            out["tgn_logits_f32"], out["tgn_hidden_f32"] = r32[0].numpy(), r32[1].numpy()
            out["tgn_logits_f64"], out["tgn_hidden_f64"] = r64[0].numpy(), r64[1].numpy()
        else:
            out["gat_logits_f32"], out["gat_logits_f64"] = r32.numpy(), r64.numpy()
    # one deterministic training step of the reference models, fp64
    y = torch.from_numpy(gold["time_steps"]) % 5 - 1            # labels in {-1, 0, 1, 2, 3} -> clamp to {-1,0,1}
    y = torch.clamp(y, max=1)
    out["train_y"] = y.numpy()
    mask = y != -1                                              # src/train.py:108
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, dtype=torch.float64))   # src/train.py:360-361
    for name, cls in (("gat", RefGAT), ("tgn", RefTGN)):
        m = cls(K, 64, 1, num_layers=3, dropout=0.0)
        m.load_state_dict(sds[name], strict=True)
        m = m.double().train()
        kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if name == "tgn" else {}
        r = m(x.double(), ei, **kw)
        logits = r[0] if name == "tgn" else r
        loss = crit(logits[mask].squeeze(1), y[mask].double())  # src/train.py:131-139
        loss.backward()
        out[f"train_{name}_loss"] = np.array(float(loss))
        out[f"train_{name}_logits"] = logits.detach().numpy()
        for pn, p in m.named_parameters():
            if "lin_dst" in pn:
                continue
            out[f"train_{name}_grad.{pn}"] = p.grad.numpy()
    return out


def shrink(full):
    """What the fixture stores of ``reference_outputs()`` (see the module docstring)."""
    out = {}
    for k, a in full.items():
        a = np.asarray(a)
        if k.endswith("_f32"):
            continue
        if a.dtype == np.float64 and a.ndim > 0:
            a = a.astype(np.float32)
        if k.startswith("train_") and "_grad." in k and a.ndim == 2 and a.shape[0] > ROW_SAMPLE_MIN_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], a.shape[0] // 2, replace=False))
            out[k + ".rows"] = rows
            a = a[rows]
        out[k] = a
    return out


def main():
    out = shrink(reference_outputs(sys.argv[1]))
    path = os.path.join(HERE, "reference_models_golden.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes;", len(out), "arrays")


if __name__ == "__main__":
    main()
