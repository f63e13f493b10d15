"""GPU parity at model level: GAT / TemporalGNN (the reference's classes, src/models/gat.py, tgn.py) with the
reference's own trained checkpoints, eval mode, against the golden fixtures and the oracle."""
import os

import numpy as np
import pytest
import torch

from gnn_fraud_detection_b200 import GAT, TemporalGNN, synth
from oracle import pyg_gatconv as O
from util import load_ckpt, maxabs, oracle_model_outputs, relerr

pytestmark = pytest.mark.gpu


def test_gat_and_tgn_eval_match_golden(golden_dir):
    gold = np.load(os.path.join(golden_dir, "golden_small.npz"))
    x, ei = torch.from_numpy(gold["x"]).cuda(), torch.from_numpy(gold["edge_index"]).cuda()
    gat = load_ckpt(GAT(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, "gat_ckpt.npz")).cuda().eval()
    tgn = load_ckpt(TemporalGNN(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, "tgn_ckpt.npz")).cuda().eval()
    with torch.no_grad():
        lg = gat(x, ei)
        lt, ht = tgn(x, ei)
        pg = gat.predict(x, ei)
    # three stacked layers + BatchNorm with trained running stats amplify rounding: 1e-4 at the logits
    assert np.abs(lg.cpu().numpy() - gold["gat_logits"]).max() <= 1e-4
    assert np.abs(lt.cpu().numpy() - gold["tgn_logits"]).max() <= 1e-4
    assert np.abs(ht.cpu().numpy() - gold["tgn_hidden"]).max() <= 1e-4
    assert torch.allclose(pg, torch.sigmoid(lg))
    assert lg.shape == (x.size(0), 1) and ht.shape == (x.size(0), 64)


def test_gat_training_step_matches_oracle_full_batch():
    """One full-batch training step (train mode, dropout off so it is deterministic) of the 2-layer default GAT
    (BASELINE config #1/#2 model) on a reduced Elliptic-shaped graph: logits and every parameter gradient."""
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    torch.manual_seed(0)
    # the truth is the oracle evaluated in fp64: through BatchNorm + BCE(pos_weight=50) the fp32 CPU oracle's own
    # sequential sums are off by up to 3e-3 relative (measured, scripts/diag_parity.py), ours by < 1e-6
    ref = O.OracleGAT(166, 64, 1, num_layers=2, dropout=0.0).double()
    ours = GAT(166, 64, 1, num_layers=2, dropout=0.0)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)   # identical fp32 values
    ours = ours.cuda()
    y = (torch.rand(x.size(0), 1, generator=torch.Generator().manual_seed(1)) < 0.1).float()
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0))        # src/train.py:360-361
    lr = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0).double())(ref(x.double(), ei), y.double()); lr.backward()
    lo = crit.cuda()(ours(x.cuda(), ei.cuda()), y.cuda()); lo.backward()
    assert abs(float(lr) - float(lo)) <= 1e-5
    for (n, p_ref), (_, p_our) in zip(ref.named_parameters(), ours.named_parameters()):
        assert maxabs(p_our.grad, p_ref.grad) <= 1e-5, n
        if float(p_ref.grad.norm()) > 1e-6:        # (the pre-BatchNorm conv bias has an exactly-zero true gradient)
            # through two layers the tensor-core GEMM chains (dx, dW: ~4e-6 each) compound: 3e-5 bound
            assert relerr(p_our.grad, p_ref.grad) <= 3e-5, n


def test_tgn_snapshots_independent():
    """BASELINE config #3: the 49 time-step snapshots are disconnected, so running TemporalGNN on the whole
    graph equals running it snapshot by snapshot (eval mode)."""
    x, ei, ts = synth.elliptic_synth(num_nodes=30_000, num_edges=34_000, num_feats=166, seed=0)
    torch.manual_seed(0)
    m = TemporalGNN(166, 64, 1, num_layers=2).cuda().eval()
    with torch.no_grad():
        full, hid = m(x.cuda(), ei.cuda())
        for t in (1, 17, 49):
            xt, et, idx = O.temporal_subgraph_oracle(x, ei, ts, t)
            lt, ht = m(xt.cuda(), et.cuda())
            assert maxabs(lt, full[idx.cuda()]) <= 1e-5 and maxabs(ht, hid[idx.cuda()]) <= 1e-5


def test_fused_eval_epilogue_matches_unfused_and_oracle(golden_dir):
    """SURVEY 8(f) rank 1: BatchNorm(eval) + ReLU + residual fused into the aggregation epilogue (the no_grad
    inference path) must equal the un-fused layer loop and the oracle."""
    gold = np.load(os.path.join(golden_dir, "golden_small.npz"))
    x, ei = torch.from_numpy(gold["x"]).cuda(), torch.from_numpy(gold["edge_index"]).cuda()
    gat = load_ckpt(GAT(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, "gat_ckpt.npz")).cuda().eval()
    with torch.no_grad():
        fused = gat(x, ei)                              # fused path (eval + no_grad)
    with torch.enable_grad():
        unfused = gat(x, ei).detach()                   # grad enabled => plain torch BatchNorm/ReLU/residual ops
    assert maxabs(fused, unfused) <= 1e-5
    assert np.abs(fused.cpu().numpy() - gold["gat_logits"]).max() <= 1e-4
    # layer-level: every epilogue option against torch ops
    from gnn_fraud_detection_b200 import GATConv
    torch.manual_seed(3)
    conv = GATConv(64, 64, heads=8, concat=False).cuda().eval()
    bn = torch.nn.BatchNorm1d(64).cuda().eval()
    with torch.no_grad():
        bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2.0); bn.weight.normal_(); bn.bias.normal_()
        h = torch.randn(x.size(0), 64, device="cuda")
        ref = h + torch.relu(bn(conv(h, ei)))
        got = conv.forward_fused_eval(h, ei, bn, relu=True, residual=h)
        assert maxabs(got, ref) <= 1e-5
        assert maxabs(conv.forward_fused_eval(h, ei, None, relu=False), conv(h, ei)) <= 1e-6


def test_models_match_the_reference_wrappers_own_outputs(golden_dir):
    """reference_models_golden.npz = the reference's unmodified GAT / TemporalGNN classes (layer := CPU oracle) with the
    reference's checkpoints: eval logits, and one full training step (train-mode BatchNorm, masked BCE(pos_weight=50),
    dropout 0) in fp64 -- loss, logits and every parameter gradient (stored as float32, half the rows of the large ones)."""
    gold = np.load(os.path.join(golden_dir, "reference_models_golden.npz"))
    small = np.load(os.path.join(golden_dir, "golden_small.npz"))
    x, ei = torch.from_numpy(small["x"]).cuda(), torch.from_numpy(small["edge_index"]).cuda()
    y = torch.from_numpy(gold["train_y"]).cuda()
    mask = y != -1
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, device="cuda"))
    oracle = oracle_model_outputs(x.cpu(), ei.cpu(), y.cpu(), golden_dir)
    for name, cls, ck in (("gat", GAT, "gat_ckpt.npz"), ("tgn", TemporalGNN, "tgn_ckpt.npz")):
        m = load_ckpt(cls(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, ck)).cuda().eval()
        with torch.no_grad():
            r = m(x, ei)
        lg = r[0] if name == "tgn" else r
        assert np.abs(lg.cpu().numpy() - gold[f"{name}_logits_f64"]).max() <= 1e-4
        if name == "tgn":
            assert np.abs(r[1].cpu().numpy() - gold["tgn_hidden_f64"]).max() <= 1e-4
        # training step
        m = load_ckpt(cls(x.size(1), 64, 1, num_layers=3, dropout=0.0), os.path.join(golden_dir, ck)).cuda().train()
        r = m(x, ei)
        lg = r[0] if name == "tgn" else r
        loss = crit(lg[mask].squeeze(1), y[mask].float())
        loss.backward()
        assert abs(float(loss) - float(gold[f"train_{name}_loss"])) <= 1e-4 * float(gold[f"train_{name}_loss"])
        assert relerr(lg, torch.from_numpy(gold[f"train_{name}_logits"])) <= 1e-5
        for pn, p in m.named_parameters():
            if "lin_dst" in pn:
                continue
            key = f"train_{name}_grad.{pn}"
            # the fixture keeps a fixed sample of the rows of the large gradients; every row is checked against the
            # oracle's restated wrappers, which reproduce the fixture (tests/test_reference_models.py)
            rows = torch.from_numpy(gold[key + ".rows"]).cuda() if key + ".rows" in gold.files else None
            for grad, ref in ((p.grad if rows is None else p.grad[rows], torch.from_numpy(gold[key])), (p.grad, oracle[key])):
                if float(ref.norm()) > 1e-9:    # (conv biases feed a train-mode BatchNorm: their true gradient is zero)
                    assert relerr(grad, ref) <= 2e-4, (name, pn, relerr(grad, ref))
                else:
                    assert maxabs(grad, ref) <= 1e-5, (name, pn)
