"""CPU tests that pin the oracle: closed-form cases, fp64 autograd vs closed-form backward, index oracles
cross-checked three ways (torch stable sort, C counting sort, numpy), golden fixtures."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import build_c
from oracle import pyg_gatconv as O
from gnn_fraud_detection_b200 import synth


def _params(K, H, Cc, dtype=torch.float64, seed=0):
    g = torch.Generator().manual_seed(seed)
    W = O.glorot_(torch.empty(H * Cc, K, dtype=dtype), g)
    a_s = O.glorot_(torch.empty(1, H, Cc, dtype=dtype), g)
    a_d = O.glorot_(torch.empty(1, H, Cc, dtype=dtype), g)
    b = torch.randn(Cc, dtype=dtype, generator=g) * 0.1
    return W, a_s, a_d, b


def test_single_node_closed_form():
    # one node, no edges: only the self-loop -> alpha == 1, out = mean_h(xw) + bias
    K, H, Cc = 5, 8, 64
    W, a_s, a_d, b = _params(K, H, Cc)
    x = torch.randn(1, K, dtype=torch.float64)
    out, (ei, alpha) = O.gatconv_forward(x, torch.zeros(2, 0, dtype=torch.long), W, a_s, a_d, b, H, Cc)
    assert ei.tolist() == [[0], [0]]
    assert torch.allclose(alpha, torch.ones(1, H, dtype=torch.float64))
    assert torch.allclose(out, (x @ W.t()).view(1, H, Cc).mean(1) + b, atol=1e-12)


def test_three_node_hand_computed():
    # edges 0->2, 1->2 (+ self loops): softmax over {0,1,2} at node 2, hand-evaluated
    K, H, Cc = 3, 8, 64
    W, a_s, a_d, b = _params(K, H, Cc, seed=3)
    x = torch.randn(3, K, dtype=torch.float64)
    ei = torch.tensor([[0, 1], [2, 2]])
    out, (ei2, alpha) = O.gatconv_forward(x, ei, W, a_s, a_d, b, H, Cc)
    assert ei2.tolist() == [[0, 1, 0, 1, 2], [2, 2, 0, 1, 2]]
    xw = (x @ W.t()).view(3, H, Cc)
    asrc, adst = (xw * a_s).sum(-1), (xw * a_d).sum(-1)
    for h in range(H):
        e = torch.stack([asrc[j, h] + adst[2, h] for j in (0, 1, 2)])
        e = torch.where(e > 0, e, 0.2 * e)
        w = torch.exp(e - e.max())
        w = w / w.sum()
        assert torch.allclose(alpha[[0, 1, 4], h], w, atol=1e-12)
        got = (out[2] - b) * 1.0
    exp2 = sum((alpha[[0, 1, 4], h][:, None] * xw[[0, 1, 2], h]).sum(0) for h in range(H)) / H + b
    assert torch.allclose(out[2], exp2, atol=1e-12)
    assert torch.allclose(out[0], xw[0].mean(0) + b, atol=1e-12)      # nodes 0,1 only see themselves


def test_self_loop_rewrite_order_and_duplicates():
    ei = torch.tensor([[3, 1, 1, 2, 2, 0], [3, 1, 0, 0, 0, 2]])          # two self loops, one duplicate
    out = O.rewrite_self_loops(ei, 4)
    assert out.tolist() == [[1, 2, 2, 0, 0, 1, 2, 3], [0, 0, 0, 2, 0, 1, 2, 3]]
    assert O.rewrite_self_loops(ei, 4, add_self_loops=False) is ei


@pytest.mark.parametrize("concat", [False, True])
def test_closed_form_backward_matches_autograd_fp64(concat):
    N, E, K, H, Cc = 40, 150, 7, 8, 64
    W, a_s, a_d, _ = _params(K, H, Cc, seed=1)
    b = torch.zeros(H * Cc if concat else Cc, dtype=torch.float64)
    x = torch.randn(N, K, dtype=torch.float64)
    ei = synth.random_graph(N, E, seed=5)
    leaves = [t.clone().requires_grad_(True) for t in (x, W, a_s, a_d, b)]
    out, _ = O.gatconv_forward(leaves[0], ei, leaves[1], leaves[2], leaves[3], leaves[4], H, Cc, concat=concat)
    d_out = torch.randn_like(out)
    out.backward(d_out)
    cf = O.gatconv_backward_closed_form(x, ei, W, a_s, a_d, H, Cc, d_out, concat=concat)
    for name, g in zip(("dx", "dW", "datt_src", "datt_dst", "dbias"), [l.grad for l in leaves]):
        assert torch.allclose(cf[name], g, atol=1e-11, rtol=1e-10), name


def test_gradcheck_fp64():
    N, E, K, H, Cc = 6, 14, 3, 8, 64
    W, a_s, a_d, b = _params(K, H, Cc, seed=2)
    x = torch.randn(N, K, dtype=torch.float64, requires_grad=True)
    W = W.requires_grad_(True)
    ei = synth.random_graph(N, E, seed=9)
    fn = lambda x_, W_: O.gatconv_forward(x_, ei, W_, a_s, a_d, b, H, Cc)[0]
    assert torch.autograd.gradcheck(fn, (x, W), eps=1e-6, atol=1e-6, nondet_tol=0.0)


def test_dropout_mask_injection():
    N, E, K, H, Cc = 30, 90, 4, 8, 64
    W, a_s, a_d, b = _params(K, H, Cc, dtype=torch.float32)
    x = torch.randn(N, K)
    ei = synth.random_graph(N, E, seed=2)
    Ep = O.rewrite_self_loops(ei, N).size(1)
    keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(1)) >= 0.2
    out, (ei2, alpha) = O.gatconv_forward(x, ei, W, a_s, a_d, b, H, Cc, dropout_mask=keep, p=0.2)
    xw = (x @ W.t()).view(N, H, Cc)
    ref = torch.zeros(N, H, Cc).index_add_(0, ei2[1], (alpha * keep / 0.8)[:, :, None] * xw[ei2[0]]).mean(1) + b
    assert torch.allclose(out, ref, atol=1e-6)


def _c_oracle():
    lib = C.CDLL(build_c.build())
    lib.gnnfd_oracle_csr.restype = C.c_int64
    lib.gnnfd_oracle_csr.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int] + [C.c_void_p] * 3
    lib.gnnfd_oracle_csc.restype = None
    lib.gnnfd_oracle_csc.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64] + [C.c_void_p] * 3
    return lib


@pytest.mark.parametrize("N,E,loops", [(1, 0, True), (7, 0, True), (50, 300, True), (50, 300, False),
                                       (1000, 20000, True), (513, 4097, True), (3, 50, True)])
def test_csr_oracle_three_ways(N, E, loops):
    ei = synth.random_graph(N, E, seed=N + E)
    rowptr, col, perm, ei2 = O.csr_oracle(ei, N, loops)
    Ep = ei2.size(1)
    # (a) numpy stable argsort
    d = ei2[1].numpy()
    p_np = np.argsort(d, kind="stable")
    assert np.array_equal(perm.numpy(), p_np)
    assert np.array_equal(col.numpy(), ei2[0].numpy()[p_np])
    assert np.array_equal(rowptr.numpy(), np.concatenate([[0], np.cumsum(np.bincount(d, minlength=N))]))
    # (b) C counting sort
    lib = _c_oracle()
    cap = E + N
    r2, c2, p2 = (np.zeros(N + 1, np.int64), np.zeros(max(cap, 1), np.int64), np.zeros(max(cap, 1), np.int64))
    ein = np.ascontiguousarray(ei.numpy())
    got = lib.gnnfd_oracle_csr(ein.ctypes.data, E, N, int(loops), r2.ctypes.data, c2.ctypes.data, p2.ctypes.data)
    assert got == Ep
    assert np.array_equal(r2, rowptr.numpy()) and np.array_equal(c2[:Ep], col.numpy()) and np.array_equal(p2[:Ep], perm.numpy())
    if loops and Ep:
        # stable => the self-loop is the last entry of every row
        last = rowptr[1:] - 1
        assert torch.equal(col[last], torch.arange(N))
    # CSC twin
    colptr, row, eid = O.csc_oracle(rowptr, col, N)
    cp, rw, ed = np.zeros(N + 1, np.int64), np.zeros(max(Ep, 1), np.int64), np.zeros(max(Ep, 1), np.int64)
    lib.gnnfd_oracle_csc(r2.ctypes.data, c2.ctypes.data, N, Ep, cp.ctypes.data, rw.ctypes.data, ed.ctypes.data)
    assert np.array_equal(cp, colptr.numpy()) and np.array_equal(rw[:Ep], row.numpy()) and np.array_equal(ed[:Ep], eid.numpy())


def test_c_oracle_rejects_out_of_range():
    lib = _c_oracle()
    ein = np.array([[0, 5], [1, 1]], np.int64)
    buf = np.zeros(16, np.int64)
    assert lib.gnnfd_oracle_csr(ein.ctypes.data, 2, 3, 1, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data) == -1


def test_temporal_subgraph_intent():
    x, ei, ts = synth.elliptic_synth(num_nodes=400, num_edges=900, num_feats=6, num_steps=5, seed=3)
    tot_n = tot_e = 0
    for t in range(1, 6):
        xt, et, idx = O.temporal_subgraph_oracle(x, ei, ts, t)
        assert torch.equal(xt, x[idx]) and torch.all(ts[idx] == t)
        assert et.numel() == 0 or (et.min() >= 0 and et.max() < idx.numel())
        # order preserved and endpoints relabelled back to the originals
        keep = (ts[ei[0]] == t) & (ts[ei[1]] == t)
        assert torch.equal(idx[et], ei[:, keep])
        tot_n += idx.numel(); tot_e += et.size(1)
    assert tot_n == 400 and tot_e == 900          # snapshots are disconnected: nothing is lost


def _load_ckpt(model, path):
    npz = np.load(path)
    sd = {k: torch.from_numpy(npz[k]) for k in npz.files}
    for k in list(sd):
        if k.endswith("lin_src.weight"):
            sd[k.replace("lin_src", "lin_dst")] = sd[k]
    model.load_state_dict(sd, strict=True)
    return model.eval()


def test_reference_checkpoints_load_strict_and_golden_vectors(golden_dir):
    gold = np.load(os.path.join(golden_dir, "golden_small.npz"))
    x, ei = torch.from_numpy(gold["x"]), torch.from_numpy(gold["edge_index"])
    gat = _load_ckpt(O.OracleGAT(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, "gat_ckpt.npz"))
    tgn = _load_ckpt(O.OracleTemporalGNN(x.size(1), 64, 1, num_layers=3), os.path.join(golden_dir, "tgn_ckpt.npz"))
    assert gat.batch_norms[0].num_batches_tracked.item() == 100      # 100 full-batch steps (SURVEY 0.4)
    with torch.no_grad():
        out0, (ei2, alpha0) = gat.gat_layers[0](x, ei, return_attention_weights=True)
        assert np.allclose(out0.numpy(), gold["layer0_out"], atol=1e-6)
        assert np.allclose(alpha0.numpy(), gold["layer0_alpha"], atol=1e-6)
        assert np.array_equal(ei2.numpy(), gold["edge_index_rewritten"])
        assert np.allclose(gat(x, ei).numpy(), gold["gat_logits"], atol=1e-5)
        lt, ht = tgn(x, ei)
        assert np.allclose(lt.numpy(), gold["tgn_logits"], atol=1e-5) and np.allclose(ht.numpy(), gold["tgn_hidden"], atol=1e-5)
        # fp32 oracle vs its own fp64 evaluation: the restatement's rounding noise is far below 1e-5
        l0 = gat.gat_layers[0]
        o64, (_, a64) = O.gatconv_forward(x.double(), ei, l0.lin_src.weight.double(), l0.att_src.double(),
                                          l0.att_dst.double(), l0.bias.double(), 8, 64)
        assert (o64 - out0.double()).abs().max() < 2e-6 and (a64 - alpha0.double()).abs().max() < 2e-6
    rowptr, col, perm, _ = O.csr_oracle(ei, x.size(0))
    assert np.array_equal(rowptr.numpy(), gold["rowptr"]) and np.array_equal(col.numpy(), gold["col"])
    assert np.array_equal(perm.numpy(), gold["perm"])


def test_glorot_bounds():
    t = O.glorot_(torch.empty(512, 166))
    assert t.abs().max() <= math.sqrt(6 / (512 + 166)) + 1e-7


def test_csr_oracle_dst_src_order_matches_numpy_lexsort():
    """order="dst_src" (PyG sort_edge_index(sort_by_row=False)) against an independent statement: numpy lexsort on
    (src, dst) is stable, so duplicates keep their order of appearance."""
    import numpy as np
    from gnn_fraud_detection_b200 import synth
    for N, E, loops in [(7, 40, True), (50, 400, False), (300, 5000, True)]:
        ei = synth.random_graph(N, E, seed=N + E)
        rowptr, col, perm, ei2 = O.csr_oracle(ei, N, loops, order="dst_src")
        src, dst = ei2[0].numpy(), ei2[1].numpy()
        ref = np.lexsort((src, dst))                    # last key is the primary one
        assert np.array_equal(perm.numpy(), ref)
        assert np.array_equal(col.numpy(), src[ref])
        assert np.array_equal(np.diff(rowptr.numpy()), np.bincount(dst, minlength=N))


@pytest.mark.parametrize("concat", [False, True])
def test_forward_matches_a_pure_python_loop_restatement(concat):
    """A second, independent statement of the published algorithm -- explicit Python loops over nodes, edges and heads in
    plain ``float`` arithmetic, no tensor ops: self-loop rewrite, per-destination LeakyReLU + max-subtracted softmax with the
    ``+1e-16``, weighted sum of projected source rows, head mean / concat, bias.  Small graph with duplicate edges, input
    self loops, an isolated node and a hub; fp64 oracle must agree to rounding."""
    import math
    import random
    rnd = random.Random(11)
    N, E, K, H, Cc = 9, 40, 5, 3, 4
    src = [rnd.randrange(N - 1) for _ in range(E)]          # node N-1 never appears: it only gets its self loop
    dst = [rnd.randrange(N - 1) if rnd.random() < 0.6 else 2 for _ in range(E)]      # node 2 is a hub
    src[3], dst[3] = 4, 4                                   # input self loops (dropped, then re-added once)
    src[7], dst[7] = 2, 2
    src[9], dst[9] = src[8], dst[8]                         # a duplicate edge counts twice
    W, a_s, a_d, b = _params(K, H, Cc, seed=5)
    if concat:
        b = torch.randn(H * Cc, dtype=torch.float64)
    x = torch.randn(N, K, dtype=torch.float64)
    out, (ei2, alpha) = O.gatconv_forward(x, torch.tensor([src, dst]), W, a_s, a_d, b, H, Cc, concat=concat)

    Wl, xl = W.tolist(), x.tolist()
    asl, adl, bl = a_s.reshape(H, Cc).tolist(), a_d.reshape(H, Cc).tolist(), b.tolist()
    edges = [(s, d) for s, d in zip(src, dst) if s != d] + [(n, n) for n in range(N)]
    assert ei2.t().tolist() == [list(e) for e in edges]
    xw = [[[sum(xl[n][k] * Wl[h * Cc + c][k] for k in range(K)) for c in range(Cc)] for h in range(H)] for n in range(N)]
    asrc = [[sum(xw[n][h][c] * asl[h][c] for c in range(Cc)) for h in range(H)] for n in range(N)]
    adst = [[sum(xw[n][h][c] * adl[h][c] for c in range(Cc)) for h in range(H)] for n in range(N)]
    exp_alpha = [[0.0] * H for _ in edges]
    exp_out = []
    for i in range(N):
        mine = [e for e, (_, d) in enumerate(edges) if d == i]
        heads = []
        for h in range(H):
            z = [asrc[edges[e][0]][h] + adst[i][h] for e in mine]
            z = [v if v > 0 else 0.2 * v for v in z]
            m = max(z)
            p = [math.exp(v - m) for v in z]
            tot = sum(p) + 1e-16
            acc = [0.0] * Cc
            for e, pe in zip(mine, p):
                exp_alpha[e][h] = pe / tot
                for c in range(Cc):
                    acc[c] += pe / tot * xw[edges[e][0]][h][c]
            heads.append(acc)
        if concat:
            exp_out.append([heads[h][c] + bl[h * Cc + c] for h in range(H) for c in range(Cc)])
        else:
            exp_out.append([sum(heads[h][c] for h in range(H)) / H + bl[c] for c in range(Cc)])
    assert torch.allclose(alpha, torch.tensor(exp_alpha, dtype=torch.float64), atol=1e-13)
    assert torch.allclose(out, torch.tensor(exp_out, dtype=torch.float64), atol=1e-12)


def _model_masks(model, x, ei, gen, p):
    n_edges = O.rewrite_self_loops(ei, x.size(0)).size(1)
    L, hid = len(model.gat_layers), model.hidden_channels
    att = [torch.rand(n_edges, 8, generator=gen) >= p for _ in range(L)]
    feat = [torch.rand(x.size(0), hid, generator=gen) >= p for _ in range(L)]
    return att, feat


@pytest.mark.parametrize("cls", [O.OracleGAT, O.OracleTemporalGNN])
def test_models_with_all_ones_masks_and_unit_scale_equal_the_dropout_free_model(cls):
    x, ei, _ = synth.elliptic_synth(num_nodes=300, num_edges=400, num_feats=12, seed=0)
    x = x.double()
    torch.manual_seed(0)
    m = cls(12, 64, 1, num_layers=3, dropout=0.3).double().train()
    m0 = cls(12, 64, 1, num_layers=3, dropout=0.0).double().train()
    m0.load_state_dict(m.state_dict(), strict=True)
    ones_a = [torch.ones(O.rewrite_self_loops(ei, x.size(0)).size(1), 8, dtype=torch.bool)] * 3
    ones_f = [torch.ones(x.size(0), 64, dtype=torch.bool)] * 3
    kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if cls is O.OracleTemporalGNN else {}
    r = m(x, ei, att_masks=ones_a, feat_masks=ones_f, dropout_scale=1.0, **kw)
    r0 = m0(x, ei, **kw)
    out, out0 = (r[0], r0[0]) if isinstance(r, tuple) else (r, r0)
    assert torch.equal(out, out0)
    out.square().sum().backward()
    out0.square().sum().backward()
    for (n, pa), (_, pb) in zip(m.named_parameters(), m0.named_parameters()):
        assert torch.equal(pa.grad, pb.grad), n


@pytest.mark.parametrize("cls", [O.OracleGAT, O.OracleTemporalGNN])
@pytest.mark.parametrize("p", [0.2, 0.5])
def test_models_with_injected_masks_equal_a_loop_restatement_with_f_dropout(cls, p):
    """The oracle's explicit-mask path against the reference's layer loop (src/models/gat.py:78-96) written out with the
    same masks: attention dropout through ``gatconv_forward`` (``mask / (1-p)``) and feature dropout through ``F.dropout``
    itself, under a seed whose draws are the injected feature masks."""
    x, ei, _ = synth.elliptic_synth(num_nodes=300, num_edges=400, num_feats=12, seed=1)
    x = x.double()
    torch.manual_seed(0)
    m = cls(12, 64, 1, num_layers=3, dropout=p).double().train()
    att, _ = _model_masks(m, x, ei, torch.Generator().manual_seed(5), p)
    # the feature masks F.dropout draws for [N,64] under seeds 100 + i
    feat = []
    for i in range(3):
        torch.manual_seed(100 + i)
        feat.append(F.dropout(torch.ones(x.size(0), 64, dtype=torch.float64), p=p, training=True) != 0)
    kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if cls is O.OracleTemporalGNN else {}
    r = m(x, ei, att_masks=att, feat_masks=feat, **kw)
    got = r[0] if isinstance(r, tuple) else r

    h = x
    for i, conv in enumerate(m.gat_layers):
        z, _ = O.gatconv_forward(h, ei, conv.lin_src.weight, conv.att_src, conv.att_dst, conv.bias, 8, 64,
                                 dropout_mask=att[i], p=p)
        bn = m.batch_norms[i]
        z = F.relu(F.batch_norm(z, None, None, bn.weight, bn.bias, training=True, eps=bn.eps))
        torch.manual_seed(100 + i)
        z = F.dropout(z, p=p, training=True)
        h = h + z if h.size(-1) == z.size(-1) else z
    if cls is O.OracleTemporalGNN:
        h = m.gru(h, torch.zeros(x.size(0), 64, dtype=torch.float64))
    want = m.out(h)
    assert float((got - want).detach().abs().max()) <= 1e-12 * float(want.detach().abs().max())
    # an explicit scale replaces 1/(1-p) in both places: the same masks at scale s equal masks at 1/(1-p), rescaled layer
    # by layer -- checked on the first layer's output, where nothing else intervenes
    s = 1.0 / (1.0 - p) * (1 + 1e-3)
    conv = m.gat_layers[0]
    a = conv(x, ei, dropout_mask=att[0], dropout_scale=s) - conv.bias
    b = conv(x, ei, dropout_mask=att[0]) - conv.bias
    assert torch.allclose(a, b * (1 + 1e-3), rtol=1e-12, atol=1e-15)
