"""GPU parity of the gradient w.r.t. the layer input in the input-space formulation (gemm_algo=GEMM_INPUT, hidden layer
K = 64): the backward edge pass writes the (alpha_used, dz) slot records, the projected path's source-major pass turns them
into dxw, and dx = dxw W.  Checked against the fp64 oracle, against the projected-feature path, under dropout, at extreme
scales, for determinism, and at model level (GAT / TemporalGNN training, DeviceTrainStep's CUDA graph)."""
import copy

import pytest
import torch
import torch.nn as nn

from gnn_fraud_detection_b200 import GAT, GATConv, TemporalGNN, _abi, build_csr, functional as Fn, synth
from oracle import pyg_gatconv as O
from test_gat_gpu import REL32, TOL32, _assert_close, _fwd_bwd_case, _layer
from util import maxabs, relerr, seeded_params

pytestmark = pytest.mark.gpu
GRADS = ("dW", "datt_src", "datt_dst", "dbias", "dx")


def _graph(kind):
    """Edge lists that reach every branch of the edge pass and of the source-major pass."""
    if kind == "random":
        return 3000, synth.random_graph(3000, 30000, seed=2)
    if kind == "edgeless":                      # the self-loops the layer adds are the only edges
        return 500, torch.zeros(2, 0, dtype=torch.long)
    if kind == "dup_selfloops":                 # duplicate edges and explicit self-loops in edge_index
        ei = synth.random_graph(800, 5000, seed=3)
        loops = torch.arange(0, 800, 3).repeat(2, 1)
        return 800, torch.cat([ei, ei[:, :1500], loops, loops[:, :50]], 1)
    if kind == "long_and_packs":                # rows of 33..300 edges (second sweep) among packs of 1..4-edge rows
        g = torch.Generator().manual_seed(4)
        short = torch.stack([torch.randint(0, 4000, (6000,), generator=g), torch.randint(0, 4000, (6000,), generator=g)])
        rows = [torch.stack([torch.randint(0, 4000, (d,), generator=g), torch.full((d,), r)])
                for r, d in ((5, 33), (17, 64), (90, 100), (1000, 300), (3999, 40))]
        return 4000, torch.cat([short] + rows, 1)
    if kind == "dst_hub":                       # a destination row above HUB_THRESHOLD (chunked, merged)
        ei = synth.random_graph(3000, 20000, seed=5)
        hub = torch.stack([torch.randint(0, 3000, (5 * _abi.HUB_THRESHOLD,)), torch.full((5 * _abi.HUB_THRESHOLD,), 11)])
        return 3000, torch.cat([ei, hub], 1)
    if kind == "src_hub":                       # a source of out-degree 100 000: long CSC rows in the source-major pass
        ei = synth.random_graph(2000, 10000, seed=6)
        hub = torch.stack([torch.full((100_000,), 13), torch.randint(0, 2000, (100_000,))])
        return 2000, torch.cat([ei, hub], 1)
    raise ValueError(kind)


KINDS = ["random", "edgeless", "dup_selfloops", "long_and_packs", "dst_hub", "src_hub"]


@pytest.mark.parametrize("kind", KINDS)
def test_hidden_layer_input_space_against_fp64_oracle(kind):
    N, ei = _graph(kind)
    got, ref = _fwd_bwd_case(N, 0, 64, ei=ei, algo=_abi.GEMM_INPUT, need_dx=True)
    assert got["dx"] is not None and got["dx"].shape == (N, 64)
    _assert_close(got, ref)
    if kind == "dst_hub":
        assert build_csr(ei.cuda(), N).c.hub_dst.n_hub >= 1
    if kind == "src_hub":
        assert build_csr(ei.cuda(), N).c.hub_src.n_hub >= 1


@pytest.mark.parametrize("kind", ["random", "long_and_packs", "dst_hub", "src_hub"])
def test_hidden_layer_input_space_agrees_with_projected_path(kind):
    N, ei = _graph(kind)
    ours, _ = _fwd_bwd_case(N, 0, 64, ei=ei, algo=_abi.GEMM_INPUT)
    for algo in (_abi.GEMM_SIMT, _abi.GEMM_AUTO):
        other, _ = _fwd_bwd_case(N, 0, 64, ei=ei, algo=algo)
        for k in GRADS:
            assert relerr(ours[k], other[k]) <= REL32, (algo, k, relerr(ours[k], other[k]))


def test_in_kernel_dropout_equals_its_exported_mask_with_dx():
    """The counter-based dropout RNG and the mask it exports give the same layer: forward and backward (dx included) see one
    mask.  Only the survivor scale differs (65536/(65536 - thr) against 1/(1-p): 3.8e-6 relative at p = 0.2)."""
    N, E, K, H, C, p = 3000, 30000, 64, 8, 64, 0.2
    W, a_s, a_d, b = seeded_params(K, H, C, seed=5)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(0)).cuda()
    ei = torch.cat([synth.random_graph(N, E, seed=1), torch.stack([torch.randint(0, N, (900,)), torch.full((900,), 7)])], 1).cuda()
    conv = _layer(K, H, C, False, W, a_s, a_d, b, dropout=p, gemm_algo=_abi.GEMM_INPUT).train()
    d_out = torch.randn(N, C, generator=torch.Generator().manual_seed(3)).cuda() / N
    torch.manual_seed(123)
    xg = x.clone().requires_grad_(True)
    out = conv(xg, ei)
    out.backward(d_out)
    grads = [p_.grad.clone() for p_ in conv.parameters()] + [xg.grad.clone()]
    keep, _ = Fn.dropout_mask(conv.last_dropout_seed, p, conv._graph(ei, N).n_edges, H, x.device)
    conv.zero_grad()
    xg2 = x.clone().requires_grad_(True)
    out2 = conv(xg2, ei, dropout_mask=keep)
    out2.backward(d_out)
    assert relerr(out, out2) < 1e-5
    for ga, pb in zip(grads, list(conv.parameters()) + [xg2]):
        assert relerr(ga, pb.grad) < 2e-5


def test_injected_dropout_mask_against_fp64_autograd_with_dx():
    N, E, K, H, C, p = 1500, 12000, 64, 8, 64, 0.2
    W, a_s, a_d, b = seeded_params(K, H, C, seed=5)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(0))
    ei = torch.cat([synth.random_graph(N, E, seed=1), torch.stack([torch.randint(0, N, (700,)), torch.full((700,), 9)])], 1)
    Ep = O.rewrite_self_loops(ei, N).size(1)
    keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(2)) >= p
    conv = _layer(K, H, C, False, W, a_s, a_d, b, dropout=p, gemm_algo=_abi.GEMM_INPUT)
    xg = x.cuda().requires_grad_(True)
    out = conv(xg, ei.cuda(), dropout_mask=keep)
    leaves = [t.double().clone().requires_grad_(True) for t in (x, W, a_s, a_d, b)]
    ref, _ = O.gatconv_forward(leaves[0], ei, leaves[1], leaves[2], leaves[3], leaves[4], H, C, dropout_mask=keep, p=p)
    d_out = torch.randn(N, C, generator=torch.Generator().manual_seed(3)) / N
    out.backward(d_out.cuda())
    ref.backward(d_out.double())
    assert maxabs(out, ref) <= TOL32
    for name, g_, r_ in (("dx", xg.grad, leaves[0].grad), ("dW", conv.lin_src.weight.grad, leaves[1].grad),
                         ("datt_src", conv.att_src.grad, leaves[2].grad), ("datt_dst", conv.att_dst.grad, leaves[3].grad),
                         ("dbias", conv.bias.grad, leaves[4].grad)):
        assert maxabs(g_, r_) <= TOL32, name
        assert relerr(g_, r_) <= REL32, (name, relerr(g_, r_))


@pytest.mark.parametrize("x_scale,d_scale", [(1e-6, 1e6), (1e6, 1e-6), (1e-6, 1e-6), (1e6, 1e6)])
def test_dx_range(x_scale, d_scale):
    """x and d_out far from unit scale (W scaled by 1/x_scale keeps the logits O(1)): every gradient keeps REL32."""
    N, E, K, H, C = 2000, 16000, 64, 8, 64
    W, a_s, a_d, b = seeded_params(K, H, C, seed=2)
    W = W / x_scale
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(0)) * x_scale
    ei = synth.random_graph(N, E, seed=4)
    conv = _layer(K, H, C, False, W, a_s, a_d, b, gemm_algo=_abi.GEMM_INPUT)
    xg = x.cuda().requires_grad_(True)
    out = conv(xg, ei.cuda())
    ref, _ = O.gatconv_forward(x.double(), ei, W.double(), a_s.double(), a_d.double(), b.double(), H, C)
    d_out = torch.randn(N, C, generator=torch.Generator().manual_seed(3)) * (d_scale / N)
    out.backward(d_out.cuda())
    cf = O.gatconv_backward_closed_form(x.double(), ei, W.double(), a_s.double(), a_d.double(), H, C, d_out.double())
    assert relerr(out, ref) <= REL32
    for name, g_ in (("dx", xg.grad), ("dW", conv.lin_src.weight.grad), ("datt_src", conv.att_src.grad),
                     ("datt_dst", conv.att_dst.grad), ("dbias", conv.bias.grad)):
        assert relerr(g_, cf[name]) <= REL32, (name, relerr(g_, cf[name]))


def test_dx_is_deterministic():
    N, ei = _graph("dst_hub")
    runs = [_fwd_bwd_case(N, 0, 64, ei=ei, algo=_abi.GEMM_INPUT)[0] for _ in range(2)]
    for k in ("out",) + GRADS:
        assert torch.equal(runs[0][k], runs[1][k]), k


@pytest.mark.parametrize("kind", ["long_and_packs", "dst_hub"])
@pytest.mark.parametrize("p", [0.0, 0.3])
def test_record_mode_leaves_dz_and_da_dst_unchanged(kind, p):
    """The edge pass with the alpha_used records writes the same dz and da_dst, bit for bit, as without them, and the
    records hold alpha after dropout at the source-major slot of each edge."""
    N, ei = _graph(kind)
    K = 64
    W, a_s, a_d, _ = (t.cuda() for t in seeded_params(K, 8, 64, seed=1))
    asf, adf = a_s.view(-1).contiguous(), a_d.view(-1).contiguous()
    g = build_csr(ei.cuda(), N)
    xg = Fn.in_pad_x(torch.randn(N, K, generator=torch.Generator().manual_seed(0)).cuda())
    prep = Fn._aligned_u8(Fn.in_sizes(N, K)[0], xg.device)
    xmax = torch.zeros(16, device="cuda")
    a_src, a_dst = Fn.in_logits(xg, W, asf, adf, prep, xmax)
    Fn.in_prepare(W, K, xmax, prep)
    zimg, att = Fn.in_fwd(g, xg, a_src, a_dst, 0.2, prep, p_drop=p, seed=77)
    d_out = torch.randn(N, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) / N
    dz, da_dst = Fn.in_bwd_edges(g, xg, att, d_out, prep, 0.2, p_drop=p, seed=77)
    alpha_used, dz_r, da_dst_r = Fn.in_bwd_edges(g, xg, att, d_out, prep, 0.2, p_drop=p, seed=77, records=True)
    assert torch.equal(dz, dz_r) and torch.equal(da_dst, da_dst_r)
    assert dz_r.data_ptr() == alpha_used.data_ptr() + 32
    want = att.alpha.abs()
    if p > 0:
        keep, scale = Fn.dropout_mask(77, p, g.n_edges, 8, xg.device)
        want = want * keep[g.perm.long()].float() * scale
    got = alpha_used[g.csr2csc.long()]
    assert relerr(got, want) <= 1e-5 and torch.equal(got == 0, want == 0)


def test_input_space_dx_rejects_what_it_cannot_do():
    ei = synth.random_graph(50, 200, seed=1).cuda()
    for K in (16, 166):                         # a gradient w.r.t. x exists at K = 64 only
        with pytest.raises(_abi.GnnfdError):
            GATConv(K, 64, heads=8, concat=False, gemm_algo=_abi.GEMM_INPUT).cuda()(
                torch.randn(50, K, device="cuda", requires_grad=True), ei)
    with pytest.raises(_abi.GnnfdError):
        GATConv(64, 64, heads=8, concat=True, gemm_algo=_abi.GEMM_INPUT).cuda()(
            torch.randn(50, 64, device="cuda", requires_grad=True), ei)
    with pytest.raises(_abi.GnnfdError):
        GATConv(64, 32, heads=8, concat=False, gemm_algo=_abi.GEMM_INPUT).cuda()(
            torch.randn(50, 64, device="cuda", requires_grad=True), ei)


# ---- models -----------------------------------------------------------------------------------------------------------
def _model_pair(cls, dropout=0.0):
    torch.manual_seed(0)
    ref = (O.OracleGAT if cls is GAT else O.OracleTemporalGNN)(166, 64, 1, num_layers=3, dropout=dropout).double()
    ours = cls(166, 64, 1, num_layers=3, dropout=dropout, gemm_algo=_abi.GEMM_INPUT)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    return ref.train(), ours.cuda().train()


def _model_data():
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    y = (torch.rand(x.size(0), generator=torch.Generator().manual_seed(1)) < 0.1).long()
    y[::7] = -1
    return x, ei, y


def _train_grads(m, x, ei, y):
    """One forward / masked BCE(pos_weight=50) / backward (src/train.py:108-142); {name: grad}."""
    mask = y != -1
    # the oracle's default zero state is fp32: hand it an fp64 one (ours takes None, the reference's zero state)
    kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if isinstance(m, O.OracleTemporalGNN) else {}
    r = m(x, ei, **kw)
    lg = r[0] if isinstance(r, tuple) else r
    crit = nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, dtype=lg.dtype, device=lg.device))
    crit(lg[mask].squeeze(1), y[mask].to(lg.dtype)).backward()
    return lg.detach(), {n: p.grad.detach().clone() for n, p in m.named_parameters() if "lin_dst" not in n}


@pytest.mark.parametrize("cls", [GAT, TemporalGNN])
def test_models_train_in_input_space_against_fp64_oracle_and_projected_path(cls):
    x, ei, y = _model_data()
    ref, ours = _model_pair(cls)
    auto = copy.deepcopy(ours)
    for conv in auto.gat_layers:
        conv.gemm_algo = _abi.GEMM_AUTO
    lr, gr = _train_grads(ref, x.double(), ei, y)
    lo, go = _train_grads(ours, x.cuda(), ei.cuda(), y.cuda())
    la, ga = _train_grads(auto, x.cuda(), ei.cuda(), y.cuda())
    assert relerr(lo, lr) <= 1e-5 and relerr(la, lr) <= 1e-5
    assert set(go) == set(gr) == set(ga)
    for n in gr:
        # conv biases feed a train-mode BatchNorm: their true gradient is zero, only rounding noise remains
        if float(gr[n].norm()) > 1e-6:
            assert relerr(go[n], gr[n]) <= 2e-4, (cls.__name__, n, relerr(go[n], gr[n]))
            assert relerr(go[n], ga[n]) <= 2e-4, (cls.__name__, n, relerr(go[n], ga[n]))
        else:
            assert maxabs(go[n], gr[n]) <= 1e-5, (cls.__name__, n)


@pytest.mark.parametrize("cls", [GAT, TemporalGNN])
def test_models_with_dropout_reproduce_under_one_seed(cls):
    x, ei, y = _model_data()
    _, m = _model_pair(cls, dropout=0.2)
    assert m.fused_tail
    runs = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        torch.manual_seed(42)
        runs.append(_train_grads(m, x.cuda(), ei.cuda(), y.cuda()))
    assert torch.equal(runs[0][0], runs[1][0])
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n


def test_device_train_step_graph_replay_in_input_space():
    """DeviceTrainStep (forward + loss + backward + Adam captured in one CUDA graph) of a 3-layer GEMM_INPUT GAT against the
    same model stepped eagerly."""
    from gnn_fraud_detection_b200.train_step import DeviceTrainStep
    x, ei, _ = synth.elliptic_synth(num_nodes=8000, num_edges=9200, num_feats=166, seed=0)
    y = (torch.rand(x.size(0), generator=torch.Generator().manual_seed(1)) < 0.1).long()
    y[::5] = -1
    xg, eg, yg = x.cuda(), ei.cuda(), y.cuda()
    torch.manual_seed(0)
    a = GAT(166, 64, 1, num_layers=3, dropout=0.0, gemm_algo=_abi.GEMM_INPUT).cuda().train()
    b = copy.deepcopy(a)
    trainer = DeviceTrainStep(a, xg, eg, yg, pos_weight=50.0, use_cuda_graph=True)
    assert trainer.graph is not None
    opt = torch.optim.Adam(b.parameters(), lr=1e-3, weight_decay=5e-4)
    crit = nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, device="cuda"))
    mask = yg != -1

    def eager_step():
        opt.zero_grad()
        loss = crit(b(xg, eg)[mask].squeeze(1), yg[mask].float())
        loss.backward()
        opt.step()
        return float(loss.detach())

    for _ in range(3):                          # the trainer's construction ran three warm-up steps
        eager_step()
    for _ in range(4):
        loss_d, _ = trainer.step()
        le = eager_step()
        assert abs(float(loss_d) - le) <= 2e-4 * abs(le)
    for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        if n.startswith("gat_layers.") and n.endswith(".bias"):
            continue        # feeds a train-mode BatchNorm: true gradient 0, Adam turns the rounding noise into +-lr steps
        assert relerr(pa, pb) <= 1e-3, (n, relerr(pa, pb))
    trainer.close()
