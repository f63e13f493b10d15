"""The 8-head layer at hidden widths 32 and 128 (H*C = 256 and 1024), from the tensor-core projection to the backward:
layer parity against the fp64 oracle, the tcgen05 projection against the SIMT kernel, the source-major structure cases
built like the C=64 ones, the models at hidden_channels 32 / 128, and the refusals that still hold."""
import copy
import ctypes
from types import SimpleNamespace

import pytest
import torch
import torch.nn as nn

from gnn_fraud_detection_b200 import GAT, GATConv, NeighborLoader, TemporalGNN, _abi, fused, functional as Fn, synth
from oracle import pyg_gatconv as O
from util import maxabs, relerr, seeded_params
import test_bwd_record_gpu as REC
import test_bwd_srcmajor_gpu as BS
import test_fwd_srcmajor_gpu as FS
from test_gat_gpu import _assert_close, _fwd_bwd_case, TOL32

pytestmark = pytest.mark.gpu
WIDTHS = [32, 128]


# ---- layer parity -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("algo", [_abi.GEMM_SIMT, _abi.GEMM_TC])
@pytest.mark.parametrize("N,E,K", [(1, 0, 5), (100, 300, 7), (1000, 5000, 166), (777, 9000, 165), (3000, 20000, 32),
                                   (2000, 15000, 128)])
def test_layer_fwd_bwd_mean(C, algo, N, E, K):
    _assert_close(*_fwd_bwd_case(N, E, K, C=C, algo=algo))


# With concat the output is a convex combination of projected rows, so it carries the projection's relative error without
# the head mean's averaging.  On the tensor cores (3xTF32, ~2.4e-6 relative on this output at every width, C=64 included)
# the K=166 case reaches |out| ~ 3.4 at C=32 and 1.04e-5 max-abs, past the absolute bar; it runs on the SIMT path here.
@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("algo,N,E,K", [(_abi.GEMM_SIMT, 100, 300, 7), (_abi.GEMM_SIMT, 900, 6000, 166),
                                        (_abi.GEMM_SIMT, 900, 6000, 32), (_abi.GEMM_SIMT, 900, 6000, 128),
                                        (_abi.GEMM_TC, 100, 300, 7), (_abi.GEMM_TC, 900, 6000, 32),
                                        (_abi.GEMM_TC, 900, 6000, 128)])
def test_layer_fwd_bwd_concat(C, algo, N, E, K):
    _assert_close(*_fwd_bwd_case(N, E, K, C=C, concat=True, algo=algo))


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("concat", [False, True])
def test_rows_longer_than_one_chunk_and_hub_rows(C, concat):
    # in-degrees 33..511 (second sweep) and > 512 (hub splitting with merge); an out-degree hub on the CSC side
    ei = synth.fraud_ring_skew(num_nodes=3000, background_edges=20000, num_hubs=4, hub_degree=2500, num_rings=20,
                               ring_len=16, seed=7)
    extra = torch.stack([torch.randint(0, 3000, (700,)), torch.full((700,), 11)])
    mid = torch.stack([torch.randint(0, 3000, (100,)), torch.full((100,), 12)])
    hub_src = torch.stack([torch.full((1500,), 13), torch.randint(0, 3000, (1500,))])
    ei = torch.cat([ei, extra, mid, hub_src], 1)
    _assert_close(*_fwd_bwd_case(3000, 0, C, C=C, concat=concat, ei=ei, algo=_abi.GEMM_TC))


# ---- projection ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("N,K", [(1, 7), (1000, 166), (777, 165), (4100, 32), (3000, 128), (130, 200)])
def test_projection_tensor_core(C, N, K):
    """tcgen05 xw and the epilogue's per-head logits against the SIMT kernel and the fp64 product"""
    H = 8
    W, a_s, a_d, _ = seeded_params(K, H, C, seed=3)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(N + K))
    xg, Wg, asg, adg = x.cuda(), W.cuda(), a_s.cuda().view(-1), a_d.cuda().view(-1)
    xw_t, as_t, ad_t = Fn.project_fwd(xg, Wg, asg, adg, H, C, torch.float32, _abi.GEMM_TC)
    xw_s, as_s, ad_s = Fn.project_fwd(xg, Wg, asg, adg, H, C, torch.float32, _abi.GEMM_SIMT)
    ref = x.double() @ W.double().t()
    ra = (ref.view(N, H, C) * a_s.double()).sum(-1)
    rd = (ref.view(N, H, C) * a_d.double()).sum(-1)
    assert maxabs(xw_t, ref) <= TOL32 and maxabs(xw_s, ref) <= TOL32 and relerr(xw_t, ref) <= 2e-6
    assert maxabs(as_t, ra) <= TOL32 and maxabs(ad_t, rd) <= TOL32
    assert maxabs(as_t, as_s) <= TOL32 and maxabs(ad_t, ad_s) <= TOL32
    # GEMM_AUTO takes the tensor cores at these widths
    xw_a, _, _ = Fn.project_fwd(xg, Wg, asg, adg, H, C, torch.float32, _abi.GEMM_AUTO)
    assert torch.equal(xw_a, xw_t)


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("N,K", [(1000, 166), (3000, 32), (3000, 128), (9000, 165)])
def test_projection_backward_hidden_shapes(C, N, K):
    """dx (reduction over D = 256 / 1024) and dW at the hidden-layer shapes K = C"""
    H = 8
    D = H * C
    W, _, _, _ = seeded_params(K, H, C, seed=4)
    g = torch.Generator().manual_seed(N)
    x, dxw = torch.randn(N, K, generator=g), torch.randn(N, D, generator=g)
    xw = x @ W.t()
    das, dad, dout = torch.randn(N, H, generator=g), torch.randn(N, H, generator=g), torch.randn(N, C, generator=g)
    args = [t.cuda() for t in (x, W, dxw, xw, das, dad, dout)]
    for algo in (_abi.GEMM_TC, _abi.GEMM_SIMT):
        dW, datt_s, datt_d, dbias, dx = Fn.project_bwd(*args, H, C, C, True, algo)
        assert relerr(dx, dxw.double() @ W.double()) <= 1e-5
        assert relerr(dW, dxw.double().t() @ x.double()) <= 1e-5
        xw64 = (x.double() @ W.double().t()).view(N, H, C)
        assert relerr(datt_s, (das.double()[:, :, None] * xw64).sum(0).view(-1)) <= 2e-6
        assert relerr(datt_d, (dad.double()[:, :, None] * xw64).sum(0).view(-1)) <= 2e-6
        assert relerr(dbias, dout.double().sum(0)) <= 2e-6


# ---- source-major structure cases -----------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("drop", [None, "injected", "seed"])
def test_fwd_srcmajor_degrees_hubs_and_modes(C, drop):
    H = 8
    ei, N = FS._degree_graph(seed=5)
    t = FS._inputs(ei, N, 16, H, C, seed=41, add_self_loops=False, hub_threshold=FS.THR, hub_chunk=FS.THR)
    g = t["g"]
    assert g.c.hub_src.n_hub >= 2 and g.c.hub_dst.n_hub >= 1 and g.c.hub_dst.n_chunk >= 6
    kw, keep, scale = FS._dropout(drop, g.n_edges, H)
    FS._check(t, H, C, keep, scale, **kw)


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("drop", [None, "injected", "seed"])
def test_bwd_record_long_rows_among_packs_and_hub_source(C, drop):
    H, p, seed = 8, 0.3, 17
    ei, N, long_rows = REC._record_graph(seed=9)
    t = BS._inputs(ei, N, 16, H, C, seed=71, add_self_loops=False, hub_threshold=REC.THR, hub_chunk=128)
    g = t["g"]
    rowptr, colptr = g.rowptr.cpu(), g.colptr.cpu()
    for deg, i in long_rows.items():
        assert int(rowptr[i + 1] - rowptr[i]) == deg
    assert int(colptr[REC.HUB_SRC + 1] - colptr[REC.HUB_SRC]) == 2 * REC.THR + 5
    assert g.c.hub_src.n_hub >= 1 and g.c.hub_dst.n_hub >= 1
    Ep = g.n_edges
    kw, keep, scale = {}, None, 1.0
    if drop == "injected":
        keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(4)) >= p
        one = torch.ones((), dtype=torch.float32)
        scale = float(one / (one - torch.tensor(p, dtype=torch.float32)))
        kw = dict(keep_mask=keep, p_drop=p)
    elif drop == "seed":
        keep, scale = Fn.dropout_mask(seed, p, Ep, H, torch.device("cuda"))
        keep, kw = keep.bool().cpu(), dict(p_drop=p, seed=seed)
    au, dz, dad = BS._check_same_as_gather(t, H, C, **kw)          # alpha_used bit-equal to the gather kernel
    r_au, r_dz, r_dad = BS._ref_dst_pass(t, H, C, keep, scale)
    BS._close(BS._csr_order(g, au), r_au)
    BS._close(BS._csr_order(g, dz), r_dz)
    BS._close(dad, r_dad)


@pytest.mark.parametrize("C", WIDTHS)
def test_bwd_srcmajor_degrees_against_closed_form(C):
    """out-degrees 31..3*THR and in-degrees up to the hub row of the forward's degree graph through the ring-fed d_alpha
    pass, against the gather kernel and the fp64 closed form"""
    H = 8
    ei, N = FS._degree_graph(seed=8)
    t = BS._inputs(ei, N, 16, H, C, seed=43, add_self_loops=False, hub_threshold=FS.THR, hub_chunk=FS.THR)
    assert t["g"].c.hub_src.n_hub >= 2
    au, dz, dad = BS._check_same_as_gather(t, H, C)
    r_au, r_dz, r_dad = BS._ref_dst_pass(t, H, C)
    BS._close(BS._csr_order(t["g"], au), r_au)
    BS._close(BS._csr_order(t["g"], dz), r_dz)
    BS._close(dad, r_dad)


@pytest.mark.parametrize("C", WIDTHS)
def test_workspace_one_byte_short_is_refused(C):
    N, H = 3000, 8
    ei = synth.random_graph(N, 20000, seed=3)
    t = BS._inputs(ei, N, 16, H, C, seed=61, hub_threshold=64, hub_chunk=64)
    g = t["g"]
    L = _abi.lib()
    bias = torch.zeros(C, device="cuda")
    out = torch.empty(N, C, dtype=torch.float32, device="cuda")
    rowmax = torch.empty(N, H, dtype=torch.float32, device="cuda")
    rowsum = torch.empty(N, H, dtype=torch.float32, device="cuda")
    nb = ctypes.c_size_t()
    _abi.check(L.gnnfd_gat_fwd_workspace_bytes(g.ref(), H, C, ctypes.byref(nb)))
    need = nb.value - 256
    assert need >= g.n_edges * (H + C) * 4
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")

    def fwd(ws_bytes):
        return L.gnnfd_gat_fwd_fused(g.ref(), t["xw"].data_ptr(), Fn._DT[t["xw"].dtype], t["a_src"].data_ptr(),
                                     t["a_dst"].data_ptr(), bias.data_ptr(), H, C, 0.2, 0, 0, None, 0.0, 0, None, None,
                                     None, out.data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(), ws.data_ptr(), ws_bytes,
                                     Fn._stream())

    assert fwd(need - 1) == -3                    # GNNFD_ERR_WORKSPACE
    assert fwd(need) == 0
    torch.cuda.synchronize()
    _, rowmax2, rowsum2 = Fn.gat_fwd(g, t["xw"], t["a_src"], t["a_dst"], None, H, C, 0.2, False)
    _abi.check(L.gnnfd_gat_bwd_workspace_bytes(g.ref(), H, C, ctypes.byref(nb)))
    need = nb.value - 256
    assert need >= g.n_edges * 2 * H * 4
    eg = torch.empty(g.n_edges, 2 * H, dtype=torch.float32, device="cuda")
    dad = torch.empty(N, H, dtype=torch.float32, device="cuda")
    d_out = t["d_out"].cuda()
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")

    def bwd(ws_bytes):
        return L.gnnfd_gat_bwd_dst(g.ref(), t["xw"].data_ptr(), Fn._DT[t["xw"].dtype], t["a_src"].data_ptr(),
                                   t["a_dst"].data_ptr(), rowmax2.data_ptr(), rowsum2.data_ptr(), d_out.data_ptr(), H, C,
                                   0.2, 0, 0, 0.0, 0, eg[:, :H].data_ptr(), eg[:, H:].data_ptr(), dad.data_ptr(),
                                   ws.data_ptr(), ws_bytes, Fn._stream())

    assert bwd(need - 1) == -3
    assert bwd(need) == 0
    torch.cuda.synchronize()


# ---- models -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDTHS)
def test_gat_training_step_matches_oracle_full_batch(C):
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    torch.manual_seed(0)
    ref = O.OracleGAT(166, C, 1, num_layers=2, dropout=0.0).double()
    ours = GAT(166, C, 1, num_layers=2, dropout=0.0)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    ours = ours.cuda()
    y = (torch.rand(x.size(0), 1, generator=torch.Generator().manual_seed(1)) < 0.1).float()
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0))
    lr = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0).double())(ref(x.double(), ei), y.double()); lr.backward()
    lo = crit.cuda()(ours(x.cuda(), ei.cuda()), y.cuda()); lo.backward()
    assert abs(float(lr) - float(lo)) <= 1e-5
    for (n, p_ref), (_, p_our) in zip(ref.named_parameters(), ours.named_parameters()):
        assert maxabs(p_our.grad, p_ref.grad) <= 1e-5, n
        if float(p_ref.grad.norm()) > 1e-6:
            assert relerr(p_our.grad, p_ref.grad) <= 3e-5, n


@pytest.mark.parametrize("C", WIDTHS)
def test_fused_eval_matches_unfused(C):
    x, ei, _ = synth.elliptic_synth(num_nodes=6000, num_edges=7000, num_feats=166, seed=2)
    x, ei = x.cuda(), ei.cuda()
    torch.manual_seed(4)
    gat = GAT(166, C, 1, num_layers=3).cuda().eval()
    for bn in gat.batch_norms:
        with torch.no_grad():
            bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2.0)
    with torch.no_grad():
        fused_out = gat(x, ei)
    with torch.enable_grad():
        unfused = gat(x, ei).detach()
    assert maxabs(fused_out, unfused) <= 1e-5
    conv = GATConv(C, C, heads=8, concat=False).cuda().eval()
    bn = torch.nn.BatchNorm1d(C).cuda().eval()
    with torch.no_grad():
        bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2.0); bn.weight.normal_(); bn.bias.normal_()
        h = torch.randn(x.size(0), C, device="cuda")
        ref = h + torch.relu(bn(conv(h, ei)))
        assert maxabs(conv.forward_fused_eval(h, ei, bn, relu=True, residual=h), ref) <= 1e-5
        assert maxabs(conv.forward_fused_eval(h, ei, None, relu=False), conv(h, ei)) <= 1e-6


@pytest.mark.parametrize("C", WIDTHS)
def test_temporal_gnn_forward_matches_oracle(C):
    """the GRU head at these widths is torch's GRUCell (the fused head is built for 64 only)"""
    x, ei, _ = synth.elliptic_synth(num_nodes=5000, num_edges=6000, num_feats=166, seed=3)
    torch.manual_seed(5)
    ours = TemporalGNN(166, C, 1, num_layers=2).eval()
    ref = O.OracleTemporalGNN(166, C, 1, num_layers=2).double().eval()
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    ours = ours.cuda()
    assert not fused.gru_head_supported(ours.gru, ours.out)
    with torch.no_grad():
        lg, hid = ours(x.cuda(), ei.cuda())
        rl, rh = ref(x.double(), ei, hidden_state=torch.zeros(x.size(0), C, dtype=torch.float64))
    assert hid.shape == (x.size(0), C)
    assert maxabs(lg, rl) <= 1e-4 and relerr(lg, rl) <= 1e-5
    assert maxabs(hid, rh) <= 1e-4 and relerr(hid, rh) <= 1e-5


@pytest.mark.parametrize("C", WIDTHS)
def test_device_train_step_replay_equals_eager(C):
    from gnn_fraud_detection_b200.train_step import DeviceTrainStep
    x, ei, _ = synth.elliptic_synth(num_nodes=8000, num_edges=9200, num_feats=166, seed=0)
    y = (torch.rand(x.size(0), generator=torch.Generator().manual_seed(1)) < 0.1).long()
    y[::5] = -1
    xg, eg, yg = x.cuda(), ei.cuda(), y.cuda()
    torch.manual_seed(0)
    a = GAT(166, C, 1, num_layers=2, dropout=0.0).cuda().train()
    b = copy.deepcopy(a)
    trainer = DeviceTrainStep(a, xg, eg, yg, pos_weight=50.0, use_cuda_graph=True)
    opt = torch.optim.Adam(b.parameters(), lr=1e-3, weight_decay=5e-4)
    crit = nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, device="cuda"))
    mask = yg != -1

    def eager_step():
        opt.zero_grad()
        loss = crit(b(xg, eg)[mask].squeeze(1), yg[mask].float())
        loss.backward()
        opt.step()
        return float(loss)

    for _ in range(3):
        eager_step()
    loss_d, _ = trainer.step()
    le = eager_step()
    assert abs(float(loss_d) - le) <= 2e-4 * abs(le)
    for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        if n.startswith("gat_layers.") and n.endswith(".bias"):
            continue        # feeds a train-mode BatchNorm: true gradient 0, Adam turns rounding noise into +-lr steps
        assert relerr(pa, pb) <= 1e-3, (n, relerr(pa, pb))
    trainer.close()


@pytest.mark.parametrize("C", WIDTHS)
def test_neighbor_loader_batch_through_three_layers(C):
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    loader = NeighborLoader(SimpleNamespace(x=x.cuda(), edge_index=ei.cuda()), [10, 10, 10], batch_size=256, shuffle=True)
    torch.manual_seed(0)
    batch = next(iter(loader))
    bs = batch.batch_size
    ref = O.OracleGAT(166, C, 1, num_layers=3, dropout=0.0).double()
    ours = GAT(166, C, 1, num_layers=3, dropout=0.0)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    ours = ours.cuda()
    y = (torch.rand(batch.n_id.numel(), 1, generator=torch.Generator().manual_seed(1)) < 0.1).float()
    logits_ref = ref(batch.x.cpu().double(), batch.edge_index.cpu())
    lr = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0).double())(logits_ref[:bs], y[:bs].double())
    lr.backward()
    logits = ours(batch.x, batch.edge_index)
    lo = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0)).cuda()(logits[:bs], y[:bs].cuda())
    lo.backward()
    assert abs(lr.item() - lo.item()) <= 1e-5
    assert maxabs(logits, logits_ref) <= 1e-5 and relerr(logits, logits_ref) <= 1e-5
    for (n, p_ref), (_, p_our) in zip(ref.named_parameters(), ours.named_parameters()):
        assert maxabs(p_our.grad, p_ref.grad) <= 1e-5, n
        if float(p_ref.grad.norm()) > 1e-6:
            assert relerr(p_our.grad, p_ref.grad) <= 3e-5, n


# ---- refusals -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDTHS)
def test_bf16_features_refused_at_new_widths(C):
    x = torch.randn(50, 16, device="cuda")
    W, a_s, a_d, _ = seeded_params(16, 8, C, seed=1)
    for algo in (_abi.GEMM_AUTO, _abi.GEMM_TC, _abi.GEMM_SIMT):
        with pytest.raises(_abi.GnnfdError):
            Fn.project_fwd(x, W.cuda(), a_s.cuda().view(-1), a_d.cuda().view(-1), 8, C, torch.bfloat16, algo)
    conv = GATConv(16, C, heads=8, concat=False, feature_dtype=torch.bfloat16).cuda()
    with pytest.raises(_abi.GnnfdError):
        conv(x, synth.random_graph(50, 200, seed=1).cuda())


def test_width_16_is_not_built():
    conv = GATConv(16, 16, heads=8, concat=False).cuda()
    with pytest.raises(_abi.GnnfdError):
        conv(torch.randn(50, 16, device="cuda"), synth.random_graph(50, 200, seed=1).cuda())


@pytest.mark.parametrize("C", WIDTHS)
def test_input_space_formulation_stays_c64(C):
    conv = GATConv(16, C, heads=8, concat=False, gemm_algo=_abi.GEMM_INPUT).cuda()
    with pytest.raises(_abi.GnnfdError):
        conv(torch.randn(50, 16, device="cuda"), synth.random_graph(50, 200, seed=1).cuda())
