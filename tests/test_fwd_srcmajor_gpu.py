"""The source-major head-mean forward: an attention pass writes alpha_used and the exact row statistics, a source-major
pass writes one C-float message per edge, a CSR pass sums them and applies the row epilogue.  Checked against the gather
forward (the CSC hidden from gat_fwd) and against an fp64 closed form (per-edge softmax, dropout, head mean, epilogue)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from gnn_fraud_detection_b200 import _abi, build_csr, functional as Fn, synth
from util import maxabs, relerr, seeded_params

pytestmark = pytest.mark.gpu
THR = 64                  # hub_threshold of the degree graph: rows above it (either orientation) go to the hub kernels
SLOPE = 0.2


def _degree_graph(seed):
    """Sources with out-degrees 0, 1, 31, 32, 33, THR-1, THR, THR+1, 3*THR; destinations with in-degrees 1, 32, 33 and
    5*THR+7 (a hub row of several chunks); a run of 1200 nodes that are never sources and one of 1200 that are never
    destinations; a sparse background (packs of short rows), duplicated edges and repeated self loops."""
    N = 4000
    rnd = torch.Generator().manual_seed(seed)
    special_src = {0: 10, 1: 11, 31: 12, 32: 13, 33: 14, THR - 1: 15, THR: 16, THR + 1: 17, 3 * THR: 18}
    special_dst = {1: 20, 32: 21, 33: 22, 5 * THR + 7: 23}
    src_ok = torch.ones(N, dtype=torch.bool)
    src_ok[1000:2200] = False
    src_ok[list(special_src.values())] = False
    dst_ok = torch.ones(N, dtype=torch.bool)
    dst_ok[2500:3700] = False
    dst_ok[list(special_dst.values())] = False
    srcs, dsts = torch.nonzero(src_ok).view(-1), torch.nonzero(dst_ok).view(-1)
    srcs = srcs[srcs != 7]
    dsts = dsts[dsts != 7]

    def pick(pool, n):
        return pool[torch.randint(0, pool.numel(), (n,), generator=rnd)]

    bg = torch.stack([pick(srcs, 9000), pick(dsts, 9000)])
    parts = [bg, bg[:, :300], torch.tensor([[7, 7, 7], [7, 7, 7]])]
    for deg, j in special_src.items():
        parts.append(torch.stack([torch.full((deg,), j), pick(dsts, deg)]))
    for deg, i in special_dst.items():
        parts.append(torch.stack([pick(srcs, deg), torch.full((deg,), i)]))
    return torch.cat(parts, 1), N


def _inputs(ei, N, K, H, C, seed, xw_dtype=torch.float32, **csr_kw):
    W, a_s, a_d, bias = seeded_params(K, H, C, seed=seed)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(seed + 1))
    g = build_csr(ei.cuda(), N, **csr_kw)
    asf, adf = a_s.view(-1).contiguous().cuda(), a_d.view(-1).contiguous().cuda()
    xw, a_src, a_dst = Fn.project_fwd(x.cuda(), W.cuda(), asf, adf, H, C, xw_dtype)
    return dict(g=g, xw=xw, a_src=a_src, a_dst=a_dst, a_s=asf, a_d=adf, bias=bias.cuda())


def _fwd(t, H, C, gather=False, **kw):
    """Fn.gat_fwd (head mean); gather=True hides the CSC so that the gather kernels run instead"""
    g = t["g"]
    saved = g.c.colptr
    if gather:
        g.c.colptr = None
    try:
        res = Fn.gat_fwd(g, t["xw"], t["a_src"], t["a_dst"], t["bias"], H, C, SLOPE, False, **kw)
    finally:
        g.c.colptr = saved
    torch.cuda.synchronize()
    return res


def _ref_fwd(t, H, C, keep=None, scale=1.0, act=_abi.ACT_NONE, post_scale=None, post_shift=None, residual=None):
    """fp64 closed form: out, rowmax, rowsum (the kernels' conventions: rowsum includes +1e-16, empty rows (0, 1e-16))"""
    g = t["g"]
    N = g.n_dst
    deg = (g.rowptr[1:] - g.rowptr[:-1]).long()
    dst = torch.repeat_interleave(torch.arange(N, device=deg.device), deg)
    src = g.col.long()
    xw, a_src, a_dst = t["xw"].double(), t["a_src"].double(), t["a_dst"].double()
    e = F.leaky_relu(a_src[src] + a_dst[dst], SLOPE)
    m = torch.full((N, H), -torch.inf, dtype=torch.float64, device=e.device).scatter_reduce(
        0, dst[:, None].expand_as(e), e, "amax", include_self=True)
    p = (e - m[dst]).exp()
    s = torch.zeros(N, H, dtype=torch.float64, device=e.device).index_add_(0, dst, p) + 1e-16
    k = torch.ones_like(p) if keep is None else keep.cuda()[g.perm.long()].double() * scale
    a = p / s[dst] * k
    msg = (a[:, :, None] * xw[src].view(-1, H, C)).sum(1) / H
    out = torch.zeros(N, C, dtype=torch.float64, device=e.device).index_add_(0, dst, msg) + t["bias"].double()
    if post_scale is not None:
        out = out * post_scale.double() + post_shift.double()
    if act == _abi.ACT_RELU:
        out = out.clamp_min(0)
    elif act == _abi.ACT_ELU:
        out = F.elu(out)
    if residual is not None:
        out = out + residual.double()
    empty = (deg == 0)[:, None]
    return out, torch.where(empty, 0.0, m), torch.where(empty, 1e-16, s)


def _close(got, ref, tol=1e-5, rel=1e-5):
    assert maxabs(got, ref) <= tol, f"max-abs {maxabs(got, ref):.3e}"
    if float(ref.double().norm()) > 1e-12:
        assert relerr(got, ref) <= rel, f"relative L2 {relerr(got, ref):.3e}"


def _close_rowsum(got, ref, rel=2e-5):
    """rowsum spans 1e-16 (empty rows) to the hundreds: compared element by element, relative to the reference"""
    r = ((got.double() - ref.double()).abs() / ref.double().abs()).max()
    assert float(r) <= rel, f"max relative {float(r):.3e}"


def _dropout(mode, Ep, H, p=0.3, seed=31):
    """(kwargs of gat_fwd, keep bits [E',H] in edge_index' order, survivor scale)"""
    if mode == "injected":
        keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(2)) >= p
        one = torch.ones((), dtype=torch.float32)
        scale = float(one / (one - torch.tensor(p, dtype=torch.float32)))
        return dict(keep_mask=keep.to(torch.uint8).cuda(), p_drop=p), keep, scale
    if mode == "seed":
        keep, scale = Fn.dropout_mask(seed, p, Ep, H, torch.device("cuda"))
        return dict(p_drop=p, seed=seed), keep.bool().cpu(), scale
    return {}, None, 1.0


def _check(t, H, C, keep=None, scale=1.0, **kw):
    new = _fwd(t, H, C, **kw)
    old = _fwd(t, H, C, gather=True, **kw)
    assert torch.equal(new[1], old[1])                 # rowmax: a max does not depend on the order
    _close_rowsum(new[2], old[2], rel=1e-6)             # the same sums in another order
    _close(new[0], old[0], tol=1e-5, rel=1e-6)
    fw = {k: kw[k] for k in ("act", "post_scale", "post_shift", "residual") if k in kw}
    r_out, r_m, r_s = _ref_fwd(t, H, C, keep, scale, **fw)
    _close(new[0], r_out)
    _close(new[1], r_m)
    _close_rowsum(new[2], r_s)                         # fp32 logits and exp against fp64
    return new


CASES = [
    dict(H=8, C=64, dtype=torch.float32, drop=None),
    dict(H=8, C=64, dtype=torch.float32, drop="injected"),
    dict(H=8, C=64, dtype=torch.float32, drop="seed"),
    dict(H=8, C=64, dtype=torch.bfloat16, drop=None),
    dict(H=8, C=64, dtype=torch.bfloat16, drop="seed"),
    dict(H=4, C=32, dtype=torch.float32, drop=None),
    dict(H=4, C=32, dtype=torch.float32, drop="injected"),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"H{c['H']}C{c['C']}-{str(c['dtype'])[6:]}-{c['drop']}")
def test_degrees_hubs_and_modes(case):
    H, C = case["H"], case["C"]
    ei, N = _degree_graph(seed=5)
    t = _inputs(ei, N, 16, H, C, seed=41, xw_dtype=case["dtype"], add_self_loops=False, hub_threshold=THR, hub_chunk=THR)
    g = t["g"]
    assert g.c.hub_src.n_hub >= 2 and g.c.hub_dst.n_hub >= 1 and g.c.hub_dst.n_chunk >= 6
    deg_out = (g.colptr[1:] - g.colptr[:-1]).cpu()
    deg_in = (g.rowptr[1:] - g.rowptr[:-1]).cpu()
    assert int(deg_out[1000:2200].abs().sum()) == 0 and int(deg_in[2500:3700].abs().sum()) == 0
    kw, keep, scale = _dropout(case["drop"], g.n_edges, H)
    _check(t, H, C, keep, scale, **kw)


def test_fused_epilogue():
    H, C = 8, 64
    ei, N = _degree_graph(seed=6)
    t = _inputs(ei, N, 16, H, C, seed=43, add_self_loops=False, hub_threshold=THR, hub_chunk=THR)
    rnd = torch.Generator().manual_seed(9)
    ps = (torch.rand(C, generator=rnd) + 0.5).cuda()
    sh = (torch.randn(C, generator=rnd) * 0.1).cuda()
    res = torch.randn(N, C, generator=rnd).cuda()
    kw, keep, scale = _dropout("injected", t["g"].n_edges, H)
    for act in (_abi.ACT_RELU, _abi.ACT_ELU):
        _check(t, H, C, keep, scale, act=act, post_scale=ps, post_shift=sh, residual=res, **kw)


@pytest.mark.parametrize("drop", [None, "seed"])
def test_round_trip_through_the_backward(drop):
    """gat_bwd from the new forward's statistics gives the gradients it gives from the gather forward's"""
    H, C = 8, 64
    ei, N = _degree_graph(seed=7)
    t = _inputs(ei, N, 16, H, C, seed=45, add_self_loops=False, hub_threshold=THR, hub_chunk=THR)
    g = t["g"]
    kw, _, _ = _dropout(drop, g.n_edges, H)
    d_out = (torch.randn(N, C, generator=torch.Generator().manual_seed(3)) / N).cuda()
    grads = []
    for gather in (False, True):
        _, rowmax, rowsum = _fwd(t, H, C, gather=gather, **kw)
        grads.append(Fn.gat_bwd(g, t["xw"], t["a_src"], t["a_dst"], rowmax, rowsum, d_out, t["a_s"], t["a_d"], H, C,
                                SLOPE, False, kw.get("keep_mask"), kw.get("p_drop", 0.0), seed=kw.get("seed", 0)))
        torch.cuda.synchronize()
    for a, b in zip(*grads):
        _close(a, b, tol=1e-7, rel=1e-6)


def test_powerlaw_2m_nodes_20m_edges():
    N, E, H, C = 2_000_000, 20_000_000, 8, 64
    ei = synth.powerlaw_graph(N, E, seed=1234, device="cuda")
    t = _inputs(ei, N, 16, H, C, seed=51)
    new = _fwd(t, H, C)
    old = _fwd(t, H, C, gather=True)
    assert torch.equal(new[1], old[1])
    assert relerr(new[2], old[2]) <= 1e-6
    assert relerr(new[0], old[0]) <= 1e-6


def test_workspace_one_byte_short_is_refused():
    N, H, C = 3000, 8, 64
    ei = synth.random_graph(N, 20000, seed=3)
    t = _inputs(ei, N, 16, H, C, seed=61, hub_threshold=64, hub_chunk=64)
    g = t["g"]
    L = _abi.lib()
    nb = ctypes.c_size_t()
    _abi.check(L.gnnfd_gat_fwd_workspace_bytes(g.ref(), H, C, ctypes.byref(nb)))
    need = nb.value - 256                         # the reported size less its 256-byte slack
    assert need >= g.n_edges * (H + C) * 4        # alpha_used [E',H] and the messages [E',C]
    out = torch.empty(N, C, dtype=torch.float32, device="cuda")
    rowmax = torch.empty(N, H, dtype=torch.float32, device="cuda")
    rowsum = torch.empty(N, H, dtype=torch.float32, device="cuda")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")

    def call(ws_bytes):
        return L.gnnfd_gat_fwd_fused(g.ref(), t["xw"].data_ptr(), Fn._DT[t["xw"].dtype], t["a_src"].data_ptr(),
                                     t["a_dst"].data_ptr(), t["bias"].data_ptr(), H, C, SLOPE, 0, 0, None, 0.0, 0, None,
                                     None, None, out.data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(), ws.data_ptr(),
                                     ws_bytes, Fn._stream())

    assert call(need - 1) == -3                   # GNNFD_ERR_WORKSPACE
    assert call(need) == 0
    torch.cuda.synchronize()
    _close(out, _fwd(t, H, C, gather=True)[0], tol=1e-5, rel=1e-6)
