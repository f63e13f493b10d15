"""The streamed head-mean backward: pass 1 walks each source work item's out-edges in CSC order across row boundaries
(dO rows and xw rows through per-warp rings) and writes d_alpha in CSR order; pass 2 reads its edges contiguously and
recomputes alpha.  Checked against the single-pass gather kernel (the CSC hidden from gat_bwd_dst) and the fp64 closed
form, for gat_bwd_dst alone and for the whole Fn.gat_bwd (dxw, da_src, da_dst)."""
import ctypes

import pytest
import torch

from gnn_fraud_detection_b200 import _abi, functional as Fn, synth
from oracle import pyg_gatconv as O
from test_bwd_srcmajor_gpu import _check_same_as_gather, _close, _csr_order, _inputs, _ref_dst_pass, _run
from util import relerr

pytestmark = pytest.mark.gpu
THR = 64                  # hub_threshold of the degree graph: source rows above it go to the hub kernels


def _degree_graph(seed):
    """Sources with out-degrees 1, 31, 32, 33, 64, THR-1, THR, THR+1 and a run of 1200 sources with none;
    destinations with in-degrees 32 and 33 (second sweep) and a sparse background (packs).  No self loops are added,
    so empty source rows stay empty."""
    N = 4000
    rnd = torch.Generator().manual_seed(seed)
    special_src = {1: 10, 31: 11, 32: 12, 33: 13, 64: 14, THR - 1: 15, THR + 1: 16, 2 * 64: 17}
    special_dst = {32: 20, 33: 21}
    empty = torch.arange(1000, 2200)                         # a long run of sources with no out-edges
    fixed = torch.tensor(list(special_src.values()) + list(special_dst.values()))
    allowed = torch.ones(N, dtype=torch.bool)
    allowed[empty] = False
    allowed[fixed] = False
    srcs = torch.nonzero(allowed).view(-1)
    dst_ok = torch.ones(N, dtype=torch.bool)
    dst_ok[list(special_dst.values())] = False
    dsts = torch.nonzero(dst_ok).view(-1)

    def pick(pool, n):
        return pool[torch.randint(0, pool.numel(), (n,), generator=rnd)]

    parts = [torch.stack([pick(srcs, 9000), pick(dsts, 9000)])]
    for deg, j in special_src.items():
        parts.append(torch.stack([torch.full((deg,), j), pick(dsts, deg)]))
    for deg, i in special_dst.items():
        parts.append(torch.stack([pick(srcs, deg), torch.full((deg,), i)]))
    return torch.cat(parts, 1), N


CASES = [
    dict(H=8, C=64, dtype=torch.float32, drop=None),
    dict(H=8, C=64, dtype=torch.float32, drop="injected"),
    dict(H=8, C=64, dtype=torch.float32, drop="seed"),
    dict(H=8, C=64, dtype=torch.bfloat16, drop=None),
    dict(H=4, C=32, dtype=torch.float32, drop=None),
]


def _full_bwd(t, H, C, gather, **kw):
    """Fn.gat_bwd's dst + src passes; gather=True runs the dst pass through the gather kernel"""
    g = t["g"]
    au, dz, dad, _, _ = _run(t, H, C, gather=gather, **kw)
    asf, adf = t["a_s"].view(-1).contiguous().cuda(), t["a_d"].view(-1).contiguous().cuda()
    dxw, da_src = Fn.gat_bwd_src(g, au, dz, t["d_out"].cuda(), asf, adf, dad, H, C, False)
    torch.cuda.synchronize()
    return dxw, da_src, dad


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"H{c['H']}C{c['C']}-{str(c['dtype'])[6:]}-{c['drop']}")
def test_degrees_rings_and_modes(case):
    H, C, p, seed = case["H"], case["C"], 0.3, 31
    ei, N = _degree_graph(seed=5)
    t = _inputs(ei, N, 16, H, C, seed=41, xw_dtype=case["dtype"], add_self_loops=False, hub_threshold=THR, hub_chunk=64)
    g = t["g"]
    assert g.c.hub_src.n_hub >= 2
    colptr = g.colptr.cpu()
    outdeg = colptr[1:] - colptr[:-1]
    assert int(outdeg[1000:2200].abs().sum()) == 0
    Ep = g.n_edges
    kw, keep, scale = {}, None, 1.0
    if case["drop"] == "injected":
        keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(2)) >= p
        one = torch.ones((), dtype=torch.float32)
        scale = float(one / (one - torch.tensor(p, dtype=torch.float32)))
        kw = dict(keep_mask=keep, p_drop=p)
    elif case["drop"] == "seed":
        keep, scale = Fn.dropout_mask(seed, p, Ep, H, torch.device("cuda"))
        keep, kw = keep.bool().cpu(), dict(p_drop=p, seed=seed)
    au, dz, dad = _check_same_as_gather(t, H, C, **kw)
    r_au, r_dz, r_dad = _ref_dst_pass(t, H, C, keep, scale)
    _close(_csr_order(g, au), r_au)
    _close(_csr_order(g, dz), r_dz)
    _close(dad, r_dad)
    new = _full_bwd(t, H, C, False, **kw)
    old = _full_bwd(t, H, C, True, **kw)
    for a, b in zip(new, old):
        _close(a, b, tol=1e-9, rel=1e-6)
    if case["drop"] is None and case["dtype"] == torch.float32:
        cf = O.gatconv_backward_closed_form(t["x"].double(), ei, t["W"].double(), t["a_s"].double(), t["a_d"].double(),
                                            H, C, t["d_out"].double(), False, add_self_loops=False)
        _close(new[0].cpu(), cf["dxw"])
        _close(new[1].cpu(), cf["da_src"])
        _close(new[2].cpu(), cf["da_dst"])


def test_powerlaw_2m_nodes_20m_edges():
    N, E, H, C = 2_000_000, 20_000_000, 8, 64
    ei = synth.powerlaw_graph(N, E, seed=1234, device="cuda")
    t = _inputs(ei, N, 16, H, C, seed=51)
    _check_same_as_gather(t, H, C)
    new = _full_bwd(t, H, C, False)
    old = _full_bwd(t, H, C, True)
    for a, b in zip(new, old):
        assert relerr(a, b) <= 1e-6


def test_workspace_one_byte_short_is_refused():
    N, H, C = 3000, 8, 64
    ei = synth.random_graph(N, 20000, seed=3)
    t = _inputs(ei, N, 16, H, C, seed=61, hub_threshold=64, hub_chunk=64)
    g = t["g"]
    _, rowmax, rowsum = Fn.gat_fwd(g, t["xw"], t["a_src"], t["a_dst"], None, H, C, 0.2, False)
    L = _abi.lib()
    nb = ctypes.c_size_t()
    _abi.check(L.gnnfd_gat_bwd_workspace_bytes(g.ref(), H, C, ctypes.byref(nb)))
    # the dst pass's own need is the reported size less its 256-byte slack (no source hubs here); it must cover the
    # [E',H] d_alpha buffer
    need = nb.value - 256
    assert need >= g.n_edges * H * 4
    eg = torch.empty(g.n_edges, 2 * H, dtype=torch.float32, device="cuda")
    dad = torch.empty(N, H, dtype=torch.float32, device="cuda")
    d_out = t["d_out"].cuda()

    def call(ws_bytes):
        ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
        return L.gnnfd_gat_bwd_dst(g.ref(), t["xw"].data_ptr(), Fn._DT[t["xw"].dtype], t["a_src"].data_ptr(),
                                   t["a_dst"].data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(), d_out.data_ptr(), H, C,
                                   0.2, 0, 0, 0.0, 0, eg[:, :H].data_ptr(), eg[:, H:].data_ptr(), dad.data_ptr(),
                                   ws.data_ptr(), ws_bytes, Fn._stream())

    assert call(need - 1) == -3                   # GNNFD_ERR_WORKSPACE
    assert call(need) == 0
    torch.cuda.synchronize()
