"""The per-edge record of the two-pass head-mean backward: pass 1 writes {d_alpha, a_src[j]} at each edge's CSR position
(from the stream kernel, and from the hub kernel for sources above the hub threshold), and pass 2 reads only contiguous
streams -- the record, csr2csc and perm -- with the next chunk in flight, in the first sweep of every row and in the
second sweep of rows longer than one chunk.  Checked against the single-pass gather kernel (alpha_used bit for bit) and
the fp64 restatement of the dst pass."""
import ctypes

import pytest
import torch

from gnn_fraud_detection_b200 import _abi, functional as Fn, synth
from oracle import pyg_gatconv as O
from test_bwd_srcmajor_gpu import _check_same_as_gather, _close, _csr_order, _inputs, _ref_dst_pass

pytestmark = pytest.mark.gpu
THR = 256                 # hub_threshold: rows above it (in either direction) go to the hub kernels
HUB_SRC = 7               # a source with out-degree 2*THR + 5


def _record_graph(seed):
    """Destination rows of 33, 64, 65, 96, THR-1, THR and THR+1 edges, each placed among many short rows (packs) so
    that one work item walks packs, a multi-chunk row and packs again; and one source above the hub threshold."""
    N = 6000
    rnd = torch.Generator().manual_seed(seed)
    long_rows = {33: 1001, 64: 1503, 65: 2002, 96: 2504, THR - 1: 3001, THR: 3502, THR + 1: 4003}
    fixed = torch.tensor(list(long_rows.values()) + [HUB_SRC])
    short_ok = torch.ones(N, dtype=torch.bool)
    short_ok[fixed] = False
    pool = torch.nonzero(short_ok).view(-1)

    def pick(n):
        return pool[torch.randint(0, pool.numel(), (n,), generator=rnd)]

    parts = [torch.stack([pick(18000), pick(18000)])]                     # in-degree ~3: packs of short rows
    for deg, i in long_rows.items():
        parts.append(torch.stack([pick(deg), torch.full((deg,), i)]))
    parts.append(torch.stack([torch.full((2 * THR + 5,), HUB_SRC), pick(2 * THR + 5)]))
    return torch.cat(parts, 1), N, long_rows


CASES = [
    dict(H=8, C=64, dtype=torch.float32, drop=None),
    dict(H=8, C=64, dtype=torch.float32, drop="injected"),
    dict(H=8, C=64, dtype=torch.float32, drop="seed"),
    dict(H=8, C=64, dtype=torch.bfloat16, drop=None),
    dict(H=4, C=32, dtype=torch.float32, drop=None),
    dict(H=4, C=32, dtype=torch.float32, drop="seed"),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"H{c['H']}C{c['C']}-{str(c['dtype'])[6:]}-{c['drop']}")
def test_long_rows_among_packs_and_hub_source(case):
    H, C, p, seed = case["H"], case["C"], 0.3, 17
    ei, N, long_rows = _record_graph(seed=9)
    t = _inputs(ei, N, 16, H, C, seed=71, xw_dtype=case["dtype"], add_self_loops=False, hub_threshold=THR,
                hub_chunk=128)
    g = t["g"]
    rowptr, colptr = g.rowptr.cpu(), g.colptr.cpu()
    for deg, i in long_rows.items():
        assert int(rowptr[i + 1] - rowptr[i]) == deg
    assert int(colptr[HUB_SRC + 1] - colptr[HUB_SRC]) == 2 * THR + 5
    assert g.c.hub_src.n_hub >= 1 and g.c.hub_dst.n_hub >= 1
    Ep = g.n_edges
    kw, keep, scale = {}, None, 1.0
    if case["drop"] == "injected":
        keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(4)) >= p
        one = torch.ones((), dtype=torch.float32)
        scale = float(one / (one - torch.tensor(p, dtype=torch.float32)))
        kw = dict(keep_mask=keep, p_drop=p)
    elif case["drop"] == "seed":
        keep, scale = Fn.dropout_mask(seed, p, Ep, H, torch.device("cuda"))
        keep, kw = keep.bool().cpu(), dict(p_drop=p, seed=seed)
    au, dz, dad = _check_same_as_gather(t, H, C, **kw)          # alpha_used bit-equal, dz / da_dst to the last bits
    r_au, r_dz, r_dad = _ref_dst_pass(t, H, C, keep, scale)
    tol = dict(tol=2e-2, rel=2e-2) if case["dtype"] == torch.bfloat16 else {}
    if case["dtype"] == torch.float32:
        _close(_csr_order(g, au), r_au)
    _close(_csr_order(g, dz), r_dz, **tol)
    _close(dad, r_dad, **tol)
    if case["drop"] is None and case["dtype"] == torch.float32:
        cf = O.gatconv_backward_closed_form(t["x"].double(), ei, t["W"].double(), t["a_s"].double(), t["a_d"].double(),
                                            H, C, t["d_out"].double(), False, add_self_loops=False)
        _close(dad.cpu(), cf["da_dst"])


def test_workspace_covers_the_record_and_one_byte_short_is_refused():
    N, H, C = 3000, 8, 64
    ei = synth.random_graph(N, 20000, seed=5)
    t = _inputs(ei, N, 16, H, C, seed=81, hub_threshold=64, hub_chunk=64)
    g = t["g"]
    _, rowmax, rowsum = Fn.gat_fwd(g, t["xw"], t["a_src"], t["a_dst"], None, H, C, 0.2, False)
    L = _abi.lib()
    nb = ctypes.c_size_t()
    _abi.check(L.gnnfd_gat_bwd_workspace_bytes(g.ref(), H, C, ctypes.byref(nb)))
    need = nb.value - 256            # the dst pass's own need: the reported size less its 256-byte slack
    assert need >= g.n_edges * 2 * H * 4
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
