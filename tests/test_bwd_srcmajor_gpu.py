"""The dst-major backward of the head mean (concat=False), computed in two passes: d_alpha source-major, then the
feature-free row reductions.  Checked against the fp64 closed form, against an fp64 restatement that includes attention
dropout, and against the single-pass gather kernel: the same alpha_used bits, and dz / da_dst up to the last bits (the
gather kernel recomputes alpha for the second sweep of long rows with a contracted multiply-add)."""
import pytest
import torch
import torch.nn.functional as F

from gnn_fraud_detection_b200 import build_csr, functional as Fn, synth
from oracle import pyg_gatconv as O
from util import maxabs, relerr, seeded_params

pytestmark = pytest.mark.gpu
TOL32 = 1e-5      # the bars of test_gat_gpu.py: fp32 max-abs and relative L2 against fp64
REL32 = 1e-5
TOLBF = 2e-2      # bf16 feature storage: relative


def _inputs(ei, N, K, H, C, seed, xw_dtype=torch.float32, **csr_kw):
    W, a_s, a_d, _ = seeded_params(K, H, C, seed=seed)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(seed + 1))
    d_out = torch.randn(N, C, generator=torch.Generator().manual_seed(seed + 2)) / N
    g = build_csr(ei.cuda(), N, **csr_kw)
    asf, adf = a_s.view(-1).contiguous().cuda(), a_d.view(-1).contiguous().cuda()
    xw, a_src, a_dst = Fn.project_fwd(x.cuda(), W.cuda(), asf, adf, H, C, xw_dtype)
    return dict(x=x, W=W, a_s=a_s, a_d=a_d, d_out=d_out, g=g, xw=xw, a_src=a_src, a_dst=a_dst)


def _run(t, H, C, keep_mask=None, p_drop=0.0, seed=0, gather=False):
    """gat_fwd + gat_bwd_dst; gather=True hides the CSC so that the single-pass gather kernel runs instead."""
    g = t["g"]
    km = None if keep_mask is None else keep_mask.to(torch.uint8).cuda()
    _, rowmax, rowsum = Fn.gat_fwd(g, t["xw"], t["a_src"], t["a_dst"], None, H, C, 0.2, False, keep_mask=km,
                                   p_drop=p_drop, seed=seed)
    saved = g.c.colptr
    if gather:
        g.c.colptr = None
    try:
        au, dz, dad = Fn.gat_bwd_dst(g, t["xw"], t["a_src"], t["a_dst"], rowmax, rowsum, t["d_out"].cuda(), H, C, 0.2,
                                     False, km, p_drop, seed)
    finally:
        g.c.colptr = saved
    torch.cuda.synchronize()
    return au, dz, dad, rowmax, rowsum


def _csr_order(g, v):
    """[E',H] in source-major order -> dst-sorted (CSR) order"""
    return v[g.csr2csc.long()]


def _ref_dst_pass(t, H, C, keep=None, scale=1.0, slope=0.2):
    """fp64: alpha_used, dz in CSR order and da_dst, from the layer's own xw / logits (dropout included)."""
    g = t["g"]
    N = g.n_dst
    deg = (g.rowptr[1:] - g.rowptr[:-1]).long()
    dst = torch.repeat_interleave(torch.arange(N, device=deg.device), deg)
    src = g.col.long()
    xw, a_src, a_dst = t["xw"].double(), t["a_src"].double(), t["a_dst"].double()
    z = a_src[src] + a_dst[dst]
    e = F.leaky_relu(z, slope)
    m = torch.full((N, H), -torch.inf, dtype=torch.float64, device=z.device).scatter_reduce(
        0, dst[:, None].expand_as(e), e, "amax", include_self=True)
    p = (e - m[dst]).exp()
    s = torch.zeros(N, H, dtype=torch.float64, device=z.device).index_add_(0, dst, p)
    alpha = p / s[dst]
    k = torch.ones_like(alpha) if keep is None else keep.cuda()[g.perm.long()].double() * scale
    dal = ((t["d_out"].cuda().double() / H)[dst][:, None, :] * xw[src].view(-1, H, C)).sum(-1)
    u = alpha * k * dal
    tt = torch.zeros(N, H, dtype=torch.float64, device=z.device).index_add_(0, dst, u)
    dz = torch.where(z > 0, 1.0, slope) * (u - alpha * tt[dst])
    da_dst = torch.zeros(N, H, dtype=torch.float64, device=z.device).index_add_(0, dst, dz)
    return alpha * k, dz, da_dst


def _close(got, ref, tol=TOL32, rel=REL32):
    assert maxabs(got, ref) <= tol, f"max-abs {maxabs(got, ref):.3e}"
    if float(ref.double().norm()) > 1e-12:
        assert relerr(got, ref) <= rel, f"relative L2 {relerr(got, ref):.3e}"


def _check_closed_form(t, ei, N, H, C):
    """alpha_used, dz, da_dst against gatconv_backward_closed_form (fp64, dropout off)"""
    au, dz, dad, _, _ = _run(t, H, C)
    cf = O.gatconv_backward_closed_form(t["x"].double(), ei, t["W"].double(), t["a_s"].double(), t["a_d"].double(), H, C,
                                        t["d_out"].double(), False)
    perm = t["g"].perm.long().cpu()
    _close(_csr_order(t["g"], au).cpu(), cf["alpha"][perm])
    _close(_csr_order(t["g"], dz).cpu(), cf["dz"][perm])
    _close(dad.cpu(), cf["da_dst"])


def _check_same_as_gather(t, H, C, **kw):
    new = _run(t, H, C, **kw)[:3]
    old = _run(t, H, C, gather=True, **kw)[:3]
    assert torch.equal(new[0], old[0])
    for a, b in zip(new[1:], old[1:]):
        _close(a, b, tol=1e-9, rel=1e-6)
    return new


def test_multigraph_duplicates_self_loops_isolated_nodes():
    N, K, H, C = 600, 24, 8, 64
    ei = synth.random_graph(500, 4000, seed=3)                      # nodes 500..599 have no edges at all
    ei = torch.cat([ei, ei[:, :300], torch.tensor([[7, 7, 7], [7, 7, 7]])], 1)   # duplicates, repeated self loops
    t = _inputs(ei, N, K, H, C, seed=11)
    _check_closed_form(t, ei, N, H, C)
    _check_same_as_gather(t, H, C)


def test_hub_sources_and_hub_destinations():
    N, K, H, C = 3000, 20, 8, 64
    ei = synth.random_graph(N, 12000, seed=5)
    rnd = torch.Generator().manual_seed(21)
    hub_in = torch.stack([torch.randint(0, N, (900,), generator=rnd), torch.full((900,), 17)])     # in-degree 900
    mid_in = torch.stack([torch.randint(0, N, (70,), generator=rnd), torch.full((70,), 18)])       # several chunks, one sweep
    hub_out = torch.stack([torch.full((1300,), 19), torch.randint(0, N, (1300,), generator=rnd)])  # out-degree 1300
    ei = torch.cat([ei, hub_in, mid_in, hub_out], 1)
    t = _inputs(ei, N, K, H, C, seed=12, hub_threshold=64, hub_chunk=96)
    assert t["g"].c.hub_src.n_hub >= 1 and t["g"].c.hub_dst.n_hub >= 1
    _check_closed_form(t, ei, N, H, C)
    _check_same_as_gather(t, H, C)


def test_packed_short_rows():
    N, K, H, C = 5000, 16, 8, 64
    ei = synth.random_graph(N, 6000, seed=9, self_loops=False)     # in-degrees ~1-3: rows go through packs
    t = _inputs(ei, N, K, H, C, seed=13)
    _check_closed_form(t, ei, N, H, C)
    _check_same_as_gather(t, H, C)


def test_other_head_geometry():
    N, K, H, C = 800, 12, 4, 32
    ei = torch.cat([synth.random_graph(N, 5000, seed=4), torch.stack([torch.randint(0, N, (200,), generator=torch.Generator().manual_seed(23)), torch.full((200,), 3)])], 1)
    t = _inputs(ei, N, K, H, C, seed=14)
    _check_closed_form(t, ei, N, H, C)
    _check_same_as_gather(t, H, C)


def test_bf16_feature_storage():
    N, K, H, C = 2000, 40, 8, 64
    ei = synth.random_graph(N, 16000, seed=6)
    t = _inputs(ei, N, K, H, C, seed=15, xw_dtype=torch.bfloat16)
    au, dz, dad = _check_same_as_gather(t, H, C)
    # against fp64 from the stored (bf16) features; alpha against the fp32-feature closed form within the bf16 bar
    # (the edge gradients themselves carry the full bf16 rounding of xw: ~2e-2 relative on da_dst)
    r_au, r_dz, r_dad = _ref_dst_pass(t, H, C)
    _close(_csr_order(t["g"], au), r_au)
    _close(_csr_order(t["g"], dz), r_dz)
    _close(dad, r_dad)
    cf = O.gatconv_backward_closed_form(t["x"].double(), ei, t["W"].double(), t["a_s"].double(), t["a_d"].double(), H, C,
                                        t["d_out"].double(), False)
    assert relerr(_csr_order(t["g"], au).cpu(), cf["alpha"][t["g"].perm.long().cpu()]) <= TOLBF


@pytest.mark.parametrize("injected", [True, False])
def test_attention_dropout(injected):
    N, K, H, C, p, seed = 1500, 20, 8, 64, 0.3, 77
    ei = torch.cat([synth.random_graph(N, 12000, seed=8), torch.stack([torch.randint(0, N, (700,), generator=torch.Generator().manual_seed(24)), torch.full((700,), 5)])], 1)
    t = _inputs(ei, N, K, H, C, seed=16, hub_threshold=256, hub_chunk=128)
    Ep = t["g"].n_edges
    if injected:
        keep = torch.rand(Ep, H, generator=torch.Generator().manual_seed(1)) >= p
        one = torch.ones((), dtype=torch.float32)
        scale, kw = float(one / (one - torch.tensor(p, dtype=torch.float32))), dict(keep_mask=keep, p_drop=p)
    else:
        keep, scale = Fn.dropout_mask(seed, p, Ep, H, torch.device("cuda"))     # what the kernels draw from the seed
        keep, kw = keep.bool().cpu(), dict(p_drop=p, seed=seed)
    au, dz, dad = _check_same_as_gather(t, H, C, **kw)
    r_au, r_dz, r_dad = _ref_dst_pass(t, H, C, keep, scale)
    _close(_csr_order(t["g"], au), r_au)
    _close(_csr_order(t["g"], dz), r_dz)
    _close(dad, r_dad)
    # dropped coefficients are exactly zero, the kept ones are gat_alpha times the keep scale
    _, _, _, rowmax, rowsum = _run(t, H, C, **kw)
    alpha = Fn.gat_alpha(t["g"], t["a_src"], t["a_dst"], rowmax, rowsum, H, 0.2)
    k = keep.cuda()[t["g"].perm.long()]
    au = _csr_order(t["g"], au)
    assert torch.equal(au == 0, ~k | (alpha == 0))
    _close(au, alpha * torch.where(k, torch.tensor(scale, dtype=torch.float32).cuda(), 0.0), tol=1e-6, rel=1e-6)


def test_alpha_used_matches_gat_alpha():
    """alpha_used in CSR order is the attention coefficient gat_alpha returns (which divides by the row sum where the
    backward multiplies by its reciprocal: last-bit differences)"""
    N, K, H, C = 3000, 20, 8, 64
    rnd = torch.Generator().manual_seed(22)
    ei = torch.cat([synth.random_graph(N, 20000, seed=2),
                    torch.stack([torch.randint(0, N, (600,), generator=rnd), torch.full((600,), 9)]),
                    torch.stack([torch.full((800,), 10), torch.randint(0, N, (800,), generator=rnd)])], 1)
    t = _inputs(ei, N, K, H, C, seed=17, hub_threshold=128, hub_chunk=128)
    au, _, _, rowmax, rowsum = _run(t, H, C)
    alpha = Fn.gat_alpha(t["g"], t["a_src"], t["a_dst"], rowmax, rowsum, H, 0.2)
    _close(_csr_order(t["g"], au), alpha, tol=1e-6, rel=1e-6)
