"""CPU oracle: a pure-torch restatement of the reference's GAT message-passing hot path.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  The product path
(``gnn_fraud_detection_b200``) never imports ``oracle`` and has no CPU fallback.

What it restates
----------------
The reference (aum2606/GNN-Fraud-Detection) delegates the layer arithmetic to the third-party,
un-vendored, un-pinned ``torch_geometric.nn.GATConv`` (``setup.py:13`` ``torch-geometric>=2.0.0``;
call sites ``src/models/gat.py:39,45,51,80`` and ``src/models/tgn.py:43,49,55,94``).  The shipped
checkpoints (``results/gat_model.pt``) carry the key set ``att_src, att_dst, bias, lin_src.weight,
lin_dst.weight`` which bounds the version to PyG 2.0.x-2.4.x.  The algorithm restated here is the
published one of that GATConv (SURVEY.md section 8(a2)/(a3)):

  * ``remove_self_loops`` (order preserving) then ``add_self_loops`` (``arange(N)`` appended last)
  * shared projection ``xw = x @ W^T`` viewed ``[N,H,C]``; ``a_src = (xw*att_src).sum(-1)``, same for dst
  * ``e = leaky_relu(a_src[j] + a_dst[i], 0.2)`` for edge j -> i
  * ``softmax`` per destination: ``exp(e - max_i) / (sum_i exp(e - max_i) + 1e-16)``
  * optional dropout on alpha, ``out_h[i] = sum_j alpha * xw[j]``, head mean or concat, ``+ bias``

plus the wrappers the reference itself owns: ``GAT.forward`` (``src/models/gat.py:78-96``),
``TemporalGNN.forward`` (``src/models/tgn.py:87-113``) and the documented intent of
``create_temporal_subgraph`` (``src/data/dataset.py:198-240``).

PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures for this path, and PyG is
not installed (nor installable) in this image, so this oracle cannot be checked against the reference
running here.  It is pinned only by (a) hand-computed closed-form cases in ``tests/test_oracle.py``,
(b) fp64 autograd-vs-closed-form agreement of the backward, (c) strict ``load_state_dict`` of the
reference's own checkpoints.  If ``torch_geometric`` ever becomes importable, ``real_pyg_available()``
turns on a direct comparison test.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

__all__ = [
    "real_pyg_available", "rewrite_self_loops", "csr_oracle", "csc_oracle", "gatconv_forward",
    "gatconv_backward_closed_form", "OracleGATConv", "OracleGAT", "OracleTemporalGNN",
    "temporal_subgraph_oracle", "glorot_",
]


def real_pyg_available() -> bool:
    try:
        import torch_geometric  # noqa: F401
        return True
    except Exception:
        return False


# ----------------------------------------------------------------------------------------------
# index work (bit-exact targets for the CUDA CSR builder)
# ----------------------------------------------------------------------------------------------
def rewrite_self_loops(edge_index: torch.Tensor, num_nodes: int, add_self_loops: bool = True) -> torch.Tensor:
    """PyG ``remove_self_loops`` + ``add_self_loops`` (GATConv.forward, every call).

    Existing self-loops are dropped with an order-preserving mask; one loop per node is appended at
    positions ``E_f .. E_f+N-1``.  Returns ``edge_index' [2, E']`` int64.
    """
    if not add_self_loops:
        return edge_index
    keep = edge_index[0] != edge_index[1]
    ei = edge_index[:, keep]
    loop = torch.arange(num_nodes, dtype=edge_index.dtype, device=edge_index.device)
    return torch.cat([ei, torch.stack([loop, loop])], dim=1)


def csr_oracle(edge_index: torch.Tensor, num_nodes: int, add_self_loops: bool = True, order: str = "dst"):
    """Destination-sorted CSR of the rewritten edge list.

    ``perm`` is ``torch.sort(dst', stable=True).indices`` (positions into ``edge_index'``), ``col`` the
    source of each sorted edge, ``rowptr`` int64 ``[N+1]``.  Stable => the self-loop is the last entry
    of every row.  ``order="dst_src"`` is PyG's ``sort_edge_index(edge_index', sort_by_row=False)``: a stable
    sort on the composite key ``dst' * N + src'`` (duplicates keep their order of appearance).
    """
    ei = rewrite_self_loops(edge_index, num_nodes, add_self_loops)
    src, dst = ei[0], ei[1]
    if order == "dst_src":
        _, perm = torch.sort(dst * max(num_nodes, 1) + src, stable=True)
        dst_sorted = dst[perm]
    else:
        dst_sorted, perm = torch.sort(dst, stable=True)
    counts = torch.bincount(dst_sorted, minlength=num_nodes)
    rowptr = torch.zeros(num_nodes + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(counts, 0)
    col = src[perm]
    return rowptr, col, perm, ei


def csc_oracle(rowptr: torch.Tensor, col: torch.Tensor, num_nodes: int):
    """Source-major twin used by the backward: stable sort of the CSR-ordered ``col`` array.

    Returns ``colptr [N+1]``, ``row`` (destination of each source-sorted edge) and ``eid`` (CSR position
    of each source-sorted edge, i.e. ``torch.sort(col, stable=True).indices``).
    """
    deg = rowptr[1:] - rowptr[:-1]
    dst_of_pos = torch.repeat_interleave(torch.arange(num_nodes, dtype=torch.int64), deg)
    col_sorted, eid = torch.sort(col, stable=True)
    counts = torch.bincount(col_sorted, minlength=num_nodes)
    colptr = torch.zeros(num_nodes + 1, dtype=torch.int64)
    colptr[1:] = torch.cumsum(counts, 0)
    row = dst_of_pos[eid]
    return colptr, row, eid


def temporal_subgraph_oracle(x, edge_index, time_steps, t):
    """Documented intent of ``create_temporal_subgraph`` (``src/data/dataset.py:198-240``).

    Nodes with ``time_steps == t`` (ascending original index), edges whose two endpoints are both in the
    step, original edge order preserved, endpoints relabelled ``0..n_t-1``.  (The reference's literal
    code compares 0-d tensors with int dict keys and would keep no edges; it is dead code there.)
    Returns ``(x_t, edge_index_t, node_indices)``.
    """
    mask = time_steps == t
    node_indices = torch.nonzero(mask).reshape(-1)
    relabel = torch.full((x.size(0),), -1, dtype=torch.int64)
    relabel[node_indices] = torch.arange(node_indices.numel(), dtype=torch.int64)
    emask = mask[edge_index[0]] & mask[edge_index[1]]
    ei = relabel[edge_index[:, emask]]
    return x[node_indices], ei, node_indices


# ----------------------------------------------------------------------------------------------
# the layer
# ----------------------------------------------------------------------------------------------
def gatconv_forward(x, edge_index, W, att_src, att_dst, bias, heads: int, out_channels: int,
                    concat: bool = False, negative_slope: float = 0.2, add_self_loops: bool = True,
                    dropout_mask: Optional[torch.Tensor] = None, p: float = 0.0,
                    dropout_scale: Optional[float] = None):
    """One GATConv forward in PyG 2.0-2.4 semantics.  dtype-generic (fp32 / fp64).

    ``dropout_mask`` is an optional ``[E',H]`` keep-mask in ``edge_index'`` order, applied as
    ``alpha * mask / (1-p)`` (``F.dropout`` semantics with an injected mask).  ``dropout_scale`` replaces
    ``1/(1-p)``: the CUDA kernels' counter-based generator scales its survivors by the exact keep
    probability of its 16-bit threshold (``functional.dropout_mask`` returns it).
    Returns ``out, (edge_index', alpha [E',H])``.
    """
    N, H, C = x.size(0), heads, out_channels
    ei = rewrite_self_loops(edge_index, N, add_self_loops)
    src, dst = ei[0], ei[1]
    xw = (x @ W.t()).view(N, H, C)
    a_s = (xw * att_src.view(1, H, C)).sum(-1)
    a_d = (xw * att_dst.view(1, H, C)).sum(-1)
    e = F.leaky_relu(a_s[src] + a_d[dst], negative_slope)
    m = torch.full((N, H), -math.inf, dtype=x.dtype)
    m = m.scatter_reduce(0, dst[:, None].expand_as(e), e.detach(), "amax", include_self=True)
    m = torch.where(torch.isinf(m), torch.zeros_like(m), m)  # rows with no edge (add_self_loops=False)
    pexp = (e - m[dst]).exp()
    s = torch.zeros(N, H, dtype=x.dtype).index_add_(0, dst, pexp) + 1e-16
    alpha = pexp / s[dst]
    alpha_used = alpha
    if dropout_mask is not None:
        if dropout_scale is None:
            alpha_used = alpha * dropout_mask.to(alpha.dtype) / (1.0 - p)
        else:
            alpha_used = alpha * dropout_mask.to(alpha.dtype) * dropout_scale
    msg = alpha_used[:, :, None] * xw[src]
    out = torch.zeros(N, H, C, dtype=x.dtype).index_add_(0, dst, msg)
    out = out.reshape(N, H * C) if concat else out.mean(1)
    if bias is not None:
        out = out + bias
    return out, (ei, alpha)


def gatconv_backward_closed_form(x, edge_index, W, att_src, att_dst, heads, out_channels, d_out,
                                 concat: bool = False, negative_slope: float = 0.2,
                                 add_self_loops: bool = True, need_dx: bool = True):
    """Closed-form gradients of ``gatconv_forward`` (dropout off), SURVEY.md section 8(a3).

    These are the formulas the CUDA backward kernels implement; ``tests/test_oracle.py`` checks them
    against autograd of ``gatconv_forward`` in fp64.
    Returns dict(dx, dW, datt_src, datt_dst, dbias, alpha, dz, da_src, da_dst, dxw).
    """
    N, H, C = x.size(0), heads, out_channels
    ei = rewrite_self_loops(edge_index, N, add_self_loops)
    src, dst = ei[0], ei[1]
    xw = (x @ W.t()).view(N, H, C)
    a_s = (xw * att_src.view(1, H, C)).sum(-1)
    a_d = (xw * att_dst.view(1, H, C)).sum(-1)
    z = a_s[src] + a_d[dst]
    e = F.leaky_relu(z, negative_slope)
    m = torch.full((N, H), -math.inf, dtype=x.dtype).scatter_reduce(
        0, dst[:, None].expand_as(e), e, "amax", include_self=True)
    m = torch.where(torch.isinf(m), torch.zeros_like(m), m)
    pexp = (e - m[dst]).exp()
    s = torch.zeros(N, H, dtype=x.dtype).index_add_(0, dst, pexp) + 1e-16
    alpha = pexp / s[dst]

    dbias = d_out.sum(0)
    if concat:
        dO_h = d_out.view(N, H, C)
    else:
        dO_h = (d_out / H)[:, None, :].expand(N, H, C)
    d_alpha = (dO_h[dst] * xw[src]).sum(-1)                                   # [E',H]
    t = torch.zeros(N, H, dtype=x.dtype).index_add_(0, dst, alpha * d_alpha)  # sum_k alpha_k dalpha_k
    de = alpha * (d_alpha - t[dst])
    dz = de * torch.where(z > 0, torch.ones_like(z), torch.full_like(z, negative_slope))
    da_src = torch.zeros(N, H, dtype=x.dtype).index_add_(0, src, dz)
    da_dst = torch.zeros(N, H, dtype=x.dtype).index_add_(0, dst, dz)
    dxw = torch.zeros(N, H, C, dtype=x.dtype).index_add_(0, src, alpha[:, :, None] * dO_h[dst])
    dxw = dxw + da_src[:, :, None] * att_src.view(1, H, C) + da_dst[:, :, None] * att_dst.view(1, H, C)
    datt_src = (da_src[:, :, None] * xw).sum(0).view(1, H, C)
    datt_dst = (da_dst[:, :, None] * xw).sum(0).view(1, H, C)
    dxw2 = dxw.reshape(N, H * C)
    dW = dxw2.t() @ x
    dx = dxw2 @ W if need_dx else None
    return dict(dx=dx, dW=dW, datt_src=datt_src, datt_dst=datt_dst, dbias=dbias, alpha=alpha, dz=dz,
                da_src=da_src, da_dst=da_dst, dxw=dxw2, edge_index=ei)


def glorot_(t: torch.Tensor, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """PyG ``inits.glorot``: U(-a, a), a = sqrt(6 / (size(-2) + size(-1)))."""
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        t.uniform_(-a, a, generator=generator)
    return t


class _SharedLinear(nn.Module):
    """Bias-free linear holding ``weight [out,in]`` (PyG ``Linear(..., bias=False)``)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))


class OracleGATConv(nn.Module):
    """nn.Module wrapper with PyG 2.0-2.4 parameter names (ctor sites ``src/models/gat.py:39,45,51``)."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, dropout=0.0,
                 add_self_loops=True, bias=True):
        super().__init__()
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.negative_slope, self.dropout = concat, negative_slope, dropout
        self.add_self_loops = add_self_loops
        self.lin_src = _SharedLinear(in_channels, heads * out_channels)
        self.lin_dst = self.lin_src  # alias, exactly as PyG does for a non-bipartite input
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        if bias:
            self.bias = nn.Parameter(torch.empty(heads * out_channels if concat else out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin_src.weight)
        glorot_(self.att_src)
        glorot_(self.att_dst)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x, edge_index, return_attention_weights=None, dropout_mask=None, dropout_scale=None):
        mask = dropout_mask
        p = self.dropout if self.training else 0.0
        if mask is None and self.training and self.dropout > 0:
            n_edges = rewrite_self_loops(edge_index, x.size(0), self.add_self_loops).size(1)
            mask = torch.rand(n_edges, self.heads) >= self.dropout
        out, (ei, alpha) = gatconv_forward(
            x, edge_index, self.lin_src.weight, self.att_src, self.att_dst, self.bias, self.heads,
            self.out_channels, self.concat, self.negative_slope, self.add_self_loops, mask, p, dropout_scale)
        if return_attention_weights:
            return out, (ei, alpha)
        return out


class OracleGAT(nn.Module):
    """Restatement of ``GAT`` (``src/models/gat.py:10-122``) over ``OracleGATConv``."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers=2, dropout=0.2,
                 residual=True, use_batch_norm=True):
        super().__init__()
        self.hidden_channels, self.dropout = hidden_channels, dropout
        self.residual, self.use_batch_norm = residual, use_batch_norm
        # gat.py:38-53: first layer always, num_layers-2 hidden layers, a last layer iff num_layers > 1
        widths = [in_channels] + [hidden_channels] * max(num_layers - 1, 0)
        self.gat_layers = nn.ModuleList(
            OracleGATConv(w, hidden_channels, heads=8, concat=False, dropout=dropout) for w in widths)
        self.batch_norms = nn.ModuleList(
            nn.BatchNorm1d(hidden_channels) for _ in widths) if use_batch_norm else None
        self.out = nn.Linear(hidden_channels, out_channels)

    def _stack(self, x, edge_index, att_masks=None, feat_masks=None, dropout_scale=None):
        """``att_masks`` / ``feat_masks``: optional per-layer keep-masks, ``[E',8]`` in ``edge_index'`` order for the
        attention coefficients and ``[N,hidden]`` for the features after the ReLU, applied as ``mask * dropout_scale``
        (default ``1/(1-p)``) in place of fresh random draws.  Given masks apply whatever the module's mode is."""
        h = x
        for i, gat in enumerate(self.gat_layers):
            if att_masks is None:
                h_new = gat(h, edge_index)
            else:
                h_new = gat(h, edge_index, dropout_mask=att_masks[i], dropout_scale=dropout_scale)
            if self.use_batch_norm:
                h_new = self.batch_norms[i](h_new)
            h_new = F.relu(h_new)
            if feat_masks is None:
                h_new = F.dropout(h_new, p=self.dropout, training=self.training)
            else:
                scale = 1.0 / (1.0 - self.dropout) if dropout_scale is None else dropout_scale
                h_new = h_new * feat_masks[i].to(h_new.dtype) * scale
            h = h + h_new if (self.residual and h.size(-1) == h_new.size(-1)) else h_new
        return h

    def forward(self, x, edge_index, batch=None, att_masks=None, feat_masks=None, dropout_scale=None):
        return self.out(self._stack(x, edge_index, att_masks, feat_masks, dropout_scale))

    def predict(self, x, edge_index, batch=None, apply_sigmoid=True):
        out = self.forward(x, edge_index, batch)
        return torch.sigmoid(out) if apply_sigmoid else out


class OracleTemporalGNN(OracleGAT):
    """Restatement of ``TemporalGNN`` (``src/models/tgn.py:14-141``): GAT stack + GRUCell + Linear."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers=2, dropout=0.2,
                 residual=True, use_batch_norm=True):
        super().__init__(in_channels, hidden_channels, out_channels, num_layers, dropout, residual,
                         use_batch_norm)
        self.gru = nn.GRUCell(hidden_channels, hidden_channels)

    def forward(self, x, edge_index, batch=None, hidden_state=None, att_masks=None, feat_masks=None,
                dropout_scale=None):
        if hidden_state is None:
            hidden_state = torch.zeros(x.size(0), self.hidden_channels, device=x.device)
        h = self._stack(x, edge_index, att_masks, feat_masks, dropout_scale)
        hidden_state = self.gru(h, hidden_state)
        return self.out(hidden_state), hidden_state

    def predict(self, x, edge_index, batch=None, hidden_state=None, apply_sigmoid=True):
        out, _ = self.forward(x, edge_index, batch, hidden_state)
        return torch.sigmoid(out) if apply_sigmoid else out
