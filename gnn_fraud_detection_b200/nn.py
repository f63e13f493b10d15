"""Drop-in ``GATConv``: the name the reference imports at ``src/models/gat.py:4`` / ``src/models/tgn.py:4``.

Same constructor arguments, ``forward(x, edge_index)`` signature, parameter names and ``state_dict`` keys
as ``torch_geometric.nn.GATConv`` 2.0-2.4 (``att_src``, ``att_dst``, ``bias``, ``lin_src.weight``,
``lin_dst.weight`` with ``lin_dst`` an alias of ``lin_src``), so the reference's shipped checkpoints
(``results/gat_model.pt``) load with ``strict=True``.  The arithmetic runs in ``libgnnfd_b200.so``; there
is no PyG, Triton or CPU fallback -- a CPU tensor or a missing extension raises.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn

from . import _abi
from .functional import gat_alpha, gatconv
from .graph import GLOBAL_CSR_CACHE, GraphCSR


def glorot_(t: torch.Tensor) -> torch.Tensor:
    """PyG ``inits.glorot``: U(-a, a) with a = sqrt(6 / (size(-2) + size(-1)))."""
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        return t.uniform_(-a, a)


def fold_batch_norm(batch_norm: Optional[nn.BatchNorm1d]):
    """Eval-mode BatchNorm as the per-channel affine ``(scale, shift)`` the fused epilogues take; ``(None, None)`` for none."""
    if batch_norm is None:
        return None, None
    inv = torch.rsqrt(batch_norm.running_var + batch_norm.eps)
    w = batch_norm.weight if batch_norm.weight is not None else torch.ones_like(inv)
    b = batch_norm.bias if batch_norm.bias is not None else torch.zeros_like(inv)
    return (w * inv).contiguous(), (b - batch_norm.running_mean * w * inv).contiguous()


class _Linear(nn.Module):
    """Bias-free projection holder; key ``weight`` has shape ``[heads*out_channels, in_channels]``."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, bias=False"


class GATConv(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, dropout: float = 0.0, add_self_loops: bool = True,
                 edge_dim: Optional[int] = None, fill_value="mean", bias: bool = True,
                 feature_dtype: torch.dtype = torch.float32, gemm_algo: int = _abi.GEMM_AUTO, **kwargs):
        super().__init__()
        if isinstance(in_channels, (tuple, list)):
            raise NotImplementedError("bipartite (x_src, x_dst) inputs are not part of the reference's hot path")
        if edge_dim is not None:
            raise NotImplementedError("edge_dim/edge_attr is never used by the reference models (src/config.py:36)")
        if kwargs:
            raise NotImplementedError(f"unsupported GATConv options: {sorted(kwargs)}")
        if feature_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("feature_dtype must be torch.float32 or torch.bfloat16")
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.negative_slope, self.dropout = concat, negative_slope, dropout
        self.add_self_loops = add_self_loops
        self.feature_dtype, self.gemm_algo = feature_dtype, gemm_algo
        self.last_dropout_seed = None
        self.lin_src = _Linear(in_channels, heads * out_channels)
        self.lin_dst = self.lin_src  # same module object: state_dict() emits both keys, as PyG does
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

    def _graph(self, edge_index, num_nodes: int) -> GraphCSR:
        if isinstance(edge_index, GraphCSR):
            return edge_index
        if not isinstance(edge_index, torch.Tensor):
            raise NotImplementedError("SparseTensor adjacency input is not supported; pass edge_index [2,E]")
        need_csc = torch.is_grad_enabled()
        return GLOBAL_CSR_CACHE.get(edge_index, num_nodes, self.add_self_loops, need_csc)

    def _check_inputs(self, x: torch.Tensor, g: GraphCSR, residual: Optional[torch.Tensor] = None):
        """Shape / dtype / device checks shared by the training path and the fused inference path: the C ABI takes raw
        pointers, so a wrong dtype or row count must be caught here."""
        if not x.is_cuda:
            raise RuntimeError("gnn_fraud_detection_b200.GATConv runs on CUDA only (no CPU fallback)")
        if x.dtype != torch.float32:
            raise TypeError(f"x must be float32, got {x.dtype}")
        if x.dim() != 2 or x.size(1) != self.in_channels:
            raise ValueError(f"x must be [N,{self.in_channels}], got {tuple(x.shape)}")
        if x.size(0) != g.n_src:
            raise ValueError(f"x has {x.size(0)} rows but the graph has {g.n_src} source nodes")
        if g.device != x.device:
            raise RuntimeError(f"graph lives on {g.device} but x on {x.device}")
        if residual is not None:
            Co = self.heads * self.out_channels if self.concat else self.out_channels
            if tuple(residual.shape) != (g.n_dst, Co) or residual.dtype != torch.float32 or residual.device != x.device:
                raise ValueError(f"residual must be float32 [{g.n_dst},{Co}] on {x.device}, got {residual.dtype} "
                                 f"{tuple(residual.shape)} on {residual.device}")

    def forward(self, x: torch.Tensor, edge_index, edge_attr=None, size=None, return_attention_weights=None,
                dropout_mask: Optional[torch.Tensor] = None):
        """``x [N, in_channels]`` fp32 cuda, ``edge_index [2,E]`` int64 cuda -> ``[N, out_channels]``.

        Attention dropout (training mode, ``dropout > 0``): the kernels draw the keep bits themselves from a counter-based
        RNG keyed on (seed, position in ``edge_index'``, head) -- no ``[E',H]`` mask tensor, no ``torch.rand`` pass; the
        seed comes from torch's CPU generator (reproducible under ``torch.manual_seed``) and is kept in ``last_dropout_seed``.
        ``dropout_mask``: optional explicit ``[E',H]`` keep-mask in ``edge_index'`` order (parity tests inject one).
        """
        if edge_attr is not None or size is not None:
            raise NotImplementedError("edge_attr / size are not part of the reference's hot path")
        if not x.is_cuda:
            raise RuntimeError("gnn_fraud_detection_b200.GATConv runs on CUDA only (no CPU fallback)")
        g = self._graph(edge_index, x.size(0))
        self._check_inputs(x, g)
        H, C = self.heads, self.out_channels
        p = self.dropout if self.training else 0.0
        keep = None
        if dropout_mask is not None:
            if not self.dropout > 0.0:
                raise ValueError("dropout_mask was given but this layer has dropout=0: the mask would be ignored")
            keep = dropout_mask.to(device=x.device, dtype=torch.uint8).contiguous()
            p = self.dropout
        if p >= 1.0:
            # F.dropout(alpha, p=1) zeroes every attention coefficient: the aggregation vanishes, the bias remains
            if return_attention_weights:
                raise NotImplementedError("return_attention_weights with dropout >= 1")
            out = x.new_zeros(g.n_dst, H * C if self.concat else C)
            return out + self.bias if self.bias is not None else out
        seed = 0
        if keep is None and p > 0.0:
            seed = int(torch.randint(0, 2 ** 62, (1,), device="cpu"))
            self.last_dropout_seed = seed
        if keep is not None and tuple(keep.shape) != (g.n_edges, H):
            raise ValueError(f"dropout_mask must be [{g.n_edges},{H}], got {tuple(keep.shape)}")
        res = gatconv(x, self.lin_src.weight, self.att_src, self.att_dst, self.bias, g, H, C, self.concat,
                      self.negative_slope, keep, p, self.feature_dtype, self.gemm_algo,
                      want_stats=bool(return_attention_weights), seed=seed)
        if not return_attention_weights:
            return res
        out, a_src, a_dst, rowmax, rowsum = res
        with torch.cuda.device(x.device):
            alpha_csr = gat_alpha(g, a_src, a_dst, rowmax, rowsum, H, self.negative_slope)
            # PyG returns (edge_index', alpha) in edge_index' order: un-permute the CSR-ordered alpha
            perm = g.perm.long()
            alpha = torch.empty_like(alpha_csr)
            alpha[perm] = alpha_csr
            dst_sorted = torch.repeat_interleave(torch.arange(g.n_dst, device=x.device),
                                                 (g.rowptr[1:] - g.rowptr[:-1]).long())
            ei = torch.empty(2, g.n_edges, dtype=torch.int64, device=x.device)
            ei[0, perm] = g.col.long()
            ei[1, perm] = dst_sorted
        return out, (ei, alpha)

    @torch.no_grad()
    def forward_fused_eval(self, x: torch.Tensor, edge_index, batch_norm: Optional[nn.BatchNorm1d] = None,
                           relu: bool = True, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Inference-only fast path for the reference's layer loop (``src/models/gat.py:80-91``):
        ``residual + relu(batch_norm_eval(gat(x, edge_index)))`` with the BatchNorm (running statistics folded to
        a per-channel affine), the ReLU and the residual add fused into the aggregation kernel's row epilogue (or, for a
        ``gemm_algo=GEMM_INPUT`` first layer, into the epilogue of the output GEMM)."""
        from . import functional as Fn
        if not x.is_cuda:
            raise RuntimeError("gnn_fraud_detection_b200.GATConv runs on CUDA only (no CPU fallback)")
        g = self._graph(edge_index, x.size(0))
        self._check_inputs(x, g, residual)
        H, C = self.heads, self.out_channels
        scale, shift = fold_batch_norm(batch_norm)
        act = _abi.ACT_RELU if relu else _abi.ACT_NONE
        res = None if residual is None else residual.contiguous()
        W = self.lin_src.weight.contiguous()
        a_s, a_d = self.att_src.reshape(-1), self.att_dst.reshape(-1)
        with torch.cuda.device(x.device):
            if self.gemm_algo == _abi.GEMM_INPUT and Fn.in_supported(x.size(1), H, C, self.concat):
                K = x.size(1)
                x16 = Fn.in_pad_x(x)
                prep = Fn._aligned_u8(Fn.in_sizes(g.n_dst, K)[0], x.device)
                xmax = torch.zeros(16, dtype=torch.float32, device=x.device)
                a_src, a_dst = Fn.in_logits(x16, W, a_s, a_d, prep, xmax)
                Fn.in_prepare(W, K, xmax, prep)
                zimg, _ = Fn.in_fwd(g, x16, a_src, a_dst, self.negative_slope, prep)
                return Fn.in_out(zimg, g.n_dst, K, prep, self.bias, act, scale, shift, res)
            x = x if x.stride(1) == 1 else x.contiguous()
            xw, a_src, a_dst = Fn.project_fwd(x, W, a_s, a_d, H, C, self.feature_dtype, self.gemm_algo)
            out, _, _ = Fn.gat_fwd(g, xw, a_src, a_dst, self.bias, H, C, self.negative_slope, self.concat, act, None, 0.0,
                                   scale, shift, res)
        return out

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, heads={self.heads}, concat={self.concat}"
