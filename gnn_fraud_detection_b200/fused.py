"""Model-level fused operators around the GAT layers (``include/gnnfd_b200.h`` section (6), ``csrc/model_ops.cu``).

* ``bn_relu_dropout_residual`` -- the train-mode tail of the reference's layer loop (``src/models/gat.py:82-91`` ==
  ``src/models/tgn.py:96-105``): ``h + dropout(relu(batch_norm(z)))`` with BATCH statistics, in two kernels forward
  (column sums, one elementwise pass) and two backward; running statistics are updated exactly as ``nn.BatchNorm1d`` does.
  Across GPUs the per-channel sums are all-reduced, i.e. the statistics are those of the whole batch (SURVEY.md 8(e)).
* ``gru_head`` -- the TemporalGNN head (``src/models/tgn.py:60,88-89,108-111``): ``GRUCell`` + ``Linear(64 -> 1)``.
* ``masked_bce_with_logits`` -- the reference's loss (``src/train.py:108-139,360-361``) and confusion counters on the device.

PyTorch provides tensors, autograd bookkeeping and the process group; the arithmetic runs in ``libgnnfd_b200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _abi
from .graph import _stream


def _ws(n_rows: int, device) -> torch.Tensor:
    nb = C.c_size_t()
    _abi.check(_abi.lib().gnnfd_model_ops_workspace_bytes(int(n_rows), C.byref(nb)))
    return torch.empty(nb.value, dtype=torch.uint8, device=device)


def _draw_seed() -> int:
    return int(torch.randint(0, 2 ** 62, (1,), device="cpu"))


class _BNReluDropRes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, gamma, beta, residual, running_mean, running_var, eps, momentum, p_drop, seed, row_base, group,
                global_rows, bcast):
        L = _abi.lib()
        z = z.contiguous()
        N, Cc = z.shape
        dev = z.device
        with torch.cuda.device(dev):
            ws = _ws(N, dev)
            sums = torch.empty(2 * Cc, dtype=torch.float64, device=dev)
            _abi.check(L.gnnfd_bn_sums(z.data_ptr(), N, Cc, sums.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
            count = float(N)
            if group is not None:
                dist.all_reduce(sums, group=group)
                if global_rows is not None:           # known batch size: no second collective, no host synchronisation
                    count = float(global_rows)
                else:
                    cnt = torch.tensor([count], dtype=torch.float64, device=dev)
                    dist.all_reduce(cnt, group=group)
                    count = float(cnt.item())
            if count == 1.0:
                # as nn.BatchNorm1d: one row has no batch variance (the output would silently be relu(beta))
                raise ValueError(f"Expected more than 1 value per channel when training, got input size {[1, Cc]}")
            mean = torch.empty(Cc, dtype=torch.float32, device=dev)
            invstd = torch.empty(Cc, dtype=torch.float32, device=dev)
            _abi.check(L.gnnfd_bn_finalize(sums.data_ptr(), count, Cc, float(eps), float(momentum), _abi.ptr(running_mean),
                                           _abi.ptr(running_var), mean.data_ptr(), invstd.data_ptr(), _stream()))
            out = torch.empty_like(z)
            res = None if residual is None else residual.contiguous()
            if bcast is None:
                _abi.check(L.gnnfd_bn_relu_drop_res_fwd(z.data_ptr(), N, Cc, mean.data_ptr(), invstd.data_ptr(),
                                                        _abi.ptr(gamma), _abi.ptr(beta), float(p_drop), int(seed),
                                                        int(row_base), _abi.ptr(res), out.data_ptr(), _stream()))
            else:
                peers, row_offset, use_multicast = bcast
                _abi.check(L.gnnfd_bn_relu_drop_res_fwd_bcast(z.data_ptr(), N, Cc, mean.data_ptr(), invstd.data_ptr(),
                                                              _abi.ptr(gamma), _abi.ptr(beta), float(p_drop), int(seed),
                                                              int(row_base), _abi.ptr(res), C.byref(peers), int(row_offset),
                                                              int(use_multicast), out.data_ptr(), _stream()))
        ctx.save_for_backward(z, mean, invstd, gamma, beta)
        ctx.p, ctx.seed, ctx.row_base, ctx.group, ctx.count = p_drop, seed, row_base, group, count
        ctx.has_res = residual is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        L = _abi.lib()
        z, mean, invstd, gamma, beta = ctx.saved_tensors
        d_out = d_out.contiguous()
        N, Cc = z.shape
        dev = z.device
        with torch.cuda.device(dev):
            ws = _ws(N, dev)
            sums = torch.empty(2 * Cc, dtype=torch.float64, device=dev)
            _abi.check(L.gnnfd_bn_bwd_sums(z.data_ptr(), d_out.data_ptr(), N, Cc, mean.data_ptr(), invstd.data_ptr(),
                                           _abi.ptr(gamma), _abi.ptr(beta), float(ctx.p), int(ctx.seed), int(ctx.row_base),
                                           sums.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
            if ctx.group is not None:
                dist.all_reduce(sums, group=ctx.group)
            dz = torch.empty_like(z)
            dgamma = torch.empty_like(gamma) if gamma is not None else None
            dbeta = torch.empty_like(beta) if beta is not None else None
            _abi.check(L.gnnfd_bn_bwd_apply(z.data_ptr(), d_out.data_ptr(), N, Cc, mean.data_ptr(), invstd.data_ptr(),
                                            _abi.ptr(gamma), _abi.ptr(beta), float(ctx.p), int(ctx.seed), int(ctx.row_base),
                                            sums.data_ptr(), float(ctx.count), dz.data_ptr(), _abi.ptr(dgamma), _abi.ptr(dbeta),
                                            _stream()))
        return (dz, dgamma, dbeta, (d_out if ctx.has_res else None), None, None, None, None, None, None, None, None, None,
                None)


def bn_relu_dropout_residual(z: torch.Tensor, bn: nn.BatchNorm1d, p_drop: float = 0.0,
                             residual: Optional[torch.Tensor] = None, seed: Optional[int] = None, row_base: int = 0,
                             group=None, global_rows: Optional[int] = None, bcast=None) -> torch.Tensor:
    """``residual + dropout(relu(bn(z)))`` with ``bn`` in TRAINING mode (batch statistics, running buffers updated).

    ``group``: a process group whose ranks hold disjoint rows of one batch -- the statistics are then those of the whole
    batch and ``row_base`` is this rank's first global row (it keys the dropout generator); ``global_rows`` = the batch size
    over all ranks, if known (saves a collective and a host synchronisation: required under CUDA-graph capture).
    ``bcast = (peers, row_offset, use_multicast)``: the finished rows also go to rows ``row_offset ..`` of the symmetric
    ``[n_pos, C]`` buffer described by ``peers`` (``_abi.Peers``) on EVERY rank (``gnnfd_bn_relu_drop_res_fwd_bcast``); the
    caller puts a cross-GPU barrier between this and the first read of that buffer."""
    if not z.is_cuda or z.dtype != torch.float32 or z.dim() != 2:
        raise RuntimeError("bn_relu_dropout_residual needs a float32 CUDA tensor [N,C] (no CPU fallback)")
    if not bn.training:
        raise RuntimeError("bn_relu_dropout_residual implements the TRAINING-mode BatchNorm (batch statistics)")
    if bn.momentum is None:
        raise NotImplementedError("cumulative-average BatchNorm (momentum=None) is not used by the reference")
    if residual is not None and (residual.shape != z.shape or residual.dtype != torch.float32 or residual.device != z.device):
        raise ValueError("residual must match z in shape, dtype and device")
    if z.size(1) % 4 or z.size(1) > 256:
        raise NotImplementedError("channel count must be a multiple of 4 and <= 256")
    if p_drop > 0.0 and seed is None:
        seed = _draw_seed()
    out = _BNReluDropRes.apply(z, bn.weight, bn.bias, residual, bn.running_mean, bn.running_var, bn.eps, bn.momentum,
                               float(p_drop), int(seed or 0), int(row_base), group, global_rows, bcast)
    if bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
    return out


class _GRUHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, h_prev, w_ih, w_hh, b_ih, b_hh, w_out, b_out):
        L = _abi.lib()
        x = x.contiguous()
        hp = None if h_prev is None else h_prev.contiguous()
        N, dev = x.size(0), x.device
        h_new = torch.empty(N, 64, dtype=torch.float32, device=dev)
        out = torch.empty(N, 1, dtype=torch.float32, device=dev)
        params = [t.contiguous() for t in (w_ih, w_hh, b_ih, b_hh, w_out, b_out)]
        with torch.cuda.device(dev):
            _abi.check(L.gnnfd_gru_head_fwd(x.data_ptr(), _abi.ptr(hp), N, *[t.data_ptr() for t in params], h_new.data_ptr(),
                                            out.data_ptr(), _stream()))
        ctx.save_for_backward(x, hp, *params)
        return out, h_new

    @staticmethod
    def backward(ctx, d_out, d_hnew):
        L = _abi.lib()
        x, hp, w_ih, w_hh, b_ih, b_hh, w_out, b_out = ctx.saved_tensors
        N, dev = x.size(0), x.device
        d_o = None if d_out is None else d_out.contiguous().float()
        d_h = None if d_hnew is None else d_hnew.contiguous().float()
        dx = torch.empty_like(x)
        dhp = torch.empty_like(hp) if hp is not None else None
        grads = [torch.empty_like(t) for t in (w_ih, w_hh, b_ih, b_hh, w_out, b_out)]
        with torch.cuda.device(dev):
            gates = torch.empty(2 * max(N, 1) * 192, dtype=torch.float32, device=dev)
            ws = _ws(N, dev)
            _abi.check(L.gnnfd_gru_head_bwd(x.data_ptr(), _abi.ptr(hp), _abi.ptr(d_o), _abi.ptr(d_h), N, w_ih.data_ptr(),
                                            w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), w_out.data_ptr(), b_out.data_ptr(),
                                            dx.data_ptr(), _abi.ptr(dhp), grads[0].data_ptr(), grads[1].data_ptr(),
                                            grads[2].data_ptr(), grads[3].data_ptr(), grads[4].data_ptr(), grads[5].data_ptr(),
                                            gates.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
        return (dx, dhp, *grads)


def gru_head_supported(gru: nn.GRUCell, lin: nn.Linear) -> bool:
    return (gru.input_size == 64 and gru.hidden_size == 64 and gru.bias and lin.in_features == 64 and lin.out_features == 1
            and lin.bias is not None)


def gru_head(x: torch.Tensor, gru: nn.GRUCell, lin: nn.Linear, h_prev: Optional[torch.Tensor] = None
             ) -> Tuple[torch.Tensor, torch.Tensor]:
    """``(lin(h'), h')`` with ``h' = gru(x, h_prev)``; ``h_prev=None`` is the reference's zero state (``tgn.py:88-89``)."""
    if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.size(1) != 64:
        raise RuntimeError("gru_head needs a float32 CUDA tensor [N,64] (no CPU fallback)")
    if not gru_head_supported(gru, lin):
        raise NotImplementedError("gru_head is built for GRUCell(64, 64) + Linear(64, 1) with biases (the reference's head)")
    if h_prev is not None and (h_prev.shape != x.shape or h_prev.dtype != torch.float32 or h_prev.device != x.device):
        raise ValueError("hidden_state must be float32 [N,64] on the device of x")
    return _GRUHead.apply(x, h_prev, gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh, lin.weight.view(-1), lin.bias)


class _MaskedBCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, y, pos_weight):
        L = _abi.lib()
        lg = logits.contiguous().view(-1)
        N, dev = lg.numel(), lg.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        grad = torch.empty(N, dtype=torch.float32, device=dev)
        stats = torch.empty(8, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws = _ws(N, dev)
            _abi.check(L.gnnfd_bce_masked(lg.data_ptr(), y.data_ptr(), N, float(pos_weight), 1.0, loss.data_ptr(), grad.data_ptr(),
                                          stats.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
        ctx.save_for_backward(grad)
        ctx.shape = logits.shape
        ctx.mark_non_differentiable(stats)
        return loss.view(()), stats

    @staticmethod
    def backward(ctx, d_loss, _d_stats):
        (grad,) = ctx.saved_tensors
        return (grad * d_loss).view(ctx.shape), None, None


def masked_bce_with_logits(logits: torch.Tensor, y: torch.Tensor, pos_weight: float = 1.0):
    """Mean over the labelled nodes (``y != -1``) of ``BCEWithLogitsLoss(pos_weight)`` -- the loss of ``src/train.py:108-139``
    -- plus device-resident statistics ``[sum of losses, labelled count, TP, FP, TN, FN, 0, 0]`` (float64; threshold
    sigmoid >= 0.5 as in ``src/train.py:146-149``).  Nothing is copied to the host."""
    if not logits.is_cuda or logits.dtype != torch.float32:
        raise RuntimeError("masked_bce_with_logits needs float32 CUDA logits (no CPU fallback)")
    if y.dtype != torch.int64 or y.device != logits.device or y.numel() != logits.numel():
        raise ValueError("y must be int64 (-1 = unlabelled, 0 / 1) with one entry per logit, on the device of logits")
    return _MaskedBCE.apply(logits, y.contiguous().view(-1), float(pos_weight))
