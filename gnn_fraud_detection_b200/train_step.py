"""Device-resident full-batch training step (SURVEY.md 8(f) rank 4).

The reference's train loop (``src/train.py:103-149``) moves the whole graph to the device every step (``batch.to(device)``,
``:105``), computes a masked ``BCEWithLogitsLoss(pos_weight=50)`` (``:108-139``), steps Adam (``:142-143``) and then
synchronises three times to build Python lists of predictions (``:146-149``).  Once a layer takes about a millisecond those
copies and syncs ARE the step.  ``DeviceTrainStep`` keeps ``x``, ``edge_index`` and ``y`` resident, evaluates the loss and
the confusion counters on the device (``fused.masked_bce_with_logits``), and replays forward + loss + backward + optimizer
from ONE CUDA graph; nothing reaches the host until ``metrics()`` is called.

Dropout inside a replayed graph: the kernel seeds are launch constants, so the step bumps a device counter inside the graph
and registers it with ``gnnfd_set_dropout_seed_source`` -- every replay draws fresh attention / feature dropout masks.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _abi, fused
from .graph import GLOBAL_CSR_CACHE
from .models import TemporalGNN


class DeviceTrainStep:
    def __init__(self, model: torch.nn.Module, x: torch.Tensor, edge_index: torch.Tensor, y: torch.Tensor,
                 optimizer: Optional[torch.optim.Optimizer] = None, pos_weight: float = 50.0, use_cuda_graph: bool = True,
                 lr: float = 1e-3, weight_decay: float = 5e-4):
        if not (x.is_cuda and edge_index.is_cuda and y.is_cuda):
            raise RuntimeError("DeviceTrainStep keeps the batch resident on the GPU: move x, edge_index and y there once")
        self.model, self.x, self.edge_index, self.y = model, x, edge_index, y.contiguous().view(-1).long()
        self.pos_weight = float(pos_weight)
        # Adam(lr=1e-3, weight_decay=5e-4) as src/train.py:353-357; capturable so that its step lives in the graph
        self.optimizer = optimizer or torch.optim.Adam(model.parameters(), lr=lr, weight_decay=weight_decay, capturable=True)
        self.is_tgn = isinstance(model, TemporalGNN)
        self.loss = torch.zeros((), device=x.device)
        self.stats = torch.zeros(8, dtype=torch.float64, device=x.device)
        self.totals = torch.zeros(8, dtype=torch.float64, device=x.device)      # running sums over the steps of an epoch
        self.seed_word = torch.zeros(1, dtype=torch.int64, device=x.device)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.steps = 0
        # the CSR/CSC of the resident edge_index is built once (cache keyed on the tensor)
        GLOBAL_CSR_CACHE.get(edge_index, x.size(0), True, True)
        if use_cuda_graph:
            self._capture()

    # one step, eagerly: also what gets captured
    def _step_impl(self):
        self.seed_word.add_(0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF)            # fresh dropout masks on every (re)play
        self.optimizer.zero_grad(set_to_none=False)
        r = self.model(self.x, self.edge_index)
        logits = r[0] if self.is_tgn else r
        loss, stats = fused.masked_bce_with_logits(logits, self.y, self.pos_weight)
        loss.backward()
        self.optimizer.step()
        self.loss.copy_(loss.detach())
        self.stats.copy_(stats)
        self.totals.add_(stats)

    def _capture(self):
        dev = self.x.device
        lib = _abi.lib()
        for p in self.model.parameters():           # gradients must exist (and keep their storage) before capture
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        lib.gnnfd_set_dropout_seed_source(self.seed_word.data_ptr())
        with torch.cuda.stream(s):
            for _ in range(3):                      # warm-up: allocator, lazy initialisations, optimizer state
                self._step_impl()
            s.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=s):
                self._step_impl()
        torch.cuda.current_stream(dev).wait_stream(s)
        self.totals.zero_()
        self.steps = 0

    def step(self):
        """One optimizer step.  Returns device tensors ``(loss, stats)``; no host synchronisation."""
        self.model.train()
        if self.graph is not None:
            self.graph.replay()
        else:
            self._step_impl()
        self.steps += 1
        return self.loss, self.stats

    def metrics(self, reset: bool = True) -> Dict[str, float]:
        """Host copy of the counters accumulated since the last reset (ONE synchronisation): mean loss per labelled node and
        the confusion matrix the reference derives from its Python lists (``src/train.py:146-149``, ``utils/metrics.py``)."""
        t = self.totals.tolist()
        if reset:
            self.totals.zero_()
        return metrics_from_totals(t)

    def close(self):
        _abi.lib().gnnfd_set_dropout_seed_source(None)
        self.graph = None


def metrics_from_totals(t) -> Dict[str, float]:
    """The counters of ``masked_bce_with_logits`` summed over steps (``[sum of losses, labelled, TP, FP, TN, FN, ..]``) ->
    mean loss per labelled node and the confusion-matrix metrics."""
    n = max(t[1], 1.0)
    tp, fp, tn, fn = t[2], t[3], t[4], t[5]
    prec = tp / (tp + fp) if tp + fp else 0.0
    rec = tp / (tp + fn) if tp + fn else 0.0
    return {"loss": t[0] / n, "labelled": t[1], "tp": tp, "fp": fp, "tn": tn, "fn": fn, "accuracy": (tp + tn) / n,
            "precision": prec, "recall": rec, "f1": 2 * prec * rec / (prec + rec) if prec + rec else 0.0}
