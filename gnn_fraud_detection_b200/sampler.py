"""Neighbour sampling on the GPU: the mini-batch path of the reference (``--use_subgraph_sampling`` makes
``src/data/dataloader.py:42-66`` build ``NeighborLoader(data, num_neighbors=[10, 10, 10], batch_size=256, ...)``).

``NeighborSampler`` builds the raw destination-sorted CSR of ``edge_index`` once (``build_csr(..., add_self_loops=False)``)
and samples a batch per call through ``gnnfd_neighbor_sample`` (``csrc/sample.cu``): PyG's defaults ``replace=False``,
``directed=True``, PyG's output fields and numbering.  The selection of a node's neighbours is a function of
``(seed, node)`` only (contract: ``include/gnnfd_b200.h`` section (8)); toward PyG's own sampler, which draws from a
different generator, the contract is distributional.  ``NeighborLoader`` is the drop-in for the reference's call.
CUDA tensors only; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from types import SimpleNamespace
from typing import Optional, Sequence

import torch

from . import _abi
from .graph import build_csr

__all__ = ["NeighborSampler", "NeighborLoader"]

_U64 = (1 << 64) - 1


class NeighborSampler:
    """``sample(seeds)`` -> ``SimpleNamespace(n_id, edge_index, e_id, batch_size, num_sampled_nodes, num_sampled_edges)``:
    ``n_id`` global ids (the seeds first), ``edge_index`` [2, m] local ids (row 1 non-decreasing), ``e_id`` columns of the
    input ``edge_index``, per-hop counts under PyG's names.  ``num_neighbors[l]`` is the fanout of hop l+1 (``-1``: all)."""

    def __init__(self, edge_index: torch.Tensor, num_nodes: int, num_neighbors: Sequence[int]):
        if not isinstance(edge_index, torch.Tensor) or not edge_index.is_cuda:
            raise RuntimeError("NeighborSampler runs on CUDA tensors only (no CPU fallback)")
        self.num_neighbors = [int(k) for k in num_neighbors]
        if any(k < -1 for k in self.num_neighbors):
            raise ValueError(f"num_neighbors entries must be >= -1, got {self.num_neighbors}")
        self.num_nodes, self.num_edges = int(num_nodes), int(edge_index.size(1))
        self.device = edge_index.device
        self.graph = build_csr(edge_index, self.num_nodes, add_self_loops=False, build_csc=False)
        deg = self.graph.rowptr[1:] - self.graph.rowptr[:-1]
        self.max_degree = int(deg.max()) if self.num_nodes > 0 else 0
        self.node_map = torch.full((self.num_nodes,), -1, dtype=torch.int32, device=self.device)
        self._ws = None

    def caps(self, batch_size: int):
        """Output capacities that always suffice for ``batch_size`` distinct seeds."""
        N, E = self.num_nodes, self.num_edges
        front = nodes = int(batch_size)
        edges = 0
        for k in self.num_neighbors:
            m = min(front * (self.max_degree if k == -1 else k), E)
            edges += m
            front = min(m, N)
            nodes += front
        return max(int(batch_size), min(N, nodes)), min(E, edges)

    def sample(self, seeds: torch.Tensor, seed: Optional[int] = None) -> SimpleNamespace:
        """Sample the subgraph around ``seeds`` (distinct node ids, CUDA).  ``seed`` keys the generator; ``None`` draws it
        from torch's CPU generator, so results are reproducible under ``torch.manual_seed``.

        The outputs are allocated at the bounds of ``caps`` (8 bytes per node, 24 per edge) and returned as views of
        those buffers, so the caller owns them.  With a ``-1`` fanout the edge bound reaches ``min(E, ...)`` with the
        maximum in-degree standing for every node: on a graph with a hub, a few seeds at ``-1`` reserve about 24 * E
        bytes for the call (4.8 GB at 200M edges), however small the sample turns out."""
        if not isinstance(seeds, torch.Tensor) or not seeds.is_cuda:
            raise RuntimeError("NeighborSampler.sample takes CUDA seed tensors only (no CPU fallback)")
        if seeds.device != self.device:
            raise RuntimeError(f"seeds live on {seeds.device} but the graph on {self.device}")
        if seeds.dtype not in (torch.int64, torch.int32) or seeds.dim() != 1:
            raise ValueError(f"seeds must be a 1-D integer tensor, got {seeds.dtype} {tuple(seeds.shape)}")
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,), device="cpu"))
        seeds = seeds.long().contiguous()
        B, L, dev = seeds.numel(), len(self.num_neighbors), self.device
        node_cap, edge_cap = self.caps(B)
        lib = _abi.lib()
        nbytes = C.c_size_t()
        _abi.check(lib.gnnfd_sample_workspace_bytes(node_cap, edge_cap, L, C.byref(nbytes)))
        if self._ws is None or self._ws.numel() < nbytes.value:
            self._ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        n_id = torch.empty(node_cap, dtype=torch.int64, device=dev)
        ei = torch.empty(2, edge_cap, dtype=torch.int64, device=dev)
        e_id = torch.empty(edge_cap, dtype=torch.int64, device=dev)
        fan = (C.c_int32 * max(L, 1))(*self.num_neighbors)
        counts = (C.c_int64 * (3 + 2 * L))()
        g = self.graph
        with torch.cuda.device(dev):
            _abi.check(lib.gnnfd_neighbor_sample(
                g.rowptr.data_ptr(), _abi.ptr(g.col), _abi.ptr(g.perm), self.num_nodes, seeds.data_ptr(), B, fan, L,
                int(seed) & _U64, self.node_map.data_ptr(), n_id.data_ptr(), node_cap, ei.data_ptr(), edge_cap,
                e_id.data_ptr(), edge_cap, counts, self._ws.data_ptr(), nbytes.value,
                torch.cuda.current_stream(dev).cuda_stream))
        n, m = int(counts[0]), int(counts[1])
        return SimpleNamespace(n_id=n_id[:n], edge_index=ei[:, :m].contiguous(), e_id=e_id[:m], batch_size=B,
                               num_sampled_nodes=[int(c) for c in counts[2:3 + L]],
                               num_sampled_edges=[int(c) for c in counts[3 + L:3 + 2 * L]])


class NeighborLoader:
    """Drop-in for ``torch_geometric.loader.NeighborLoader(data, num_neighbors, input_nodes, batch_size, shuffle,
    drop_last)`` with PyG's defaults ``replace=False``, ``directed=True``.  ``data``: any object with CUDA ``x`` and
    ``edge_index`` (optionally ``y``, ``time_steps``).  ``input_nodes``: ``None`` (every node), a bool mask or an index
    tensor.  Each batch carries ``x``, ``y``, ``time_steps`` sliced by ``n_id``, ``edge_index``, ``n_id``, ``e_id``,
    ``input_id`` (positions in ``input_nodes`` of the seeds), ``batch_size``, ``num_sampled_nodes`` and
    ``num_sampled_edges``; the seeds are the first ``batch_size`` rows.  Shuffling and the sampler's seed come from torch's
    CPU generator."""

    def __init__(self, data, num_neighbors: Sequence[int], input_nodes: Optional[torch.Tensor] = None,
                 batch_size: int = 1, shuffle: bool = False, drop_last: bool = False, replace: bool = False,
                 directed: bool = True, **kwargs):
        if replace:
            raise NotImplementedError("sampling with replacement (replace=True) is not supported")
        if not directed:
            raise NotImplementedError("undirected sampling (directed=False) is not supported")
        if kwargs:
            raise NotImplementedError(f"unsupported NeighborLoader options: {sorted(kwargs)}")
        if int(batch_size) < 1:
            raise ValueError("batch_size must be >= 1")
        x, edge_index = data.x, data.edge_index
        if not (x.is_cuda and edge_index.is_cuda):
            raise RuntimeError("NeighborLoader runs on CUDA tensors only (no CPU fallback)")
        self.data, self.batch_size, self.shuffle, self.drop_last = data, int(batch_size), bool(shuffle), bool(drop_last)
        num_nodes = x.size(0)
        self.sampler = NeighborSampler(edge_index, num_nodes, num_neighbors)
        if input_nodes is None:
            input_nodes = torch.arange(num_nodes, device=x.device)
        elif input_nodes.dtype == torch.bool:
            input_nodes = torch.nonzero(input_nodes.to(x.device)).reshape(-1)
        self.input_nodes = input_nodes.to(device=x.device, dtype=torch.int64).reshape(-1)

    def __len__(self) -> int:
        n = self.input_nodes.numel()
        return n // self.batch_size if self.drop_last else math.ceil(n / self.batch_size)

    def __iter__(self):
        n = self.input_nodes.numel()
        order = torch.randperm(n).to(self.input_nodes.device) if self.shuffle else \
            torch.arange(n, device=self.input_nodes.device)
        for b in range(len(self)):
            input_id = order[b * self.batch_size:(b + 1) * self.batch_size]
            s = self.sampler.sample(self.input_nodes[input_id])
            d = self.data
            y, ts = getattr(d, "y", None), getattr(d, "time_steps", None)
            yield SimpleNamespace(x=d.x[s.n_id], y=None if y is None else y[s.n_id],
                                  time_steps=None if ts is None else ts[s.n_id], edge_index=s.edge_index, n_id=s.n_id,
                                  e_id=s.e_id, input_id=input_id, batch_size=s.batch_size,
                                  num_sampled_nodes=s.num_sampled_nodes, num_sampled_edges=s.num_sampled_edges)
