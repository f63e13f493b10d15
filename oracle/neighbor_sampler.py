"""CPU oracle of the neighbour sampler -- TEST INFRASTRUCTURE ONLY (and the host baseline of scripts/bench_sampler.py).

A pure-Python / numpy restatement of the contract in ``include/gnnfd_b200.h`` section (8), which is PyG's
``NeighborLoader`` (``src/data/dataloader.py:42-66``) with its defaults ``replace=False, directed=True`` and a
counter-based generator:

  * neighbours of v = its in-edges ``j -> v`` (duplicates and self-loops included), position p = the p-th in-edge of v in
    ``edge_index`` order (row v of the stable destination sort);
  * hop 1 expands the seeds, hop l exactly the nodes first discovered in hop l-1;
  * node v with in-degree d and fanout k: every position if ``k == -1`` or ``d <= k``, else Floyd's algorithm
    (``for i in 0..k-1: j = d-k+i; t = U_i(j); add j if t is chosen else t``), positions sorted ascending;
    ``U_i(j) = mulhi64(w, j+1)``, ``w = splitmix64(seed + 0x9E3779B97F4A7C15 * (2*(v*2^32 + i) + 1))`` mod 2^64;
  * ``n_id``: the seeds, then the nodes new in hop 1 in order of first appearance in hop 1's edge list, then hop 2, ...;
    edges by hop, then local destination, then position; ``edge_index`` rows = (local source, local destination);
    ``e_id`` = column in the input ``edge_index``.

PyG's own sampler draws from a different generator, so its exact samples cannot be matched; toward PyG the contract is
distributional (at most k, uniform without replacement, all neighbours when ``d <= k``).  Toward the CUDA sampler it is
bit-exact.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

__all__ = ["mix", "select_positions", "raw_csr", "neighbor_sample"]

_M64 = (1 << 64) - 1
_GOLDEN = 0x9E3779B97F4A7C15


def mix(z: int) -> int:
    """splitmix64 finaliser (``KeepMask::mix`` in ``csrc/gat_common.cuh``)."""
    z &= _M64
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & _M64
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & _M64
    z ^= z >> 31
    return z


def select_positions(seed: int, v: int, d: int, k: int):
    """The ascending positions (in ``0..d-1``) that node ``v`` of in-degree ``d`` keeps at fanout ``k``."""
    if k == -1 or d <= k:
        return list(range(d))
    chosen = []
    seen = set()
    for i in range(k):
        j = d - k + i
        w = mix(seed + _GOLDEN * (2 * ((v << 32) + i) + 1))
        t = (w * (j + 1)) >> 64
        c = j if t in seen else t
        seen.add(c)
        chosen.append(c)
    return sorted(chosen)


def raw_csr(edge_index, num_nodes: int):
    """Row pointers, sources and edge ids of the stable destination sort of the raw ``edge_index`` (no self-loop rewrite)."""
    ei = np.asarray(edge_index, dtype=np.int64)
    src, dst = ei[0], ei[1]
    order = np.argsort(dst, kind="stable")
    rowptr = np.zeros(num_nodes + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum(np.bincount(dst, minlength=num_nodes))
    return rowptr, src[order], order


def neighbor_sample(edge_index, num_nodes: int, seeds, num_neighbors, seed: int, csr=None):
    """One batch.  Returns ``SimpleNamespace(n_id, edge_index, e_id, batch_size, num_sampled_nodes, num_sampled_edges)``
    with numpy int64 arrays; ``csr`` = a precomputed ``raw_csr(edge_index, num_nodes)``."""
    rowptr, col, eid = csr if csr is not None else raw_csr(edge_index, num_nodes)
    seed &= _M64
    n_id = [int(s) for s in np.asarray(seeds, dtype=np.int64).reshape(-1)]
    local = {}
    for i, s in enumerate(n_id):
        if not 0 <= s < num_nodes:
            raise IndexError(f"seed {s} outside [0, {num_nodes})")
        if s in local:
            raise ValueError(f"duplicate seed {s}")
        local[s] = i
    for k in num_neighbors:
        if k < -1:
            raise ValueError(f"fanout {k} < -1")
    rows, cols, eids = [], [], []
    num_nodes_hop, num_edges_hop = [len(n_id)], []
    front = range(0, len(n_id))
    for k in num_neighbors:
        start, m0 = len(n_id), len(eids)
        for li in front:
            v = n_id[li]
            r0, d = int(rowptr[v]), int(rowptr[v + 1] - rowptr[v])
            for p in select_positions(seed, v, d, k):
                s = int(col[r0 + p])
                if s not in local:
                    local[s] = len(n_id)
                    n_id.append(s)
                rows.append(local[s])
                cols.append(li)
                eids.append(int(eid[r0 + p]))
        num_nodes_hop.append(len(n_id) - start)
        num_edges_hop.append(len(eids) - m0)
        front = range(start, len(n_id))
    return SimpleNamespace(n_id=np.asarray(n_id, dtype=np.int64),
                           edge_index=np.asarray([rows, cols], dtype=np.int64).reshape(2, -1),
                           e_id=np.asarray(eids, dtype=np.int64), batch_size=num_nodes_hop[0],
                           num_sampled_nodes=num_nodes_hop, num_sampled_edges=num_edges_hop)
