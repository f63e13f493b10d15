"""Multi-GPU partitioning of the GAT hot path on one 8xB200 NVSwitch box (one process per GPU).

Two seams, both from the dataset's structure (BASELINE.json north_star item 5):

* **time-step sharding** (`lpt_assign`, `snapshot_batches`): the 49 Elliptic time steps are disconnected
  subgraphs (`create_temporal_subgraph`, ``src/data/dataset.py:198-240`` keeps only intra-step edges), so
  snapshots are dealt to GPUs by longest-processing-time and each GPU runs its block-diagonal batch with
  **no data-path collective**;
* **destination-range partition** (`DstRangePlan`, `DstRangePartition`): for a scaled graph every GPU
  owns a contiguous range of destination rows chosen on the in-degree prefix sum so that each owns
  ~E'/G edges.  Forward: each GPU projects its own rows and the projected rows (+ source logits) are
  exchanged with one NCCL all-gather; softmax/aggregation are then local.  Backward: the partial dxw /
  da_src over all sources are reduce-scattered back to their owners; the small weight gradients are
  all-reduced.

Node ids are remapped to a *padded position space* ``pos(g) = owner(g) * P + (g - start[owner])`` with
``P = max rows per rank`` so that every rank contributes an equal-sized chunk to the collectives.
The plan (`DstRangePlan`) is pure index arithmetic and runs on any device; `DstRangePartition` executes it
with the CUDA library.
"""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch
import torch.distributed as dist


# ------------------------------------------------------------------------------------------------
# time-step sharding
# ------------------------------------------------------------------------------------------------
def lpt_assign(weights: Sequence[float], n_bins: int) -> List[List[int]]:
    """Longest-processing-time assignment of items (snapshots, cost = n_t + e_t) to ``n_bins`` GPUs."""
    order = sorted(range(len(weights)), key=lambda i: (-weights[i], i))
    loads = [0.0] * n_bins
    bins: List[List[int]] = [[] for _ in range(n_bins)]
    for i in order:
        b = min(range(n_bins), key=lambda k: (loads[k], k))
        bins[b].append(i)
        loads[b] += weights[i]
    return [sorted(b) for b in bins]


def snapshot_batches(x: torch.Tensor, edge_index: torch.Tensor, time_steps: torch.Tensor, rank: int, world: int):
    """Block-diagonal batch of the snapshots owned by ``rank``.

    Returns ``(x_local, edge_index_local, node_ids)``: the nodes of the owned time steps (ascending original
    id), the edges with both endpoints inside (original order), relabelled to the local numbering.  Because
    no edge crosses a time step this is exactly the union of the per-snapshot subgraphs
    (``create_temporal_subgraph`` semantics) and needs no communication.
    """
    steps = torch.unique(time_steps)
    n_t = torch.stack([(time_steps == t).sum() for t in steps]).tolist()
    e_t = torch.stack([(time_steps[edge_index[1]] == t).sum() for t in steps]).tolist()
    mine = lpt_assign([a + b for a, b in zip(n_t, e_t)], world)[rank]
    if x.is_cuda:
        # selection + relabelling + order-preserving edge compaction in libgnnfd_b200.so (gnnfd_subgraph_build)
        from .snapshot import select_steps
        node_ids, ei_local, _ = select_steps(time_steps, edge_index, [int(steps[i]) for i in mine])
        return x[node_ids], ei_local, node_ids
    # host-side planning on CPU tensors (gloo tests): same semantics with torch index ops
    own = torch.zeros(int(steps.max()) + 1, dtype=torch.bool, device=x.device)
    own[steps[torch.tensor(mine, dtype=torch.long, device=steps.device)]] = True
    nmask = own[time_steps]
    node_ids = torch.nonzero(nmask).reshape(-1)
    relabel = torch.full((x.size(0),), -1, dtype=torch.int64, device=x.device)
    relabel[node_ids] = torch.arange(node_ids.numel(), device=x.device)
    emask = nmask[edge_index[0]] & nmask[edge_index[1]]
    return x[node_ids], relabel[edge_index[:, emask]].contiguous(), node_ids


# ------------------------------------------------------------------------------------------------
# destination-range partition: the plan (index arithmetic only)
# ------------------------------------------------------------------------------------------------
@dataclass
class DstRangePlan:
    num_nodes: int
    world: int
    start: torch.Tensor        # [world+1] int64 row boundaries (global ids)
    rows_padded: int           # P

    @staticmethod
    def build(edge_index: torch.Tensor, num_nodes: int, world: int) -> "DstRangePlan":
        """Boundaries on the prefix sum of (in-degree without self-loops + 1) so each rank owns ~E'/world edges."""
        keep = edge_index[0] != edge_index[1]
        deg = torch.bincount(edge_index[1][keep], minlength=num_nodes) + 1
        csum = torch.cumsum(deg, 0)
        total = int(csum[-1]) if num_nodes > 0 else 0
        targets = torch.tensor([total * r / world for r in range(1, world)], dtype=csum.dtype, device=csum.device)
        cuts = torch.searchsorted(csum, targets, right=False) + 1 if world > 1 else targets.long()
        start = torch.cat([torch.zeros(1, dtype=torch.int64, device=csum.device), cuts.long().clamp(max=num_nodes),
                           torch.tensor([num_nodes], dtype=torch.int64, device=csum.device)])
        start = torch.cummax(start, 0).values
        rows = (start[1:] - start[:-1])
        return DstRangePlan(num_nodes, world, start.cpu(), int(rows.max()) if num_nodes > 0 else 0)

    def owner(self, ids: torch.Tensor) -> torch.Tensor:
        return torch.bucketize(ids, self.start[1:].to(ids.device), right=True)

    def to_pos(self, ids: torch.Tensor) -> torch.Tensor:
        """global node id -> padded position."""
        own = self.owner(ids)
        return own * self.rows_padded + (ids - self.start.to(ids.device)[own])

    def local_edges(self, edge_index: torch.Tensor, rank: int) -> torch.Tensor:
        """Edges whose destination is owned by ``rank`` (self-loops rewritten PyG-style), in padded positions.

        Order: the surviving original edges in their original order, then one self-loop per owned node --
        the same relative order as the reference's ``edge_index'`` restricted to these destinations, so the
        stable destination sort gives rows identical to the single-GPU CSR.
        """
        lo, hi = int(self.start[rank]), int(self.start[rank + 1])
        src, dst = edge_index[0], edge_index[1]
        m = (dst >= lo) & (dst < hi) & (src != dst)
        loops = torch.arange(lo, hi, dtype=edge_index.dtype, device=edge_index.device)
        s = torch.cat([src[m], loops])
        d = torch.cat([dst[m], loops])
        return torch.stack([self.to_pos(s), self.to_pos(d)]).contiguous()


# ------------------------------------------------------------------------------------------------
# destination-range partition: execution with the CUDA library + NCCL
# ------------------------------------------------------------------------------------------------
class DstRangePartition:
    def __init__(self, plan: DstRangePlan, rank: int, device):
        self.plan, self.rank, self.device = plan, rank, device
        self.world, self.rows_padded = plan.world, plan.rows_padded
        self.n_local = int(plan.start[rank + 1] - plan.start[rank])
        self.n_pos = plan.world * plan.rows_padded
        self.graph = None
        self.build_ms = 0.0
        self.local_ei: Optional[torch.Tensor] = None

    @classmethod
    def build(cls, edge_index: torch.Tensor, num_nodes: int, rank: int, world: int, device) -> "DstRangePartition":
        plan = DstRangePlan.build(edge_index, num_nodes, world)
        self = cls(plan, rank, device)
        self.local_ei = plan.local_edges(edge_index, rank)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.graph = self.build_graph(self.local_ei)
        torch.cuda.synchronize()
        self.build_ms = (time.perf_counter() - t0) * 1e3
        return self

    def build_graph(self, local_ei: torch.Tensor):
        """CSR over the padded position space, then the row view of this rank's destinations."""
        from .graph import GraphCSR, build_csr
        full = build_csr(local_ei, self.n_pos, add_self_loops=False, build_csc=True)
        lo = self.rank * self.rows_padded
        rowptr = full.rowptr[lo: lo + self.n_local + 1].contiguous()     # earlier rows are empty => starts at 0
        csc_row = (full.csc_row - lo).contiguous()                        # local destination row of each CSC entry
        g = GraphCSR(self.n_local, self.n_pos, full.n_edges, rowptr, full.col, full.perm, full.colptr, csc_row,
                     full.csc_eid)
        return g

    def layer_fwd_bwd(self, x_local, W, a_s, a_d, bias, d_out, H, C, xw_dtype, algo, marks=None, graph=None):
        """One GATConv layer forward + backward on this rank's destination rows.

        ``x_local`` is ``[rows_padded, K]`` (rows beyond ``n_local`` are padding).  Returns
        ``(out [n_local, C], (dW, datt_src, datt_dst, dbias))`` with the weight gradients already all-reduced.
        """
        from . import functional as Fn
        g = graph or self.graph
        P, D, dev = self.rows_padded, H * C, self.device
        lo = self.rank * P
        if marks: marks[0].record()
        # forward: project own rows straight into this rank's slice of the gathered buffers
        xw_full = torch.empty(self.n_pos, D, dtype=xw_dtype, device=dev)
        asrc_full = torch.empty(self.n_pos, H, dtype=torch.float32, device=dev)
        a_dst = torch.empty(P, H, dtype=torch.float32, device=dev)
        Fn.project_fwd(x_local, W, a_s, a_d, H, C, xw_dtype, algo, out=(xw_full[lo:lo + P], asrc_full[lo:lo + P], a_dst))
        if self.world > 1:
            dist.all_gather_into_tensor(xw_full, xw_full[lo:lo + P])
            dist.all_gather_into_tensor(asrc_full, asrc_full[lo:lo + P])
        if marks: marks[1].record()
        out, rowmax, rowsum = Fn.gat_fwd(g, xw_full, asrc_full, a_dst, bias, H, C, 0.2, False)
        if marks: marks[2].record()
        # backward: partials over every source position, reduce-scattered to the owners
        da_dst_pos = torch.zeros(self.n_pos, H, dtype=torch.float32, device=dev)
        dxw_part, dasrc_part, da_dst = Fn.gat_bwd(g, xw_full, asrc_full, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C, 0.2,
                                                  False, da_dst_full=da_dst_pos, da_dst_view=(lo, self.n_local))
        if self.world > 1:
            dxw = torch.empty(P, D, dtype=torch.float32, device=dev)
            da_src = torch.empty(P, H, dtype=torch.float32, device=dev)
            dist.reduce_scatter_tensor(dxw, dxw_part)
            dist.reduce_scatter_tensor(da_src, dasrc_part)
        else:
            dxw, da_src = dxw_part, dasrc_part
        if marks: marks[3].record()
        n = self.n_local
        grads = Fn.project_bwd(x_local[:n], W, dxw[:n], xw_full[lo:lo + n], da_src[:n], da_dst, d_out, H, C, C, False, algo)
        dW, datt_s, datt_d, dbias, _ = grads
        if self.world > 1:
            flat = torch.cat([dW.reshape(-1), datt_s, datt_d, dbias])
            dist.all_reduce(flat)
            k = dW.numel()
            dW, datt_s, datt_d, dbias = flat[:k].view_as(dW), flat[k:k + D], flat[k + D:k + 2 * D], flat[k + 2 * D:]
        if marks: marks[4].record()
        return out, (dW, datt_s, datt_d, dbias)

    def e2e(self, args, conv, x_local, N, E_total, K, dev):
        """End-to-end with HOST buffers on every rank: per step H2D of this rank's feature rows and of its
        destination-range edge list, CSR/CSC rebuild, forward + backward with the collectives, D2H of the
        (all-reduced) weight gradients."""
        H, C = conv.heads, conv.out_channels
        x_host = torch.empty(x_local.shape, dtype=x_local.dtype, pin_memory=True).copy_(x_local)
        ei_host = torch.empty(self.local_ei.shape, dtype=self.local_ei.dtype, pin_memory=True).copy_(self.local_ei)
        W = conv.lin_src.weight.detach()
        a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
        bias = conv.bias.detach()
        d_out = torch.full((self.n_local, C), 1.0 / N, device=dev)
        steps = max(1, min(args.steps, args.e2e_steps))
        self.graph = None
        torch.cuda.empty_cache()

        def one():
            xd = x_host.to(dev, non_blocking=True)
            ed = ei_host.to(dev, non_blocking=True)
            g = self.build_graph(ed)
            out, grads = self.layer_fwd_bwd(xd, W, a_s, a_d, bias, d_out, H, C, conv.feature_dtype, args.algo, graph=g)
            return [t.cpu() for t in grads] + [out[:1].cpu()]

        one()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = one()
        torch.cuda.synchronize()
        dist.barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        h2d = x_host.numel() * x_host.element_size() + ei_host.numel() * ei_host.element_size()
        d2h = sum(t.numel() * t.element_size() for t in res)
        return {"value": E_total / dt, "unit": "edges/s", "h2d_bytes_per_step": h2d * self.world,
                "d2h_bytes_per_step": d2h * self.world, "steps": steps, "ms_per_step": dt * 1e3,
                "includes": "per rank: H2D of own x rows + own edge list, CSR/CSC rebuild, fwd+bwd with all-gather/"
                            "reduce-scatter/all-reduce, D2H of grads"}


class ReplicatedInputPartition(DstRangePartition):
    """Destination-range partition without the two feature-sized collectives (SURVEY.md 7.4 #1, variant (c)).

    * forward: the layer INPUT ``x [N,K]`` (664 B/row instead of 2 KB/row, and static for layer 1) is resident on
      every GPU and projected redundantly -- writing xw locally at HBM speed is ~8x faster than receiving it
      over NVLink -- so the forward needs no communication at all;
    * backward: instead of reduce-scattering ``dxw [N,512]`` partials (41 GB on the 200M-edge graph) the
      per-edge gradients (alpha_used, dz: 64 B/edge), which ``gat_bwd_dst`` already emits grouped by source
      owner (source-major order), are sent to the owner of each source with one all-to-all, ``dOut [N,64]`` is
      all-gathered, and every GPU runs the src-major pass for ITS OWN source rows over all of their out-edges.
      ``dxw`` is then complete where it is needed: no reduce-scatter, and the projection backward is local.
    Per step and GPU this moves ~(E'/G)*64 B + N*256 B over NVLink instead of ~2*N*2 KB.
    """

    @classmethod
    def build(cls, edge_index, num_nodes, rank, world, device):
        plan = DstRangePlan.build(edge_index, num_nodes, world)
        self = cls(plan, rank, device)
        self.local_ei = plan.local_edges(edge_index, rank)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.graph = self.build_graph(self.local_ei)
        self.rgraph = self.build_exchange(self.graph)
        torch.cuda.synchronize()
        self.build_ms = (time.perf_counter() - t0) * 1e3
        return self

    def build_exchange(self, g):
        """Receiver-side CSC: for every source row this rank owns, its out-edges on ALL ranks."""
        from .graph import GraphCSR, build_csr
        P, G, dev = self.rows_padded, self.world, self.device
        colptr = g.colptr.long()
        bounds = colptr[torch.arange(0, G + 1, device=dev) * P]
        send = (bounds[1:] - bounds[:-1]).contiguous()
        recv = torch.empty_like(send)
        if G > 1:
            dist.all_to_all_single(recv, send)
        else:
            recv.copy_(send)
        self.send_splits, self.recv_splits = send.tolist(), recv.tolist()
        M = int(sum(self.recv_splits))
        src_pos = torch.repeat_interleave(torch.arange(self.n_pos, device=dev, dtype=torch.int32),
                                          (colptr[1:] - colptr[:-1]))
        dst_pos = g.csc_row + self.rank * P
        meta_send = torch.stack([src_pos, dst_pos.to(torch.int32)], dim=1).contiguous()
        meta_recv = torch.empty(M, 2, dtype=torch.int32, device=dev)
        if G > 1:
            dist.all_to_all_single(meta_recv, meta_send, self.recv_splits, self.send_splits)
        else:
            meta_recv.copy_(meta_send)
        # stable sort of the received entries by (local) source row = CSR build of a surrogate edge list
        fake = torch.stack([meta_recv[:, 1].long(), meta_recv[:, 0].long() - self.rank * P]).contiguous()
        fg = build_csr(fake, self.n_pos, add_self_loops=False, build_csc=False)
        rg = GraphCSR(self.n_pos, P, M, fg.rowptr, fg.col, fg.perm, fg.rowptr[:P + 1].contiguous(), fg.col, fg.perm)
        rg.c.edge_grads_indirect = 1
        self.n_recv = M
        return rg

    def layer_fwd_bwd(self, x_full, W, a_s, a_d, bias, d_out, H, C, xw_dtype, algo, marks=None, graph=None, rgraph=None):
        """``x_full`` is the replicated input in padded position space ``[world*rows_padded, K]``."""
        from . import functional as Fn
        g, rg = graph or self.graph, rgraph or self.rgraph
        P, D, dev, n = self.rows_padded, H * C, self.device, self.n_local
        lo = self.rank * P
        if marks: marks[0].record()
        xw_full, asrc_full, adst_full = Fn.project_fwd(x_full, W, a_s, a_d, H, C, xw_dtype, algo)
        a_dst = adst_full[lo:lo + P]
        if marks: marks[1].record()
        out, rowmax, rowsum = Fn.gat_fwd(g, xw_full, asrc_full, a_dst, bias, H, C, 0.2, False)
        if marks: marks[2].record()
        # backward
        if self.world > 1:
            dO_pad = torch.zeros(P, d_out.size(1), dtype=torch.float32, device=dev)
            dO_pad[:n] = d_out
            dO_full = torch.empty(self.n_pos, d_out.size(1), dtype=torch.float32, device=dev)
            # asynchronous: the gather of dOut rides NVLink while the dst-major pass runs
            ag_work = dist.all_gather_into_tensor(dO_full, dO_pad, async_op=True)
        else:
            dO_full = torch.zeros(self.n_pos, d_out.size(1), dtype=torch.float32, device=dev)
            dO_full[lo:lo + n] = d_out
        alpha_used, dz, da_dst = Fn.gat_bwd_dst(g, xw_full, asrc_full, a_dst, rowmax, rowsum, d_out, H, C, 0.2, False)
        if self.world > 1:
            # alpha_used / dz are the halves of one interleaved [E',2H] buffer: one all-to-all of 64-byte rows
            eg = alpha_used._base if alpha_used._base is not None else torch.cat([alpha_used, dz], 1)
            r_eg = torch.empty(self.n_recv, 2 * H, dtype=torch.float32, device=dev)
            dist.all_to_all_single(r_eg, eg, self.recv_splits, self.send_splits)
            r_alpha, r_dz = r_eg[:, :H], r_eg[:, H:]
            ag_work.wait()
        else:
            r_alpha, r_dz = alpha_used, dz
        da_dst_pad = torch.zeros(P, H, dtype=torch.float32, device=dev)
        da_dst_pad[:n] = da_dst
        dxw, da_src = Fn.gat_bwd_src(rg, r_alpha, r_dz, dO_full, a_s, a_d, da_dst_pad, H, C, False)
        if marks: marks[3].record()
        grads = Fn.project_bwd(x_full[lo:lo + n], W, dxw[:n], xw_full[lo:lo + n], da_src[:n], da_dst, d_out, H, C, C, False,
                               algo)
        dW, datt_s, datt_d, dbias, _ = grads
        if self.world > 1:
            flat = torch.cat([dW.reshape(-1), datt_s, datt_d, dbias])
            dist.all_reduce(flat)
            k = dW.numel()
            dW, datt_s, datt_d, dbias = flat[:k].view_as(dW), flat[k:k + D], flat[k + D:k + 2 * D], flat[k + 2 * D:]
        if marks: marks[4].record()
        return out, (dW, datt_s, datt_d, dbias)

    def e2e(self, args, conv, x_full, N, E_total, K, dev):
        """End-to-end with HOST buffers: per step every rank copies the (replicated) input features and its own
        destination-range edge list host->device, rebuilds CSR/CSC and the receive-side index, runs forward +
        backward with the collectives, and reads the all-reduced weight gradients back."""
        H, C = conv.heads, conv.out_channels
        x_host = torch.empty(x_full.shape, dtype=x_full.dtype, pin_memory=True).copy_(x_full)
        ei_host = torch.empty(self.local_ei.shape, dtype=self.local_ei.dtype, pin_memory=True).copy_(self.local_ei)
        W = conv.lin_src.weight.detach()
        a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
        bias = conv.bias.detach()
        d_out = torch.full((self.n_local, C), 1.0 / N, device=dev)
        steps = max(1, min(args.steps, args.e2e_steps))
        self.graph = self.rgraph = None
        torch.cuda.empty_cache()

        copy_stream = torch.cuda.Stream(device=dev)

        def one():
            main = torch.cuda.current_stream()
            ed = ei_host.to(dev, non_blocking=True)
            copy_stream.wait_stream(main)
            with torch.cuda.stream(copy_stream):       # feature copy overlaps the index builds below
                xd = x_host.to(dev, non_blocking=True)
            g = self.build_graph(ed)
            rg = self.build_exchange(g)
            main.wait_stream(copy_stream)
            xd.record_stream(main)
            out, grads = self.layer_fwd_bwd(xd, W, a_s, a_d, bias, d_out, H, C, conv.feature_dtype, args.algo, graph=g,
                                            rgraph=rg)
            return [t.cpu() for t in grads] + [out[:1].cpu()]

        one()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = one()
        torch.cuda.synchronize()
        dist.barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        h2d = x_host.numel() * x_host.element_size() + ei_host.numel() * ei_host.element_size()
        d2h = sum(t.numel() * t.element_size() for t in res)
        return {"value": E_total / dt, "unit": "edges/s", "h2d_bytes_per_step": h2d * self.world,
                "d2h_bytes_per_step": d2h * self.world, "steps": steps, "ms_per_step": dt * 1e3,
                "includes": "per rank: H2D of x + own edge list, CSR/CSC + exchange-index rebuild, fwd+bwd with "
                            "all-to-all/all-gather/all-reduce, D2H of grads"}


class PeerExchange:
    """Symmetric (peer-accessible) buffers of the input-space exchange and the addresses the kernels need
    (include/gnnfd_b200.h section 7).  Allocation, address exchange and the cross-GPU barrier come from torch symmetric
    memory; the data itself is moved by the library's kernels (NVLink stores / loads, or NVSwitch multicast)."""

    def __init__(self, n_pos, device, mode="auto", H=8):
        import torch.distributed._symmetric_memory as symm
        from . import _abi
        grp = dist.group.WORLD
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        if self.world > _abi.MAX_PEERS:
            raise RuntimeError(f"peer exchange supports up to {_abi.MAX_PEERS} ranks")
        self.a_src = symm.empty((n_pos, H), dtype=torch.float32, device=device)       # all-gathered source logits
        self.da_part = symm.empty((n_pos, H), dtype=torch.float32, device=device)     # this rank's partial da_src
        self.xmax = symm.empty((16,), dtype=torch.float32, device=device)
        self.handles = [symm.rendezvous(t, grp) for t in (self.a_src, self.da_part, self.xmax)]
        has_mc = all(int(getattr(h, "multicast_ptr", 0) or 0) != 0 for h in self.handles[:2])
        if mode == "multicast" and not has_mc:
            raise RuntimeError("GNNFD_EXCHANGE=multicast: the symmetric allocation has no multicast mapping on this box")
        self.mode = "multicast" if (mode in ("auto", "multicast") and has_mc) else "peer"
        self.a_src_peers, self.da_peers, self.xmax_peers = (self._peers(h) for h in self.handles)
        self.da_part.zero_()
        self.xmax.zero_()
        self.side = torch.cuda.Stream(device=device)          # the da_src exchange runs here, under the dW GEMM
        self.barrier()

    def _peers(self, h):
        from . import _abi
        p = _abi.Peers()
        p.n_peers, p.rank = self.world, self.rank
        for r, ptr in enumerate(h.buffer_ptrs):
            p.ptr[r] = int(ptr)
        p.multicast = int(getattr(h, "multicast_ptr", 0) or 0) or None
        return p

    def barrier(self):
        """Cross-GPU barrier on the current stream (signal pads of the symmetric allocation): kernels enqueued before it on
        every rank have completed -- their peer stores included -- before anything enqueued after it starts."""
        self.handles[0].barrier()


def exchange_logits(part, px, x_own, W, a_s, a_d, prep, xmax):
    """The logits of this rank's rows ``x_own`` and their exchange, for one input-space layer on a destination-range
    partition.  Returns ``(a_src of every position [n_pos,H], a_dst of the own rows)`` and leaves max|input| over all ranks in
    ``xmax`` (the fp16-pair scale ``in_prepare`` needs).

    With a ``PeerExchange`` the logits kernel stores its rows into ``px.a_src`` ON EVERY RANK (NVLink stores / one multicast
    store), then a barrier and the max-reduce of ``xmax``; otherwise the own rows, zero-padded to ``rows_padded``, are
    all-gathered with NCCL."""
    from . import functional as Fn
    lo = part.rank * part.rows_padded
    if px is not None:
        px.xmax.zero_()
        a_dst = Fn.in_logits_bcast(x_own, W, a_s, a_d, prep, px.xmax, px.a_src_peers, lo, px.mode == "multicast")
        px.barrier()
        Fn.peer_reduce(px.xmax_peers, 0, 4, xmax, op="max")
        return px.a_src, a_dst
    xmax.zero_()
    a_src_own, a_dst = Fn.in_logits(x_own, W, a_s, a_d, prep, xmax)
    if part.world == 1:
        return a_src_own, a_dst
    if a_src_own.size(0) < part.rows_padded:
        a_pad = torch.zeros(part.rows_padded, a_src_own.size(1), dtype=torch.float32, device=a_src_own.device)
        a_pad[:a_src_own.size(0)] = a_src_own
        a_src_own = a_pad
    a_src_full = torch.empty(part.n_pos, a_src_own.size(1), dtype=torch.float32, device=a_src_own.device)
    dist.all_gather_into_tensor(a_src_full, a_src_own)
    dist.all_reduce(xmax, op=dist.ReduceOp.MAX)
    return a_src_full, a_dst


class InputSpacePartition(DstRangePartition):
    """Destination-range partition of the FIRST layer in the input-space formulation (csrc/in_common.cuh).

    The layer input x (static for layer 1, ``K*4`` bytes per row) is resident on every GPU in padded position space;
    each GPU aggregates INPUT rows for its destination range, so nothing is projected redundantly and no per-edge
    quantity crosses NVLink.  Per step the ranks exchange only per-node logit vectors:
      forward   all-gather of ``a_src [N,H]`` (32 B per node) and a max-reduce of one scalar (the fp16-pair scale);
      backward  reduce-scatter of the partial ``da_src [N,H]`` and the all-reduce of the weight gradients.
    ~64 B per node over NVLink instead of ~2 x 2 KB (all-gather of projected features) or 64 B per EDGE plus 256 B per node
    (the replicated-input variant above).
    """

    @classmethod
    def build(cls, edge_index, num_nodes, rank, world, device):
        plan = DstRangePlan.build(edge_index, num_nodes, world)
        self = cls(plan, rank, device)
        self.local_ei = plan.local_edges(edge_index, rank)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.graph = self.build_graph(self.local_ei)
        torch.cuda.synchronize()
        self.build_ms = (time.perf_counter() - t0) * 1e3
        return self

    def prepare_buffers(self, K):
        from . import functional as Fn
        import os
        self.prep = Fn._aligned_u8(Fn.in_sizes(self.n_local, K)[0], self.device)
        self.xmax = torch.zeros(16, dtype=torch.float32, device=self.device)
        self.redundant_logits = os.environ.get("GNNFD_LOGITS_REDUNDANT", "0") == "1"
        # exchange over peer memory (default when torch symmetric memory is available): "peer" = stores / loads per peer,
        # "multicast" = multimem.st / multimem.ld_reduce through the NVSwitch, "nccl" = the plain collectives
        mode = os.environ.get("GNNFD_EXCHANGE", "auto")
        self.px = None
        if self.world > 1 and mode != "nccl" and not self.redundant_logits:
            try:
                self.px = PeerExchange(self.n_pos, self.device, mode)
            except Exception as ex:               # no symmetric memory on this box: NCCL collectives
                if mode != "auto":
                    raise
                self.px_error = f"{type(ex).__name__}: {ex}"
        self.exchange = self.px.mode if self.px is not None else ("nccl" if self.world > 1 else "none")

    def layer_fwd_bwd(self, x_full, W, a_s, a_d, bias, d_out, H, C, xw_dtype=None, algo=None, marks=None, graph=None):
        """``x_full``: the replicated input in padded position space ``[world*rows_padded, K]`` with 16-byte aligned,
        zero-padded rows (``functional.in_pad_x`` layout).  Returns ``(out [n_local, C], (dW, datt_src, datt_dst, dbias))``
        with the weight gradients all-reduced."""
        from . import functional as Fn
        g = graph or self.graph
        P, dev, n, K = self.rows_padded, self.device, self.n_local, x_full.size(1)
        lo = self.rank * P
        if getattr(self, "prep", None) is None:
            self.prepare_buffers(K)
        prep, xmax, px = self.prep, self.xmax, self.px
        if marks: marks[0].record()
        # forward: logits of the own rows, gathered from every rank; softmax / aggregation / output GEMM are local
        x_own = x_full[lo:lo + P]
        if self.world > 1 and self.redundant_logits:
            # every rank holds all of x: 32 B of logits per node can also be recomputed locally instead of gathered
            xmax.zero_()
            a_src_full, a_dst_full = Fn.in_logits(x_full, W, a_s, a_d, prep, xmax)
            a_dst_own = a_dst_full[lo:lo + P]
        else:
            a_src_full, a_dst_own = exchange_logits(self, px, x_own, W, a_s, a_d, prep, xmax)
        Fn.in_prepare(W, K, xmax, prep)
        if marks: marks[1].record()
        zimg, att = Fn.in_fwd(g, x_full, a_src_full, a_dst_own, 0.2, prep)
        if marks: marks[2].record()
        out = Fn.in_out(zimg, n, K, prep, bias)
        if marks: marks[3].record()
        # backward: edge pass is local; the partial da_src over ALL source positions is reduce-scattered to the owners
        dz, da_dst = Fn.in_bwd_edges(g, x_full, att, d_out, prep, 0.2)
        if marks: marks[4].record()
        if px is not None:
            # the partial stays in this rank's symmetric buffer; every owner pulls (or switch-reduces) its own row range.
            # The barrier + reduction run on a side stream UNDER the tensor-core part of the weight gradient (dO^T Z),
            # which does not need da_src.
            Fn.in_dasrc(g, dz, out=px.da_part)
            if marks: marks[5].record()
            da_src = torch.empty(P, H, dtype=torch.float32, device=dev)
            main = torch.cuda.current_stream()
            px.side.wait_stream(main)
            with torch.cuda.stream(px.side):
                px.barrier()
                Fn.peer_reduce(px.da_peers, lo * H, P * H, da_src, op="sum", use_multicast=px.mode == "multicast")
            finish = Fn.in_bwd_params_split(zimg, d_out, x_own[:n], W, a_s, a_d, prep)
            main.wait_stream(px.side)
            dW, datt_s, datt_d, dbias = finish(da_src[:n], da_dst)
        else:
            da_src_part = Fn.in_dasrc(g, dz)
            if self.world > 1:
                da_src = torch.empty(P, H, dtype=torch.float32, device=dev)
                dist.reduce_scatter_tensor(da_src, da_src_part)
            else:
                da_src = da_src_part
            if marks: marks[5].record()
            dW, datt_s, datt_d, dbias = Fn.in_bwd_params(zimg, d_out, x_own[:n], W, a_s, a_d, da_src[:n], da_dst, prep)
        if self.world > 1:
            D = H * C
            flat = torch.cat([dW.reshape(-1), datt_s, datt_d, dbias])
            dist.all_reduce(flat)          # also the step-end rendezvous that keeps a fast rank out of the next step's buffers
            k = dW.numel()
            dW, datt_s, datt_d, dbias = flat[:k].view_as(dW), flat[k:k + D], flat[k + D:k + 2 * D], flat[k + 2 * D:]
        if marks: marks[6].record()
        return out, (dW, datt_s, datt_d, dbias)

    def e2e(self, args, conv, x_full, N, E_total, K, dev):
        """End-to-end with HOST buffers: per step every rank copies ITS OWN rows of the input and its destination-range
        edge list host->device, the input rows are all-gathered over NVLink (instead of every rank pulling the whole
        input through PCIe), CSR/CSC are rebuilt, forward + backward run with the collectives, and the all-reduced weight
        gradients are read back."""
        from . import functional as Fn
        H, C = conv.heads, conv.out_channels
        P, lo = self.rows_padded, self.rank * self.rows_padded
        ld = x_full.stride(0)
        rows = x_full.as_strided((self.n_pos, ld), (ld, 1))          # the whole padded rows (pad columns included)
        x_own_host = torch.empty((P, ld), dtype=x_full.dtype, pin_memory=True).copy_(rows[lo:lo + P])
        ei_host = torch.empty(self.local_ei.shape, dtype=self.local_ei.dtype, pin_memory=True).copy_(self.local_ei)
        del rows
        W = conv.lin_src.weight.detach()
        a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
        bias = conv.bias.detach()
        d_out = torch.full((self.n_local, C), 1.0 / N, device=dev)
        steps = max(1, min(args.steps, args.e2e_steps))
        self.graph = None
        del x_full
        torch.cuda.empty_cache()
        copy_stream = torch.cuda.Stream(device=dev)

        def one():
            main = torch.cuda.current_stream()
            ed = ei_host.to(dev, non_blocking=True)
            xf = torch.empty(self.n_pos, ld, dtype=torch.float32, device=dev)
            copy_stream.wait_stream(main)
            with torch.cuda.stream(copy_stream):       # feature copy AND its all-gather over NVLink overlap the index build
                xo = x_own_host.to(dev, non_blocking=True)
                if self.world > 1:
                    dist.all_gather_into_tensor(xf, xo)
                else:
                    xf.copy_(xo)
            g = self.build_graph(ed)
            main.wait_stream(copy_stream)
            xo.record_stream(main)
            xf.record_stream(copy_stream)
            out, grads = self.layer_fwd_bwd(xf[:, :K], W, a_s, a_d, bias, d_out, H, C, graph=g)
            return [t.cpu() for t in grads] + [out[:1].cpu()]

        one()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = one()
        torch.cuda.synchronize()
        dist.barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        h2d = x_own_host.numel() * x_own_host.element_size() + ei_host.numel() * ei_host.element_size()
        d2h = sum(t.numel() * t.element_size() for t in res)
        return {"value": E_total / dt, "unit": "edges/s", "h2d_bytes_per_step": h2d * self.world,
                "d2h_bytes_per_step": d2h * self.world, "steps": steps, "ms_per_step": dt * 1e3,
                "includes": "per rank: H2D of own x rows + own edge list, all-gather of x over NVLink (both under the CSR/CSC "
                            "rebuild), fwd+bwd with the [N,H] logit exchange (" + str(getattr(self, "exchange", "nccl")) + "), "
                            "all-reduce of grads, D2H of grads"}


def symmetric_buffer(shape, device):
    """A zero-filled fp32 symmetric (peer-accessible) allocation: ``(this rank's tensor, _abi.Peers with its address on every
    rank, the rendezvous handle)``.  The handle owns the mapping: keep it as long as the peers are used."""
    import torch.distributed._symmetric_memory as symm
    from . import _abi
    t = symm.empty(shape, dtype=torch.float32, device=device)
    h = symm.rendezvous(t, dist.group.WORLD)
    p = _abi.Peers()
    p.n_peers, p.rank = dist.get_world_size(), dist.get_rank()
    for r, ptr in enumerate(h.buffer_ptrs):
        p.ptr[r] = int(ptr)
    p.multicast = int(getattr(h, "multicast_ptr", 0) or 0) or None
    t.zero_()
    return t, p, h


class InputSpaceModelPartition(DstRangePartition):
    """Inference of a whole ``GAT`` / ``TemporalGNN`` (eval mode) on a destination-range partition, every layer in the
    input-space formulation (csrc/in_common.cuh) -- the cross-GPU form of ``model.eval()`` with ``gemm_algo=GEMM_INPUT`` on
    every layer.

    The model input ``x`` is replicated in padded position space; the hidden state ``h [n_pos, 64]`` lives in two buffers
    that every rank holds whole.  Per layer each rank
      1. computes the logits of its own rows and stores ``a_src`` into every rank's buffer (``in_logits_bcast``), then a
         barrier and the max-reduce of ``max|input|`` (the fp16-pair scale);
      2. aggregates the layer input over its destination rows (``in_fwd``, local);
      3. runs the output GEMM with BatchNorm (running statistics), ReLU and the residual in its epilogue and stores each
         finished row into the next hidden buffer on every rank (``in_out_bcast``), then a barrier.
    Per layer and rank ~``N * (64 + 8) * 4`` bytes cross NVLink (each rank sends its rows to every other rank) and nothing is
    projected twice.  The head runs on the own rows.  ``GNNFD_EXCHANGE=nccl``, or no symmetric memory, uses ``in_logits`` /
    ``in_out`` and NCCL all-gathers instead, with bit-identical results.
    """

    H, HIDDEN = 8, 64

    @staticmethod
    def check_model(model, training=False):
        """Refuse what this path does not compute, before anything is launched.  ``training``: checked for
        ``InputSpaceModelTrainStep`` (train mode required) instead of ``forward`` (eval mode required)."""
        from . import functional as Fn
        from .models import GAT, TemporalGNN
        if not isinstance(model, (GAT, TemporalGNN)):
            raise TypeError(f"InputSpaceModelPartition runs GAT or TemporalGNN, not {type(model).__name__}")
        if model.training and not training:
            raise RuntimeError("InputSpaceModelPartition.forward is inference only: call model.eval() first "
                               "(InputSpaceModelTrainStep trains across GPUs)")
        if training and not model.training:
            raise RuntimeError("InputSpaceModelTrainStep trains the model: call model.train() first "
                               "(InputSpaceModelPartition.forward scores it)")
        if model.hidden_channels != InputSpaceModelPartition.HIDDEN:
            raise NotImplementedError(f"InputSpaceModelPartition is built for hidden_channels=64, got {model.hidden_channels}")
        for i, conv in enumerate(model.gat_layers):
            if conv.heads != InputSpaceModelPartition.H:
                raise NotImplementedError(f"InputSpaceModelPartition is built for 8 heads, layer {i} has {conv.heads}")
            if not conv.add_self_loops:
                raise NotImplementedError("InputSpaceModelPartition adds self-loops (local_edges): layer "
                                          f"{i} has add_self_loops=False")
            if not Fn.in_supported(conv.in_channels, conv.heads, conv.out_channels, conv.concat):
                raise NotImplementedError(f"layer {i}: the input-space formulation needs in_channels <= 192, concat=False "
                                          f"(got in_channels={conv.in_channels}, concat={conv.concat})")

    def _setup_exchange(self):
        self.px, self.hidden, self.hidden_peers, self._handles, self.exchange = self.hidden_buffers(2)

    def hidden_buffers(self, count):
        """``count`` ``[n_pos, 64]`` buffers every rank holds whole, and the exchange that fills them:
        ``(PeerExchange or None, tensors, peer tables or None, rendezvous handles, exchange name)``.  Symmetric memory unless
        ``GNNFD_EXCHANGE=nccl`` or the box has none (then zero-filled plain tensors for the NCCL collectives)."""
        import os
        mode = os.environ.get("GNNFD_EXCHANGE", "auto")
        shape = (self.n_pos, self.HIDDEN)
        px = None
        if self.world > 1 and mode != "nccl":
            try:
                px_try = PeerExchange(self.n_pos, self.device, mode, self.H)
                bufs = [symmetric_buffer(shape, self.device) for _ in range(count)]
                px = px_try
            except Exception as ex:               # no symmetric memory on this box: NCCL collectives
                if mode != "auto":
                    raise
                self.px_error = f"{type(ex).__name__}: {ex}"
        exchange = px.mode if px is not None else ("nccl" if self.world > 1 else "none")
        if px is not None:
            return px, [b[0] for b in bufs], [b[1] for b in bufs], [b[2] for b in bufs], exchange
        return None, [torch.zeros(shape, dtype=torch.float32, device=self.device) for _ in range(count)], None, [], exchange

    @torch.no_grad()
    def forward(self, model, x_full, marks=None):
        """``x_full``: the model input replicated in padded position space, ``[world*rows_padded, in_channels]`` with 16-byte
        aligned zero-padded rows (``functional.in_pad_x`` layout).  ``marks``: optional per-layer lists of 4 CUDA events
        (start, logits + exchange done, aggregation done, output GEMM + broadcast done).

        Returns ``(logits, (lo, hi))`` for a GAT and ``((logits, hidden), (lo, hi))`` for a TemporalGNN (zero initial state):
        the rows of the global nodes ``lo .. hi-1`` this rank owns."""
        from . import _abi, fused
        from . import functional as Fn
        from .models import TemporalGNN
        from .nn import fold_batch_norm
        self.check_model(model)
        if (not x_full.is_cuda or x_full.dtype != torch.float32 or x_full.dim() != 2
                or tuple(x_full.shape) != (self.n_pos, model.in_channels)):
            raise ValueError(f"x_full must be float32 CUDA [{self.n_pos},{model.in_channels}] in padded position space, "
                             f"got {x_full.dtype} {tuple(x_full.shape)} on {x_full.device}")
        if getattr(self, "hidden", None) is None:
            self._setup_exchange()
        P, n, dev, px = self.rows_padded, self.n_local, self.device, self.px
        lo = self.rank * P
        h_in = x_full
        for i, conv in enumerate(model.gat_layers):
            m = marks[i] if marks else None
            if m: m[0].record()
            K = h_in.size(1)
            x_own = h_in[lo:lo + n]
            W = conv.lin_src.weight.contiguous()
            a_s, a_d = conv.att_src.reshape(-1).contiguous(), conv.att_dst.reshape(-1).contiguous()
            prep = Fn._aligned_u8(Fn.in_sizes(n, K)[0], dev)
            xmax = torch.zeros(16, dtype=torch.float32, device=dev)
            a_src_full, a_dst = exchange_logits(self, px, x_own, W, a_s, a_d, prep, xmax)
            Fn.in_prepare(W, K, xmax, prep)
            if m: m[1].record()
            zimg, att = Fn.in_fwd(self.graph, h_in, a_src_full, a_dst, conv.negative_slope, prep)
            if m: m[2].record()
            bn = model.batch_norms[i] if model.use_batch_norm else None
            scale, shift = fold_batch_norm(bn)
            res = x_own.contiguous() if (model.residual and K == conv.out_channels) else None
            h_out = self.hidden[i % 2]
            if px is not None:
                Fn.in_out_bcast(zimg, n, K, prep, conv.bias, self.hidden_peers[i % 2], lo,
                                px.mode == "multicast" and self.hidden_peers[i % 2].multicast is not None, _abi.ACT_RELU,
                                scale, shift, res)
                px.barrier()       # every rank's rows have landed, and nobody reads the previous input any more
            else:
                Fn.in_out(zimg, n, K, prep, conv.bias, _abi.ACT_RELU, scale, shift, res, out=h_out[lo:lo + n])
                if self.world > 1:
                    dist.all_gather_into_tensor(h_out, h_out[lo:lo + P])
            if m: m[3].record()
            del zimg, att          # the next layer's image and attention reuse their memory (Z of K = 166: 5.25 KB per row)
            h_in = h_out
        h_own = h_in[lo:lo + n]
        if isinstance(model, TemporalGNN):
            return fused.gru_head(h_own, model.gru, model.out), (int(self.plan.start[self.rank]), int(self.plan.start[self.rank + 1]))
        return model.out(h_own), (int(self.plan.start[self.rank]), int(self.plan.start[self.rank + 1]))


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return x ^ (x >> 31)


class _RankLayer(torch.autograd.Function):
    """One GATConv layer in the input-space formulation on this rank's destination rows.

    forward ``(x_own, W, att_src, att_dst, bias)`` -> ``z [n_local, 64]`` (no activation); ``x_full``, the layer input of every
    position, is read as data.  ``x_own`` (its own rows) is the differentiable input: backward returns ``d x_own`` = the sum
    over ranks of every rank's ``dx`` partial over all ``n_pos`` source positions, reduced to the owner -- each partial is
    written by the dx GEMM straight into this rank's symmetric buffer and pulled by the owners (``gnnfd_peer_reduce``), or
    reduce-scattered with NCCL."""

    @staticmethod
    def forward(ctx, x_own, W, att_src, att_dst, bias, step, x_full, slope, p_drop, seed, marks):
        from . import functional as Fn
        part, px = step.part, step.px
        n, K, dev = part.n_local, x_full.size(1), x_full.device
        W = W.contiguous()
        a_s, a_d = att_src.reshape(-1).contiguous(), att_dst.reshape(-1).contiguous()
        if marks: marks[0].record()
        prep = Fn._aligned_u8(Fn.in_sizes(n, K)[0], dev)
        xmax = torch.zeros(16, dtype=torch.float32, device=dev)
        a_src_full, a_dst = exchange_logits(part, px, x_own, W, a_s, a_d, prep, xmax)
        Fn.in_prepare(W, K, xmax, prep)
        if marks: marks[1].record()
        zimg, att = Fn.in_fwd(part.graph, x_full, a_src_full, a_dst, slope, prep, None, p_drop, seed)
        if marks: marks[2].record()
        z = Fn.in_out(zimg, n, K, prep, bias)
        ctx.save_for_backward(x_own, W, a_s, a_d, att.alpha, att.jflag, att.rowmax, att.rowsum, zimg, prep)
        ctx.step, ctx.x_full, ctx.slope, ctx.p, ctx.seed, ctx.marks = step, x_full, slope, p_drop, seed, marks
        ctx.att_shape, ctx.has_bias = att_src.shape, bias is not None
        return z

    @staticmethod
    def backward(ctx, d_out):
        from . import functional as Fn
        x_own, W, a_s, a_d, alpha, jflag, rowmax, rowsum, zimg, prep = ctx.saved_tensors
        step, marks = ctx.step, ctx.marks
        part, px = step.part, step.px
        g, n, P, H, dev = part.graph, part.n_local, part.rows_padded, 8, x_own.device
        lo = part.rank * P
        d_out = d_out.contiguous()
        att = Fn.InAttention(alpha, jflag, rowmax, rowsum)
        need_dx = ctx.needs_input_grad[0]
        if marks: marks[4].record()
        da_out = px.da_part if px is not None else None
        if need_dx:
            alpha_used, dz, da_dst = Fn.in_bwd_edges(g, ctx.x_full, att, d_out, prep, ctx.slope, None, ctx.p, seed=ctx.seed,
                                                     records=True)
            if marks: marks[5].record()
            da_dst_full = torch.zeros(part.n_pos, H, dtype=torch.float32, device=dev)
            da_dst_full[lo:lo + n] = da_dst
            # dxw_part [n_pos, H*C] and da_src_part: linear in this rank's edges, so their sums over ranks are the layer's
            dxw, da_part = Fn.gat_bwd_src(g, alpha_used, dz, d_out, a_s, a_d, da_dst_full, H, 64, False, da_src_out=da_out)
        else:
            dz, da_dst = Fn.in_bwd_edges(g, ctx.x_full, att, d_out, prep, ctx.slope, None, ctx.p, seed=ctx.seed)
            if marks: marks[5].record()
            da_part = Fn.in_dasrc(g, dz, out=da_out)
        if marks: marks[6].record()
        if px is not None:
            # the da_src exchange runs on the side stream under the tensor-core part of the weight gradient (dO^T Z)
            da_src = torch.empty(P, H, dtype=torch.float32, device=dev)
            main = torch.cuda.current_stream()
            px.side.wait_stream(main)
            with torch.cuda.stream(px.side):
                px.barrier()
                Fn.peer_reduce(px.da_peers, lo * H, P * H, da_src, op="sum", use_multicast=px.mode == "multicast")
            finish = Fn.in_bwd_params_split(zimg, d_out, x_own, W, a_s, a_d, prep)
            main.wait_stream(px.side)
            dW, datt_s, datt_d, dbias = finish(da_src[:n], da_dst)
        else:
            if part.world > 1:
                da_src = torch.empty(P, H, dtype=torch.float32, device=dev)
                dist.reduce_scatter_tensor(da_src, da_part)
            else:
                da_src = da_part
            dW, datt_s, datt_d, dbias = Fn.in_bwd_params(zimg, d_out, x_own, W, a_s, a_d, da_src[:n], da_dst, prep)
        if marks: marks[7].record()
        dx = None
        if need_dx:
            if px is not None:
                # every rank passed the da_src barrier above only after its previous layer's dx pulls: the buffer is free
                Fn.project_dx(dxw, W, H, 64, out=step.dx_buf)
                px.barrier()
                dh = torch.empty(P, 64, dtype=torch.float32, device=dev)
                Fn.peer_reduce(step.dx_peers, lo * 64, P * 64, dh, op="sum",
                               use_multicast=px.mode == "multicast" and step.dx_peers.multicast is not None)
            else:
                dx_part = Fn.project_dx(dxw, W, H, 64)
                if part.world > 1:
                    dh = torch.empty(P, 64, dtype=torch.float32, device=dev)
                    dist.reduce_scatter_tensor(dh, dx_part)
                else:
                    dh = dx_part
            dx = dh[:n]
        if marks: marks[8].record()
        return (dx, dW, datt_s.view(ctx.att_shape), datt_d.view(ctx.att_shape), dbias if ctx.has_bias else None,
                None, None, None, None, None, None)


class InputSpaceModelTrainStep:
    """Training of a whole ``GAT`` / ``TemporalGNN`` on a destination-range partition (``InputSpaceModelPartition``), every
    layer in the input-space formulation -- the cross-GPU form of one full-batch step of the single-GPU model with
    ``gemm_algo=GEMM_INPUT`` on every layer, ``fused.masked_bce_with_logits`` and Adam.

    ``x_full``: the model input replicated in padded position space (as ``InputSpaceModelPartition.forward`` takes it);
    ``y``: the global labels ``[N]`` (-1 = unlabelled), of which each rank uses its own rows.  The parameters and buffers are
    broadcast from rank 0 at construction.  ``step()`` runs the forward, the loss of the own rows weighted by this rank's
    share of the labelled nodes (the global mean over labelled nodes), ``backward``, one all-reduce of the flat parameter
    gradients (the BatchNorm affine gradients come out of the tail's backward already summed) and Adam, identical on every
    rank.  Per layer each rank
      forward   gathers the logits of its rows to every rank (``exchange_logits``), aggregates over its destination rows,
                runs the output GEMM, then BatchNorm with the batch statistics of all ranks (one all-reduce of the column sums),
                ReLU, feature dropout and the residual; the finished rows are stored into the next layer's input buffer on
                every rank (``gnnfd_bn_relu_drop_res_fwd_bcast``), then a barrier;
      backward  runs the edge pass and the source-major pass over its edges, reduces ``da_src`` to the owners, and -- for a
                hidden layer -- writes its ``dx`` partial over all ``n_pos`` positions (the dx GEMM) into a symmetric buffer
                that each owner reduces over its row range (``gnnfd_peer_reduce``): 256 B per node instead of 2 KB of
                ``dxw``.  The dx GEMM and ``dxw_part`` (2 KB per node, transient) cover every position on every rank: they do
                not shrink with the number of ranks.
    Every hidden layer keeps its own input buffer (the backward gathers from it), so ``num_layers - 1`` hidden buffers and
    one dx buffer are allocated once.  ``GNNFD_EXCHANGE=nccl``, or no symmetric memory, uses NCCL all-gathers and
    reduce-scatters instead.

    Dropout: the seeds of step ``s`` and layer ``l`` are ``dropout_seeds(seed, s, l)``, the same on every rank with no
    collective.  Feature dropout is keyed on global rows, so its masks equal the single-GPU model's.  Attention dropout is
    keyed on the position in this rank's local ``edge_index'`` (``DstRangePlan.local_edges``: the original order, then the
    self-loops): the masks have the single-GPU distribution, and at one rank the single-GPU bits, but not the same bits when
    there is more than one rank.
    """

    def __init__(self, part: InputSpaceModelPartition, model, x_full: torch.Tensor, y: torch.Tensor, pos_weight: float = 50.0,
                 lr: float = 1e-3, weight_decay: float = 5e-4, seed: int = 0):
        from . import fused
        from .models import TemporalGNN
        InputSpaceModelPartition.check_model(model, training=True)
        if not model.use_batch_norm:
            raise NotImplementedError("InputSpaceModelTrainStep needs use_batch_norm=True: the hidden rows are broadcast by the "
                                      "BatchNorm tail")
        if not model.fused_tail:
            raise NotImplementedError("InputSpaceModelTrainStep runs the fused BatchNorm tail: fused_tail=False is not supported")
        if not 0.0 <= model.dropout <= 0.9:
            raise NotImplementedError(f"the input-space formulation supports dropout <= 0.9, got {model.dropout}")
        self.is_tgn = isinstance(model, TemporalGNN)
        if self.is_tgn and not (model.fused_head and fused.gru_head_supported(model.gru, model.out)):
            raise NotImplementedError("InputSpaceModelTrainStep runs the TemporalGNN head as fused.gru_head")
        if (not x_full.is_cuda or x_full.dtype != torch.float32 or x_full.dim() != 2
                or tuple(x_full.shape) != (part.n_pos, model.in_channels)):
            raise ValueError(f"x_full must be float32 CUDA [{part.n_pos},{model.in_channels}] in padded position space, "
                             f"got {x_full.dtype} {tuple(x_full.shape)} on {x_full.device}")
        N = part.plan.num_nodes
        if y.dim() != 1 or y.numel() != N or y.device != x_full.device:
            raise ValueError(f"y must be the global labels [{N}] on {x_full.device}, got {tuple(y.shape)} on {y.device}")
        self.part, self.model, self.x_full, self.pos_weight, self.seed = part, model, x_full, float(pos_weight), int(seed)
        self.lo, self.hi = int(part.plan.start[part.rank]), int(part.plan.start[part.rank + 1])
        self.y_own = y[self.lo:self.hi].long().contiguous()
        dev, world = x_full.device, part.world
        if world > 1:
            state = [t for t in list(model.parameters()) + list(model.buffers()) if t.dtype == torch.float32]
            flat = torch.cat([t.detach().reshape(-1) for t in state])
            dist.broadcast(flat, src=0)
            k = 0
            with torch.no_grad():
                for t in state:
                    t.copy_(flat[k:k + t.numel()].view_as(t))
                    k += t.numel()
        n_lab = torch.tensor([float((self.y_own != -1).sum())], dtype=torch.float64, device=dev)
        own_lab = float(n_lab.item())
        if world > 1:
            dist.all_reduce(n_lab)
        self.w_lab = own_lab / max(float(n_lab.item()), 1.0)        # this rank's share of the labelled nodes
        self.params = list(model.parameters())
        # the BatchNorm tails' backward all-reduces its column sums: dgamma / dbeta are already the whole batch's on every rank
        bn_params = {id(q) for bn in model.batch_norms for q in bn.parameters()}
        self.reduced = [q for q in self.params if id(q) not in bn_params]
        self.optimizer = torch.optim.Adam(self.params, lr=lr, weight_decay=weight_decay)
        L = model.num_layers
        self.px, bufs, peers, self._handles, self.exchange = part.hidden_buffers(L if L > 1 else 0)
        self.hidden, self.dx_buf = bufs[:L - 1], (bufs[L - 1] if L > 1 else None)
        self.hidden_peers = peers[:L - 1] if peers else None
        self.dx_peers = peers[L - 1] if (peers and L > 1) else None
        self.totals = torch.zeros(8, dtype=torch.float64, device=dev)
        self.steps = 0

    @staticmethod
    def dropout_seeds(seed: int, step: int, layer: int):
        """(attention seed, feature seed) of ``layer`` in step ``step``: host arithmetic, the same on every rank."""
        base = _splitmix64(_splitmix64(_splitmix64(int(seed) & 0xFFFFFFFFFFFFFFFF) ^ int(step)) ^ int(layer))
        return _splitmix64(base ^ 1) >> 2, _splitmix64(base ^ 2) >> 2

    def step(self, marks=None):
        """One optimizer step.  Returns device tensors ``(loss, stats)``: the global loss (mean over all labelled nodes) and
        this rank's counters.  ``marks``: optional per-layer lists of 9 CUDA events -- forward: start, logits + exchange done,
        aggregation done, output GEMM + BatchNorm + broadcast done; backward: start, edge pass done, source pass done,
        parameter gradients (with the da_src exchange) done, dx GEMM + reduce done -- and one more list of 2 (head start,
        optimizer done)."""
        from . import fused
        model, part, px = self.model, self.part, self.px
        model.train()
        n, P, world = part.n_local, part.rows_padded, part.world
        lo = part.rank * P
        group = dist.group.WORLD if world > 1 else None
        self.optimizer.zero_grad(set_to_none=True)
        x_own, h_full = self.x_full[lo:lo + n], self.x_full
        L = len(model.gat_layers)
        for i, conv in enumerate(model.gat_layers):
            m = marks[i] if marks else None
            s_att, s_feat = self.dropout_seeds(self.seed, self.steps, i)
            z = _RankLayer.apply(x_own, conv.lin_src.weight, conv.att_src, conv.att_dst, conv.bias, self, h_full,
                                 conv.negative_slope, conv.dropout, s_att, m)
            res = x_own.contiguous() if (model.residual and x_own.size(1) == z.size(1)) else None
            bcast = None
            if i < L - 1 and px is not None:
                bcast = (self.hidden_peers[i], lo, px.mode == "multicast" and self.hidden_peers[i].multicast is not None)
            h = fused.bn_relu_dropout_residual(z, model.batch_norms[i], model.dropout, res, seed=s_feat, row_base=self.lo,
                                               group=group, global_rows=part.plan.num_nodes, bcast=bcast)
            if i < L - 1:
                h_full = self.hidden[i]
                if px is not None:
                    px.barrier()       # every rank's rows have landed
                else:
                    h_full[lo:lo + n].copy_(h.detach())
                    if world > 1:
                        dist.all_gather_into_tensor(h_full, h_full[lo:lo + P])
            if m: m[3].record()
            x_own = h
        if marks: marks[L][0].record()
        logits = fused.gru_head(x_own, model.gru, model.out)[0] if self.is_tgn else model.out(x_own)
        self.logits = logits.detach()       # the own rows' logits of this step (before the update)
        loss, stats = fused.masked_bce_with_logits(logits, self.y_own, self.pos_weight)
        (loss * self.w_lab).backward()
        loss = loss.detach() * self.w_lab
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in self.reduced] + [loss.reshape(1)])
            dist.all_reduce(flat)      # also the step-end rendezvous that keeps a fast rank out of the next step's buffers
            k = 0
            for p in self.reduced:
                p.grad.copy_(flat[k:k + p.numel()].view_as(p))
                k += p.numel()
            loss = flat[k]
        self.optimizer.step()
        if marks: marks[L][1].record()
        self.totals.add_(stats)
        self.steps += 1
        return loss, stats

    def metrics(self, reset: bool = True):
        """As ``DeviceTrainStep.metrics``, with the counters summed over the ranks (one all-reduce, one synchronisation)."""
        from .train_step import metrics_from_totals
        t = self.totals.clone()
        if self.part.world > 1:
            dist.all_reduce(t)
        if reset:
            self.totals.zero_()
        return metrics_from_totals(t.tolist())
