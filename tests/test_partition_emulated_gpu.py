"""The multi-GPU partitions of ``partition.py`` on ONE GPU: G emulated ranks run the real ``build`` / ``layer_fwd_bwd`` in
lockstep threads on cuda:0, with the collectives and the peer-memory exchange replaced by exact in-process fakes.

Every mode the partitions drive in the library is a plain kernel call on device pointers -- rank views of the padded CSR
(``n_src = n_pos > n_dst``, shifted ``csc_row``, ``da_dst_view``), the indirect edge gradients of the receive-side CSC
(``edge_grads_indirect``), the input-space passes on a row view, and the peer kernels (``gnnfd_in_logits_bcast``,
``gnnfd_peer_reduce``).  Only the collectives couple the ranks, so emulating them exactly lets a single-GPU machine check
the partitions against the single-GPU layer and the fp64 oracle.

The fakes reduce in rank order with sequential fp32 adds, so every rank's all-reduced gradients are bit-identical and the
exchange mechanisms (collectives, peer stores / loads, redundant logits) must agree bit for bit.
"""
import ctypes as C
import functools
import threading
import time
import types

import pytest
import torch
import torch.distributed

from gnn_fraud_detection_b200 import _abi, build_csr, functional as Fn, partition, synth
from gnn_fraud_detection_b200.partition import DstRangePartition, InputSpacePartition, ReplicatedInputPartition
from oracle import pyg_gatconv as O
from util import maxabs, relerr, seeded_params

N, E, K, H, C_ = 20_000, 200_000, 166, 8, 64
BARRIER_TIMEOUT = 120.0
CLASSES = {"dst_range": DstRangePartition, "replicated_input": ReplicatedInputPartition, "input_space": InputSpacePartition}


# ------------------------------------------------------------------------------------------------
# lockstep harness: one thread per rank, exact collectives
# ------------------------------------------------------------------------------------------------
def _sync():
    if torch.cuda.is_available():
        torch.cuda.synchronize()


class _Done:
    """What ``async_op=True`` returns: the fake collective has already completed."""

    def wait(self):
        return True


class EmulatedWorld:
    """G ranks in one process.  Each collective: deposit a clone of the input, synchronize, barrier, compute this rank's
    result with torch ops (sums in rank order, fp32, sequential adds), synchronize, barrier.  Both synchronizations are
    device-wide, so the ordering holds whatever streams the caller uses."""

    def __init__(self, G, timeout=BARRIER_TIMEOUT):
        self.G, self.timeout = G, timeout
        self.barrier = threading.Barrier(G, timeout=timeout)
        self.local = threading.local()
        self.slots = [None] * G
        self.sum_inputs = [[] for _ in range(G)]     # per rank: (collective, nonzero count, all finite) of every SUM input
        self.px = [None] * G                          # the fake PeerExchange of every rank

    @property
    def rank(self):
        return self.local.rank

    def _deposit(self, *item):
        r = self.rank
        self.slots[r] = item
        _sync()
        self.barrier.wait()
        return list(self.slots)

    def _finish(self):
        _sync()
        self.barrier.wait()

    def _record_sum(self, name, t):
        self.sum_inputs[self.rank].append((name, int(torch.count_nonzero(t)), bool(torch.isfinite(t).all())))

    # -- the subset of torch.distributed that partition.py calls --
    def get_rank(self):
        return self.rank

    def get_world_size(self):
        return self.G

    def all_gather_into_tensor(self, out, inp, async_op=False):
        ins = self._deposit(inp.clone())            # the input may be a slice of ``out`` itself
        assert out.size(0) == self.G * inp.size(0) and out.shape[1:] == inp.shape[1:]
        out.copy_(torch.cat([s[0] for s in ins], 0))
        self._finish()
        return _Done() if async_op else None

    def reduce_scatter_tensor(self, out, inp, async_op=False):
        self._record_sum("reduce_scatter", inp)
        ins = self._deposit(inp.clone())
        n = out.size(0)
        assert inp.size(0) == self.G * n
        r = self.rank
        acc = ins[0][0][r * n:(r + 1) * n].clone()
        for s in range(1, self.G):
            acc = acc + ins[s][0][r * n:(r + 1) * n]
        out.copy_(acc)
        self._finish()
        return _Done() if async_op else None

    def all_reduce(self, t, op=torch.distributed.ReduceOp.SUM, async_op=False):
        if op == torch.distributed.ReduceOp.SUM:
            self._record_sum("all_reduce", t)
        elif op != torch.distributed.ReduceOp.MAX:
            raise NotImplementedError(f"fake all_reduce: op {op}")
        ins = self._deposit(t.clone())
        acc = ins[0][0].clone()
        for s in range(1, self.G):
            acc = acc + ins[s][0] if op == torch.distributed.ReduceOp.SUM else torch.maximum(acc, ins[s][0])
        t.copy_(acc)
        self._finish()
        return _Done() if async_op else None

    def all_to_all_single(self, out, inp, output_split_sizes=None, input_split_sizes=None, async_op=False):
        G = self.G
        if input_split_sizes is None:
            assert inp.size(0) % G == 0
            input_split_sizes = [inp.size(0) // G] * G
        ins = self._deposit(inp.clone(), list(input_split_sizes))
        r = self.rank
        chunks = []
        for s in range(G):
            t, splits = ins[s]
            assert sum(splits) == t.size(0)
            lo = sum(splits[:r])
            chunks.append(t[lo:lo + splits[r]])
        if output_split_sizes is not None:
            assert [c.size(0) for c in chunks] == list(output_split_sizes), "output splits disagree with the senders"
        res = torch.cat(chunks, 0)
        assert res.shape == out.shape, (tuple(res.shape), tuple(out.shape))
        out.copy_(res)
        self._finish()
        return _Done() if async_op else None

    def module(self):
        """A stand-in for ``torch.distributed`` inside ``partition.py``."""
        return types.SimpleNamespace(
            all_gather_into_tensor=self.all_gather_into_tensor, reduce_scatter_tensor=self.reduce_scatter_tensor,
            all_reduce=self.all_reduce, all_to_all_single=self.all_to_all_single, get_rank=self.get_rank,
            get_world_size=self.get_world_size, ReduceOp=torch.distributed.ReduceOp)

    def peer_exchange_class(self):
        """A stand-in for ``partition.PeerExchange``: every rank's symmetric buffers are separate allocations on the one
        device, so a wrong rank index reads the wrong data; there is no multicast mapping."""
        world = self

        class FakePeerExchange:
            def __init__(self, n_pos, device, mode="auto", H=8):
                if mode == "multicast":
                    raise RuntimeError("GNNFD_EXCHANGE=multicast: the emulated ranks have no multicast mapping")
                self.world, self.rank, self.mode = world.G, world.rank, "peer"
                # a_src starts as NaN: a row that no rank stored shows up in every comparison
                self.a_src = torch.full((n_pos, H), float("nan"), dtype=torch.float32, device=device)
                self.da_part = torch.empty((n_pos, H), dtype=torch.float32, device=device)
                self.xmax = torch.empty((16,), dtype=torch.float32, device=device)
                world.px[self.rank] = self
                self.barrier()                          # every rank has registered its buffers
                self.a_src_peers, self.da_peers, self.xmax_peers = (
                    self._peers([getattr(world.px[r], name) for r in range(world.G)]) for name in ("a_src", "da_part", "xmax"))
                self.da_part.zero_()
                self.xmax.zero_()
                self.side = torch.cuda.Stream(device=device)
                self.barrier()

            def _peers(self, bufs):
                p = _abi.Peers()
                p.n_peers, p.rank = len(bufs), self.rank
                for r, b in enumerate(bufs):
                    p.ptr[r] = b.data_ptr()
                p.multicast = None
                return p

            def barrier(self):
                world._finish()

        return FakePeerExchange

    def run(self, fn, join_timeout=None):
        """``fn(rank)`` on G threads; returns the per-rank results.  A rank that raises breaks the barrier, so the others
        fail fast instead of waiting; the first exception that is not a broken barrier is re-raised."""
        results, errors = [None] * self.G, [None] * self.G

        def body(r):
            self.local.rank = r
            try:
                results[r] = fn(r)
            except BaseException as ex:      # noqa: BLE001 -- re-raised by the main thread
                errors[r] = ex
                self.barrier.abort()

        threads = [threading.Thread(target=body, args=(r,), daemon=True, name=f"emulated-rank-{r}") for r in range(self.G)]
        for t in threads:
            t.start()
        deadline = time.monotonic() + (join_timeout if join_timeout is not None else 4 * self.timeout + 600)
        for t in threads:
            t.join(max(0.0, deadline - time.monotonic()))
        hung = [t.name for t in threads if t.is_alive()]
        if hung:
            self.barrier.abort()
            raise AssertionError(f"emulated ranks did not finish: {hung}")
        real = [e for e in errors if e is not None and not isinstance(e, threading.BrokenBarrierError)]
        if real:
            raise real[0]
        broken = [e for e in errors if e is not None]
        if broken:
            raise broken[0]
        return results


@pytest.fixture
def emulate(monkeypatch):
    """``emulate(G)``: an EmulatedWorld whose fakes are installed in ``partition`` for this test."""

    def make(G):
        world = EmulatedWorld(G)
        monkeypatch.setattr(partition, "dist", world.module())
        monkeypatch.setattr(partition, "PeerExchange", world.peer_exchange_class())
        return world
    return make


# ------------------------------------------------------------------------------------------------
# harness self-test (CPU tensors; runs without a GPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3, 8])
def test_fake_collectives_match_hand_built_results(G):
    world = EmulatedWorld(G, timeout=30)
    n = 5
    data = [torch.randn(G * n, 3, generator=torch.Generator().manual_seed(100 + r)) * 10.0 ** (r % 4) for r in range(G)]
    # all-to-all with uneven splits, zero splits included: rank s sends (s + d) % 3 rows to rank d
    split = [[(s + d) % 3 for d in range(G)] for s in range(G)]
    a2a_in = [torch.arange(sum(split[s]), dtype=torch.float32)[:, None] + 1000.0 * s for s in range(G)]

    def fn(r):
        out = {}
        own = torch.full((G * 2, 4), -1.0)
        own[r * 2:(r + 1) * 2] = torch.arange(8, dtype=torch.float32).view(2, 4) + 10.0 * r
        h = world.all_gather_into_tensor(own, own[r * 2:(r + 1) * 2], async_op=True)     # input aliases the output
        h.wait()
        out["ag"] = own
        rs = torch.empty(n, 3)
        world.reduce_scatter_tensor(rs, data[r])
        out["rs"] = rs
        s, m = data[r][:4].clone(), data[r][:4].clone()
        world.all_reduce(s)
        world.all_reduce(m, op=torch.distributed.ReduceOp.MAX)
        out["sum"], out["max"] = s, m
        recv = [split[s_][r] for s_ in range(G)]
        o = torch.empty(sum(recv), 1)
        world.all_to_all_single(o, a2a_in[r], recv, split[r])
        out["a2a"] = o
        eq = torch.arange(G * 2, dtype=torch.float32) + 100.0 * r
        oe = torch.empty(G * 2)
        world.all_to_all_single(oe, eq)
        out["a2a_even"] = oe
        return out

    res = world.run(fn)
    gathered = torch.cat([torch.arange(8, dtype=torch.float32).view(2, 4) + 10.0 * r for r in range(G)])
    for r in range(G):
        assert torch.equal(res[r]["ag"], gathered)
        acc = data[0][r * n:(r + 1) * n].clone()
        for s in range(1, G):
            acc = acc + data[s][r * n:(r + 1) * n]
        assert torch.equal(res[r]["rs"], acc)
        acc = data[0][:4].clone()
        for s in range(1, G):
            acc = acc + data[s][:4]
        assert torch.equal(res[r]["sum"], acc)
        assert torch.equal(res[r]["max"], torch.stack([d[:4] for d in data]).amax(0))
        exp = torch.cat([a2a_in[s][sum(split[s][:r]):sum(split[s][:r + 1])] for s in range(G)])
        assert torch.equal(res[r]["a2a"], exp)
        exp_even = torch.cat([torch.arange(2 * r, 2 * r + 2, dtype=torch.float32) + 100.0 * s for s in range(G)])
        assert torch.equal(res[r]["a2a_even"], exp_even)
        assert [name for name, _, _ in world.sum_inputs[r]] == ["reduce_scatter", "all_reduce"]


def test_fake_collectives_rank_order_is_sequential_fp32():
    """The sum is (((r0 + r1) + r2) + ...) in fp32, not a pairwise or fp64 reduction: 1 + 2^-24 + 2^-24 stays 1."""
    world = EmulatedWorld(3, timeout=30)
    vals = [1.0, 2.0 ** -24, 2.0 ** -24]

    def fn(r):
        t = torch.tensor([vals[r]], dtype=torch.float32)
        world.all_reduce(t)
        return t

    for t in world.run(fn):
        assert t.item() == 1.0


def test_failing_rank_fails_fast():
    world = EmulatedWorld(3, timeout=60)

    def fn(r):
        if r == 1:
            raise ValueError("rank 1 failed")
        t = torch.zeros(2)
        world.all_reduce(t)

    t0 = time.monotonic()
    with pytest.raises(ValueError, match="rank 1 failed"):
        world.run(fn)
    assert time.monotonic() - t0 < 30


def test_missing_rank_times_out():
    world = EmulatedWorld(3, timeout=1.0)

    def fn(r):
        if r == 2:
            return None                 # never joins the collective
        world.all_reduce(torch.zeros(2))

    t0 = time.monotonic()
    with pytest.raises(threading.BrokenBarrierError):
        world.run(fn)
    assert time.monotonic() - t0 < 30


# ------------------------------------------------------------------------------------------------
# graphs, inputs, single-GPU and fp64 references (built once per module)
# ------------------------------------------------------------------------------------------------
HUB_DST, HUB_SRC, BIG_DST = 4321, 9876, 777


def _edges(name):
    """``hubs``: the 200K-edge power-law graph plus a destination with ~3000 in-edges, a source with 1500 out-edges (the
    background's out-degree is at most ~26, so without it no hub-source kernel runs), duplicated edges and explicit self
    loops.  ``empty_ranks``: the power-law graph plus 150,000 edges into one destination, so that at G = 8 the plan gives
    ranks 1 and 2 empty ranges."""
    ei = synth.powerlaw_graph(N, E, seed=11)
    g = torch.Generator().manual_seed(13)
    if name == "hubs":
        into = torch.stack([torch.randint(0, N, (3000,), generator=g), torch.full((3000,), HUB_DST)])
        # the hub source's destinations sit in one narrow id range, so one rank's CSC holds all 1500 out-edges at every G
        outof = torch.stack([torch.full((1500,), HUB_SRC), torch.randint(100, 400, (1500,), generator=g)])
        dup = ei[:, torch.randint(0, E, (4000,), generator=g)]
        loops = torch.randint(0, N, (500,), generator=g).repeat(2, 1)
        ei = torch.cat([ei, into, outof, dup, loops, into[:, :50]], 1)
        ei = ei[:, torch.randperm(ei.size(1), generator=g)]
    else:
        ei = torch.cat([ei, torch.stack([torch.randint(0, N, (150_000,), generator=g), torch.full((150_000,), BIG_DST)])], 1)
    return ei.contiguous()


def _single_gpu(ei, x, prm, d_out, xw_dtype):
    W, a_s, a_d, b = prm
    g = build_csr(ei, N)
    xw, a_src, a_dst = Fn.project_fwd(x, W, a_s, a_d, H, C_, xw_dtype, _abi.GEMM_AUTO)
    out, rowmax, rowsum = Fn.gat_fwd(g, xw, a_src, a_dst, b, H, C_, 0.2, False)
    dxw, da_src, da_dst = Fn.gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C_, 0.2, False)
    dW, ds, dd, db, _ = Fn.project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C_, C_, False, _abi.GEMM_AUTO)
    torch.cuda.synchronize()
    return out, (dW, ds, dd, db)


def _make_case(name):
    """Inputs, the single-GPU fp32 layer and the fp64 oracle of one graph."""
    dev = torch.device("cuda", 0)
    ei = _edges(name)
    W, a_s, a_d, b = seeded_params(K, H, C_, seed=3)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(4))
    d_out = torch.randn(N, C_, generator=torch.Generator().manual_seed(5)) / N
    gpu = dict(ei=ei.to(dev), x=x.to(dev), d_out=d_out.to(dev),
               prm=(W.to(dev), a_s.view(-1).to(dev), a_d.view(-1).to(dev), b.to(dev)))
    ref = _single_gpu(gpu["ei"], gpu["x"], gpu["prm"], gpu["d_out"], torch.float32)
    xd, Wd = x.double(), W.double()
    ro, _ = O.gatconv_forward(xd, ei, Wd, a_s.double(), a_d.double(), b.double(), H, C_, False)
    cf = O.gatconv_backward_closed_form(xd, ei, Wd, a_s.double(), a_d.double(), H, C_, d_out.double(), False, need_dx=False)
    oracle = (ro, (cf["dW"], cf["datt_src"].reshape(-1), cf["datt_dst"].reshape(-1), cf["dbias"]))
    return dict(gpu, ref=ref, oracle=oracle)


@pytest.fixture(scope="module")
def cases():
    """``cases(name)``: the case of one graph, built the first time a test asks for it and kept for the module."""
    return functools.lru_cache(maxsize=None)(_make_case)


def _rank_input(part, x):
    """The layer input in the layout each class takes: own rows padded to P, or the replicated input in position space."""
    rank = part.rank
    lo, hi = int(part.plan.start[rank]), int(part.plan.start[rank + 1])
    if type(part) is DstRangePartition:
        xl = torch.zeros(part.rows_padded, K, device=x.device)
        xl[:hi - lo] = x[lo:hi]
        return xl
    pos = part.plan.to_pos(torch.arange(N, device=x.device))
    if type(part) is ReplicatedInputPartition:
        xp = torch.zeros(part.n_pos, K, device=x.device)
        xp[pos] = x
        return xp
    x16 = torch.zeros(part.n_pos, Fn.in_sizes(0, K)[3], device=x.device)     # 16-byte aligned zero-padded rows
    x16[pos, :K] = x
    return x16[:, :K]


def _run_partition(world, cls, case, xw_dtype=torch.float32, weights=None):
    """Every rank builds its partition and runs ``layer_fwd_bwd`` once per entry of ``weights`` (default: the case's W)."""
    W, a_s, a_d, b = case["prm"]
    weights = [W] if weights is None else weights

    def fn(r):
        dev = torch.device("cuda", 0)
        part = cls.build(case["ei"], N, r, world.G, dev)
        lo, hi = int(part.plan.start[r]), int(part.plan.start[r + 1])
        xin = _rank_input(part, case["x"])
        dO = case["d_out"][lo:hi].contiguous()
        steps = []
        for Wk in weights:
            out, grads = part.layer_fwd_bwd(xin, Wk, a_s, a_d, b, dO, H, C_, xw_dtype, _abi.GEMM_AUTO)
            torch.cuda.synchronize()
            steps.append((out.clone(), tuple(t.clone() for t in grads)))
        rg = getattr(part, "rgraph", None)
        return dict(lo=lo, hi=hi, n_local=part.n_local, steps=steps, exchange=getattr(part, "exchange", None),
                    indirect=int(rg.c.edge_grads_indirect) if rg is not None else 0,
                    hubs=(part.graph.c.hub_dst.n_hub, part.graph.c.hub_src.n_hub, rg.c.hub_src.n_hub if rg is not None else 0))

    return world.run(fn)


GRAD_NAMES = ("dW", "datt_src", "datt_dst", "dbias")


def _check_against(res, ref, oracle=None, out_tol=1e-5, rel_tol=3e-5):
    ref_out, ref_grads = ref
    for r, rr in enumerate(res):
        out, grads = rr["steps"][0]
        lo, hi = rr["lo"], rr["hi"]
        assert out.shape == (hi - lo, C_), (r, tuple(out.shape))
        assert maxabs(out, ref_out[lo:hi]) <= out_tol, (r, "out vs 1 GPU", maxabs(out, ref_out[lo:hi]))
        if oracle is not None:
            assert maxabs(out, oracle[0][lo:hi]) <= 1e-5, (r, "out vs fp64 oracle", maxabs(out, oracle[0][lo:hi]))
    covered = torch.zeros(N, dtype=torch.bool)
    for rr in res:
        covered[rr["lo"]:rr["hi"]] = True
    assert bool(covered.all()), "the ranks' row ranges do not cover the graph"
    grads0 = res[0]["steps"][0][1]
    for name, g, gr in zip(GRAD_NAMES, grads0, ref_grads):
        assert relerr(g, gr) <= rel_tol, (name, "vs 1 GPU", relerr(g, gr))
    if oracle is not None:
        o_out = torch.cat([rr["steps"][0][0].double().cpu() for rr in res])
        assert relerr(o_out, oracle[0]) <= 1e-5, ("out vs fp64 oracle", relerr(o_out, oracle[0]))
        for name, g, go in zip(GRAD_NAMES, grads0, oracle[1]):
            assert maxabs(g, go) <= 1e-5, (name, "vs fp64 oracle max-abs", maxabs(g, go))
            assert relerr(g, go) <= 1e-5, (name, "vs fp64 oracle rel L2", relerr(g, go))
    # the fakes reduce in one order: every rank holds the same bits
    for r, rr in enumerate(res[1:], 1):
        for name, g, g0 in zip(GRAD_NAMES, rr["steps"][0][1], grads0):
            assert torch.equal(g, g0), (r, name, "differs from rank 0")


def _check_empty_ranks_contribute_zero(world, res):
    for r, rr in enumerate(res):
        if rr["n_local"] != 0:
            continue
        for name, nonzero, finite in world.sum_inputs[r]:
            assert finite and nonzero == 0, (r, name, "an empty rank contributed", nonzero, finite)
        if world.px[r] is not None:
            da = world.px[r].da_part
            assert torch.count_nonzero(da) == 0 and bool(torch.isfinite(da).all()), (r, "peer da_src partial not zero")


# ------------------------------------------------------------------------------------------------
# the partitions against the single-GPU layer and the fp64 oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["hubs", "empty_ranks"])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("cls_name", list(CLASSES))
def test_partition_matches_single_gpu_and_oracle(emulate, monkeypatch, cases, cls_name, G, graph):
    """G = 1 is a sanity check: DstRangePartition and InputSpacePartition take their plain single-GPU paths, and
    ReplicatedInputPartition sets edge_grads_indirect with an identity csc_eid.  Only G >= 2 makes csc_eid a non-identity
    permutation of the received edge gradients, so the G >= 2 cases are the ones that test the indirection."""
    monkeypatch.delenv("GNNFD_EXCHANGE", raising=False)            # auto: the (fake) peer exchange of InputSpacePartition
    monkeypatch.delenv("GNNFD_LOGITS_REDUNDANT", raising=False)
    case = cases(graph)
    world = emulate(G)
    res = _run_partition(world, CLASSES[cls_name], case)
    if graph == "empty_ranks" and G == 8:
        assert [rr["n_local"] for rr in res][1:3] == [0, 0], [rr["n_local"] for rr in res]
    hubs = [rr["hubs"] for rr in res]
    if graph == "hubs":       # the row-view hub plan and the hub-source chunks run on some rank
        assert any(h[0] > 0 for h in hubs) and any(h[1] > 0 for h in hubs), hubs
    if cls_name == "replicated_input":
        assert all(rr["indirect"] == 1 for rr in res)
        if graph == "hubs":   # ... and the indirect hub-source chunks on the receive side
            assert any(h[2] > 0 for h in hubs), hubs
    if cls_name == "input_space":
        assert all(rr["exchange"] == ("peer" if G > 1 else "none") for rr in res), [rr["exchange"] for rr in res]
    _check_against(res, case["ref"], case["oracle"])
    _check_empty_ranks_contribute_zero(world, res)


@pytest.mark.gpu
def test_dst_range_bf16_features_match_single_gpu_bf16(emulate, cases):
    case = cases("hubs")
    ref = _single_gpu(case["ei"], case["x"], case["prm"], case["d_out"], torch.bfloat16)
    world = emulate(3)
    res = _run_partition(world, DstRangePartition, case, xw_dtype=torch.bfloat16)
    _check_against(res, ref)


def _run_input_space_mode(emulate, monkeypatch, mode, case, G, weights=None):
    monkeypatch.setenv("GNNFD_EXCHANGE", "auto" if mode == "redundant" else mode)
    monkeypatch.setenv("GNNFD_LOGITS_REDUNDANT", "1" if mode == "redundant" else "0")
    world = emulate(G)
    res = _run_partition(world, InputSpacePartition, case, weights=weights)
    assert all(rr["exchange"] == ("peer" if mode == "peer" else "nccl") for rr in res), [rr["exchange"] for rr in res]
    return world, res


@pytest.mark.gpu
@pytest.mark.parametrize("graph,G", [("hubs", 2), ("hubs", 3), ("hubs", 8), ("empty_ranks", 8)])
def test_input_space_exchange_modes_are_bit_identical(emulate, monkeypatch, cases, graph, G):
    """Collectives, peer stores / loads and redundant logits: the logit rows come from the same kernel (a row's logits do
    not depend on its tile), both da_src reductions add the ranks in rank order, and xmax is a max -- so the layer's
    output and gradients agree bit for bit."""
    case = cases(graph)
    runs = {}
    for mode in ("nccl", "peer", "redundant"):
        world, res = _run_input_space_mode(emulate, monkeypatch, mode, case, G)
        _check_against(res, case["ref"])
        _check_empty_ranks_contribute_zero(world, res)
        runs[mode] = res
    for mode in ("peer", "redundant"):
        for r in range(G):
            (o, gr), (o0, gr0) = runs[mode][r]["steps"][0], runs["nccl"][r]["steps"][0]
            assert torch.equal(o, o0), (mode, r, "out", maxabs(o, o0))
            for name, a, b in zip(GRAD_NAMES, gr, gr0):
                assert torch.equal(a, b), (mode, r, name, maxabs(a, b))


@pytest.mark.gpu
def test_input_space_peer_second_step_sees_no_stale_buffers(emulate, monkeypatch, cases):
    """Three steps through the same partition and peer buffers: W, W/2, W.  The third must reproduce the first bit for bit."""
    case = cases("hubs")
    W = case["prm"][0]
    _, res = _run_input_space_mode(emulate, monkeypatch, "peer", case, 3, weights=[W, W * 0.5, W])
    for r, rr in enumerate(res):
        (o1, g1), (o2, g2), (o3, g3) = rr["steps"]
        assert not torch.equal(o1, o2) or rr["n_local"] == 0
        assert torch.equal(o3, o1), (r, "out", maxabs(o3, o1))
        for name, a, b in zip(GRAD_NAMES, g3, g1):
            assert torch.equal(a, b), (r, name, maxabs(a, b))


# ------------------------------------------------------------------------------------------------
# the peer kernels, with G separate buffers on one device as the "peers"
# ------------------------------------------------------------------------------------------------
def _peers(bufs, multicast=None):
    p = _abi.Peers()
    p.n_peers, p.rank = len(bufs), 0
    for r, b in enumerate(bufs):
        p.ptr[r] = b if (b is None or isinstance(b, int)) else b.data_ptr()
    p.multicast = multicast
    return p


def _peer_reduce_raw(p, offset, n, op, use_multicast, out):
    return _abi.lib().gnnfd_peer_reduce(C.byref(p), int(offset), int(n), int(op), int(use_multicast), out.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 5, 16])
def test_peer_reduce_is_rank_ordered_sum_and_max(G):
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(20 + G)
    L = 4099 + 6 + 16
    # magnitudes spread over six decades, so a different summation order changes the bits
    bufs = [torch.randn(L, device=dev, generator=gen) * 10.0 ** torch.randint(-3, 3, (L,), device=dev, generator=gen)
            for _ in range(G)]
    p = _peers(bufs)
    for n in (0, 1, 3, 4, 1023, 4099):
        for offset in (0, 1, 2, 4, 6):
            seg = [b[offset:offset + n] for b in bufs]
            want_sum = seg[0].clone()
            for s in seg[1:]:
                want_sum = want_sum + s
            want_max = torch.stack(seg).amax(0)
            for shift in (0, 1):              # out 16-byte aligned (float4 body + scalar tail), or one float off (scalar path)
                for op, want in ((0, want_sum), (1, want_max)):
                    base = torch.full((n + 8,), float("nan"), device=dev)
                    out = base[shift:]
                    assert _peer_reduce_raw(p, offset, n, op, 0, out) == 0, _abi.lib().gnnfd_last_error()
                    torch.cuda.synchronize()
                    assert torch.equal(out[:n], want), (G, n, offset, shift, op, maxabs(out[:n], want))
                    assert bool(torch.isnan(out[n:]).all()) and bool(torch.isnan(base[:shift]).all()), (G, n, offset, shift, op)


@pytest.mark.gpu
def test_peer_reduce_rejects_bad_arguments_before_launch():
    dev = torch.device("cuda", 0)
    bufs = [torch.randn(64, device=dev) for _ in range(3)]
    bad = []
    p0 = _peers(bufs[:1])
    p0.n_peers = 0
    bad.append(("0 peers", p0, 0, 0))
    p17 = _peers([bufs[0]] * 16)
    p17.n_peers = 17
    bad.append(("17 peers", p17, 0, 0))
    bad.append(("NULL peer", _peers([bufs[0], None, bufs[2]]), 0, 0))
    bad.append(("op 2", _peers(bufs), 2, 0))
    bad.append(("multicast without mapping", _peers(bufs), 0, 1))
    for what, p, op, mc in bad:
        out = torch.full((16,), float("nan"), device=dev)
        rc = _peer_reduce_raw(p, 0, 16, op, mc, out)
        torch.cuda.synchronize()
        assert rc == -1, (what, rc)
        assert bool(torch.isnan(out).all()), (what, "out was written")


def _bcast_raw(x, W, a_s, a_d, p, row_offset, use_multicast, a_dst, xmax, prep):
    return _abi.lib().gnnfd_in_logits_bcast(x.data_ptr(), x.stride(0), x.size(0), x.size(1), W.data_ptr(), a_s.data_ptr(),
                                            a_d.data_ptr(), C.byref(p), int(row_offset), int(use_multicast), a_dst.data_ptr(),
                                            xmax.data_ptr(), prep.data_ptr(), torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3, 8])
def test_in_logits_bcast_stores_every_rank_rows_into_every_buffer(G):
    dev = torch.device("cuda", 0)
    P = 1000                       # not a multiple of the kernel's row tile
    W, a_s, a_d, _ = (t.to(dev) for t in seeded_params(K, H, C_, seed=7))
    a_s, a_d = a_s.view(-1).contiguous(), a_d.view(-1).contiguous()
    x = Fn.in_pad_x(torch.randn(G * P, K, device=dev, generator=torch.Generator(device=dev).manual_seed(8)))
    prep = Fn._aligned_u8(Fn.in_sizes(G * P, K)[0], dev)
    a_src_full, _ = Fn.in_logits(x, W, a_s, a_d, prep, torch.zeros(16, device=dev))
    bufs = [torch.full((G * P, H), float("nan"), device=dev) for _ in range(G)]
    peers = _peers(bufs)
    for r in range(G):
        rows = x[r * P:(r + 1) * P]
        xmax = torch.zeros(16, device=dev)
        a_dst = Fn.in_logits_bcast(rows, W, a_s, a_d, prep, xmax, peers, r * P)
        torch.cuda.synchronize()
        for g, b in enumerate(bufs):
            assert torch.equal(b[r * P:(r + 1) * P], a_src_full[r * P:(r + 1) * P]), (r, g)
            assert bool(torch.isnan(b[(r + 1) * P:]).all()), (r, g, "rows of later ranks were written")
        xm_l = torch.zeros(16, device=dev)
        _, a_dst_l = Fn.in_logits(rows, W, a_s, a_d, prep, xm_l)
        assert torch.equal(a_dst, a_dst_l), r
        assert torch.equal(xmax, xm_l), r
    for g, b in enumerate(bufs):
        assert torch.equal(b, a_src_full), g


@pytest.mark.gpu
def test_in_logits_bcast_rejects_misaligned_peer_and_missing_multicast():
    dev = torch.device("cuda", 0)
    W, a_s, a_d, _ = (t.to(dev) for t in seeded_params(K, H, C_, seed=7))
    a_s, a_d = a_s.view(-1).contiguous(), a_d.view(-1).contiguous()
    x = Fn.in_pad_x(torch.randn(64, K, device=dev))
    prep = Fn._aligned_u8(Fn.in_sizes(64, K)[0], dev)
    bufs = [torch.full((64 * H + 4,), float("nan"), device=dev) for _ in range(3)]
    cases = [("misaligned peer", _peers([bufs[0], bufs[1].data_ptr() + 4, bufs[2]]), 0),
             ("multicast without mapping", _peers(bufs), 1)]
    for what, p, mc in cases:
        a_dst = torch.full((64, H), float("nan"), device=dev)
        rc = _bcast_raw(x, W, a_s, a_d, p, 0, mc, a_dst, torch.zeros(16, device=dev), prep)
        torch.cuda.synchronize()
        assert rc == -1, (what, rc)
        assert all(bool(torch.isnan(b).all()) for b in bufs) and bool(torch.isnan(a_dst).all()), (what, "a buffer was written")
