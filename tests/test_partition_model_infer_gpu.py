"""Whole-model inference across GPUs (``partition.InputSpaceModelPartition``) on ONE GPU: G emulated ranks run the real
``build`` / ``forward`` in lockstep threads on cuda:0, with the collectives, the peer exchange and the symmetric hidden
buffers replaced by exact in-process fakes -- every rank's buffers are separate allocations, so the real peer kernels
(``gnnfd_in_logits_bcast``, ``gnnfd_peer_reduce``, ``gnnfd_in_out_bcast``) store into and load from the right ranks or the
results show it.  The fake symmetric buffers start as NaN: a row that no rank stored, or a padding row that is read,
poisons every comparison.

Also the output-GEMM broadcast kernel on its own (``gnnfd_in_out_bcast`` against ``gnnfd_in_out``) and the refusals, which
need no GPU.
"""
import ctypes as C
import functools
import os
import threading
import time
import types

import numpy as np
import pytest
import torch
import torch.distributed

from gnn_fraud_detection_b200 import GAT, TemporalGNN, _abi, build_csr, functional as Fn, models, partition, synth
from gnn_fraud_detection_b200.partition import DstRangePlan, InputSpaceModelPartition
from oracle import pyg_gatconv as O
from util import load_ckpt, maxabs, relerr

BARRIER_TIMEOUT = 120.0
NAN = float("nan")


# ------------------------------------------------------------------------------------------------
# lockstep harness: one thread per rank, exact collectives, peer buffers as separate allocations
# ------------------------------------------------------------------------------------------------
class EmulatedWorld:
    """G ranks in one process.  A collective deposits a clone of its input, synchronizes the device, waits for every rank,
    computes this rank's result with torch ops and synchronizes again; a cross-GPU barrier is a device synchronization
    plus a thread barrier."""

    def __init__(self, G):
        self.G = G
        self.barrier = threading.Barrier(G, timeout=BARRIER_TIMEOUT)
        self.local = threading.local()
        self.slots = [None] * G
        self.sym = [[] for _ in range(G)]       # per rank: its symmetric buffers in allocation order

    @property
    def rank(self):
        return self.local.rank

    def _deposit(self, item):
        self.slots[self.rank] = item
        torch.cuda.synchronize()
        self.barrier.wait()
        return list(self.slots)

    def _finish(self):
        torch.cuda.synchronize()
        self.barrier.wait()

    def all_gather_into_tensor(self, out, inp, async_op=False):
        ins = self._deposit(inp.clone())            # the input may be a slice of ``out`` itself
        assert out.size(0) == self.G * inp.size(0) and out.shape[1:] == inp.shape[1:]
        out.copy_(torch.cat(ins, 0))
        self._finish()

    def all_reduce(self, t, op=torch.distributed.ReduceOp.SUM, async_op=False):
        ins = self._deposit(t.clone())
        acc = ins[0].clone()
        for s in ins[1:]:
            acc = acc + s if op == torch.distributed.ReduceOp.SUM else torch.maximum(acc, s)
        t.copy_(acc)
        self._finish()

    def module(self):
        """A stand-in for ``torch.distributed`` inside ``partition.py``."""
        return types.SimpleNamespace(all_gather_into_tensor=self.all_gather_into_tensor, all_reduce=self.all_reduce,
                                     get_rank=lambda: self.rank, get_world_size=lambda: self.G,
                                     ReduceOp=torch.distributed.ReduceOp, group=types.SimpleNamespace(WORLD=None))

    def _peers(self, bufs):
        p = _abi.Peers()
        p.n_peers, p.rank = len(bufs), self.rank
        for r, b in enumerate(bufs):
            p.ptr[r] = b.data_ptr()
        p.multicast = None
        return p

    def symmetric(self, t):
        """Register this rank's allocation; returns the peer table of the allocation every rank made at the same point."""
        self.sym[self.rank].append(t)
        k = len(self.sym[self.rank]) - 1
        self._finish()
        return self._peers([self.sym[r][k] for r in range(self.G)])

    def symmetric_buffer(self, shape, device):
        t = torch.full(shape, NAN, dtype=torch.float32, device=device)
        return t, self.symmetric(t), None

    def peer_exchange_class(self):
        world = self

        class FakePeerExchange:
            def __init__(self, n_pos, device, mode="auto", H=8):
                if mode == "multicast":
                    raise RuntimeError("GNNFD_EXCHANGE=multicast: the emulated ranks have no multicast mapping")
                self.world, self.rank, self.mode = world.G, world.rank, "peer"
                self.a_src = torch.full((n_pos, H), NAN, dtype=torch.float32, device=device)
                self.da_part = torch.zeros((n_pos, H), dtype=torch.float32, device=device)
                self.xmax = torch.zeros((16,), dtype=torch.float32, device=device)
                self.a_src_peers, self.da_peers, self.xmax_peers = (world.symmetric(t) for t in (self.a_src, self.da_part,
                                                                                                 self.xmax))

            def barrier(self):
                world._finish()

        return FakePeerExchange

    def run(self, fn):
        """``fn(rank)`` on G threads; a rank that raises breaks the barrier so that the others fail fast."""
        results, errors = [None] * self.G, [None] * self.G

        def body(r):
            self.local.rank = r
            try:
                results[r] = fn(r)
            except BaseException as ex:      # noqa: BLE001 -- re-raised by the main thread
                errors[r] = ex
                self.barrier.abort()

        threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(self.G)]
        for t in threads:
            t.start()
        deadline = time.monotonic() + 4 * BARRIER_TIMEOUT + 600
        for t in threads:
            t.join(max(0.0, deadline - time.monotonic()))
        if any(t.is_alive() for t in threads):
            self.barrier.abort()
            raise AssertionError("emulated ranks did not finish")
        real = [e for e in errors if e is not None and not isinstance(e, threading.BrokenBarrierError)]
        if real or any(e is not None for e in errors):
            raise (real or [e for e in errors if e is not None])[0]
        return results


@pytest.fixture
def emulate(monkeypatch):
    def make(G, mode):
        monkeypatch.setenv("GNNFD_EXCHANGE", mode)
        world = EmulatedWorld(G)
        monkeypatch.setattr(partition, "dist", world.module())
        monkeypatch.setattr(partition, "PeerExchange", world.peer_exchange_class())
        monkeypatch.setattr(partition, "symmetric_buffer", world.symmetric_buffer)
        return world
    return make


# ------------------------------------------------------------------------------------------------
# gnnfd_in_out_bcast against gnnfd_in_out
# ------------------------------------------------------------------------------------------------
def _peer_table(bufs, multicast=None):
    p = _abi.Peers()
    p.n_peers, p.rank = len(bufs), 0
    for r, b in enumerate(bufs):
        p.ptr[r] = b if (b is None or isinstance(b, int)) else b.data_ptr()
    p.multicast = multicast
    return p


def _image(n, K, seed):
    """A real output-GEMM operand: the aggregation image and prep of n destination rows of a random graph."""
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(seed)
    prep = Fn._aligned_u8(Fn.in_sizes(n, K)[0], dev)
    if n == 0:
        return Fn._aligned_u8(1024, dev), prep
    W, a_s, a_d = (O.glorot_(torch.empty(*s), gen).reshape(s[0], -1).to(dev) for s in ((512, K), (1, 8, 64), (1, 8, 64)))
    a_s, a_d = a_s.reshape(-1).contiguous(), a_d.reshape(-1).contiguous()
    x = Fn.in_pad_x(torch.randn(n, K, generator=gen).to(dev))
    ei = torch.randint(0, n, (2, 8 * n), generator=gen).to(dev)
    g = build_csr(ei, n)
    xmax = torch.zeros(16, device=dev)
    a_src, a_dst = Fn.in_logits(x, W, a_s, a_d, prep, xmax)
    Fn.in_prepare(W, K, xmax, prep)
    zimg, _ = Fn.in_fwd(g, x, a_src, a_dst, 0.2, prep)
    return zimg, prep


def _epilogues(n, seed):
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(seed)
    bias = torch.randn(64, generator=gen).to(dev)
    scale, shift = (torch.rand(64, generator=gen) + 0.5).to(dev), torch.randn(64, generator=gen).to(dev)
    res = torch.randn(n, 64, generator=gen).to(dev)
    return {"bias": dict(bias=bias), "none": dict(bias=None),
            "bn_relu": dict(bias=bias, act=_abi.ACT_RELU, post_scale=scale, post_shift=shift),
            "relu_residual": dict(bias=None, act=_abi.ACT_RELU, residual=res),
            "all": dict(bias=bias, act=_abi.ACT_RELU, post_scale=scale, post_shift=shift, residual=res)}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 127, 129, 1000])
@pytest.mark.parametrize("G", [1, 3, 8])
def test_in_out_bcast_stores_exactly_the_rows_of_in_out_into_every_buffer(G, n):
    """Each "rank" r broadcasts the same n rows to rows [r*P, r*P + n) of G buffers (P = n + 5: padding rows between the
    ranges); every buffer gets exactly those rows, bit-equal to gnnfd_in_out, and keeps its NaN sentinel everywhere else."""
    dev = torch.device("cuda", 0)
    P = n + 5
    for K in (64, 166):
        zimg, prep = _image(n, K, seed=100 + n + K)
        for name, epi in _epilogues(n, seed=7 + n).items():
            ref = Fn.in_out(zimg, n, K, prep, **epi)
            bufs = [torch.full((G * P, 64), NAN, device=dev) for _ in range(G)]
            peers = _peer_table(bufs)
            want = torch.full((G * P, 64), NAN, device=dev)
            for r in range(G):
                own = torch.full((n + 1, 64), NAN, device=dev) if r % 2 == 0 else None     # out given on even ranks
                got = Fn.in_out_bcast(zimg, n, K, prep, peers=peers, row_offset=r * P, out=None if own is None else own[:n],
                                      **epi)
                torch.cuda.synchronize()
                want[r * P:r * P + n] = ref
                if own is not None:
                    assert got is not None and torch.equal(own[:n], ref), (K, name, r, maxabs(own[:n], ref))
                    assert bool(torch.isnan(own[n:]).all()), (K, name, r, "out written beyond its n rows")
                for g, b in enumerate(bufs):
                    assert torch.equal(b.view(torch.int32), want.view(torch.int32)), (K, name, r, g)


def _bcast_raw(peers, use_multicast, n, zimg, prep, out):
    return _abi.lib().gnnfd_in_out_bcast(zimg.data_ptr(), n, 64, prep.data_ptr(), None, 0, None, None, None, C.byref(peers),
                                         0, int(use_multicast), _abi.ptr(out), torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
def test_in_out_bcast_refuses_bad_peers_and_missing_multicast_before_launch():
    dev = torch.device("cuda", 0)
    n = 64
    zimg, prep = _image(n, 64, seed=3)
    bufs = [torch.full((n * 64 + 4,), NAN, device=dev) for _ in range(3)]
    p0 = _peer_table(bufs[:1])
    p0.n_peers = 0
    p17 = _peer_table([bufs[0]] * 16)
    p17.n_peers = 17
    cases = [("0 peers", p0, 0), ("17 peers", p17, 0), ("NULL peer", _peer_table([bufs[0], None, bufs[2]]), 0),
             ("misaligned peer", _peer_table([bufs[0], bufs[1].data_ptr() + 4, bufs[2]]), 0),
             ("multicast without mapping", _peer_table(bufs), 1)]
    for what, p, mc in cases:
        for rows in (n, 0):                  # refused also when there is nothing to store
            out = torch.full((n, 64), NAN, device=dev)
            rc = _bcast_raw(p, mc, rows, zimg, prep, out)
            torch.cuda.synchronize()
            assert rc == -1, (what, rows, rc)
            assert all(bool(torch.isnan(b).all()) for b in bufs) and bool(torch.isnan(out).all()), (what, "a buffer was written")
    assert _bcast_raw(_peer_table(bufs[:1]), 0, 0, zimg, prep, None) == 0        # n = 0 with good peers: nothing to do


# ------------------------------------------------------------------------------------------------
# the model partition against the single-GPU model
# ------------------------------------------------------------------------------------------------
N_BIG, E_BIG, HUB_DST, HUB_SRC, BIG_DST = 20_000, 200_000, 4321, 9876, 777
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _edges(name):
    """The graphs of test_partition_emulated_gpu: ``hubs`` (a ~3000-in-edge destination, a 1500-out-edge source,
    duplicates, explicit self-loops) and ``empty_ranks`` (150,000 edges into one destination: at G = 8 ranks 1 and 2 own
    no rows)."""
    ei = synth.powerlaw_graph(N_BIG, E_BIG, seed=11)
    g = torch.Generator().manual_seed(13)
    if name == "hubs":
        into = torch.stack([torch.randint(0, N_BIG, (3000,), generator=g), torch.full((3000,), HUB_DST)])
        outof = torch.stack([torch.full((1500,), HUB_SRC), torch.randint(100, 400, (1500,), generator=g)])
        dup = ei[:, torch.randint(0, E_BIG, (4000,), generator=g)]
        loops = torch.randint(0, N_BIG, (500,), generator=g).repeat(2, 1)
        ei = torch.cat([ei, into, outof, dup, loops, into[:, :50]], 1)
        ei = ei[:, torch.randperm(ei.size(1), generator=g)]
    else:
        ei = torch.cat([ei, torch.stack([torch.randint(0, N_BIG, (150_000,), generator=g),
                                         torch.full((150_000,), BIG_DST)])], 1)
    return ei.contiguous()


def _graph(name):
    """(x, edge_index) on cpu: golden_small (600 nodes, 165 features), or a 20K-node graph with 165 random features."""
    if name == "golden_small":
        gold = np.load(os.path.join(GOLDEN, "golden_small.npz"))
        return torch.from_numpy(gold["x"]), torch.from_numpy(gold["edge_index"])
    return torch.randn(N_BIG, 165, generator=torch.Generator().manual_seed(4)), _edges(name)


_graph_cached = functools.lru_cache(maxsize=None)(_graph)


def _checkpointed():
    gat = load_ckpt(GAT(165, 64, 1, num_layers=3), os.path.join(GOLDEN, "gat_ckpt.npz")).cuda().eval()
    tgn = load_ckpt(TemporalGNN(165, 64, 1, num_layers=3), os.path.join(GOLDEN, "tgn_ckpt.npz")).cuda().eval()
    return gat, tgn


def _single_gpu(model, x, ei):
    """The reference: the single-GPU model, eval, no_grad, gemm_algo=GEMM_INPUT on every layer."""
    algos = [c.gemm_algo for c in model.gat_layers]
    for c in model.gat_layers:
        c.gemm_algo = _abi.GEMM_INPUT
    try:
        with torch.no_grad():
            r = model(x, ei)
    finally:
        for c, a in zip(model.gat_layers, algos):
            c.gemm_algo = a
    torch.cuda.synchronize()
    return r if isinstance(r, tuple) else (r,)


def _x_full(part, x):
    """The model input replicated in padded position space, 16-byte aligned zero-padded rows."""
    pos = part.plan.to_pos(torch.arange(x.size(0), device=x.device))
    x16 = torch.zeros(part.n_pos, Fn.in_sizes(0, x.size(1))[3], device=x.device)
    x16[pos, :x.size(1)] = x
    return x16[:, :x.size(1)]


def _run(world, model_list, x, ei):
    """Every rank builds the partition and runs each model of ``model_list`` through it (in order, same buffers).
    Returns per rank: dict(lo, hi, n_local, exchange, outs = [tuple of output tensors per model])."""
    N = x.size(0)

    def fn(r):
        dev = torch.device("cuda", 0)
        part = InputSpaceModelPartition.build(ei, N, r, world.G, dev)
        xf = _x_full(part, x)
        outs = []
        for m in model_list:
            res, (lo, hi) = part.forward(m, xf)
            torch.cuda.synchronize()
            outs.append(tuple(t.clone() for t in (res if isinstance(res, tuple) else (res,))))
        return dict(lo=lo, hi=hi, n_local=part.n_local, exchange=part.exchange, outs=outs)

    return world.run(fn)


def _gather(res, k):
    """Rank results of model k, concatenated in global row order (the ranges are contiguous and ascending)."""
    assert [rr["lo"] for rr in res[1:]] == [rr["hi"] for rr in res[:-1]] and res[0]["lo"] == 0
    return tuple(torch.cat([rr["outs"][k][j] for rr in res]) for j in range(len(res[0]["outs"][k])))


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["golden_small", "hubs", "empty_ranks"])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_checkpointed_models_match_single_gpu(emulate, graph, G):
    """GAT and TemporalGNN (logits and hidden state) from the reference's checkpoints: bit-identical at G = 1, max-abs
    <= 1e-5 at G > 1, and the peer exchange bit-identical to the NCCL collectives."""
    x, ei = (t.cuda() for t in _graph_cached(graph))
    gat, tgn = _checkpointed()
    refs = [_single_gpu(gat, x, ei), _single_gpu(tgn, x, ei)]
    runs = {}
    for mode in ("auto", "nccl"):
        world = emulate(G, mode)
        res = _run(world, [gat, tgn], x, ei)
        assert all(rr["exchange"] == ("none" if G == 1 else "peer" if mode == "auto" else "nccl") for rr in res)
        runs[mode] = res
        if graph == "empty_ranks" and G == 8:
            assert [rr["n_local"] for rr in res][1:3] == [0, 0], [rr["n_local"] for rr in res]
        for k, ref in enumerate(refs):
            got = _gather(res, k)
            for name, a, b in zip(("logits", "hidden"), got, ref):
                assert a.shape == b.shape and bool(torch.isfinite(a).all()), (k, name)
                if G == 1:
                    assert torch.equal(a, b), (mode, k, name, maxabs(a, b))
                else:
                    assert maxabs(a, b) <= 1e-5, (mode, k, name, maxabs(a, b))
    for r in range(G):
        for k in range(2):
            for a, b in zip(runs["auto"][r]["outs"][k], runs["nccl"][r]["outs"][k]):
                assert torch.equal(a, b), (r, k, "peer vs nccl", maxabs(a, b))


# rel L2 against the reference's fp64 outputs (and the fp64 oracle models: the same values), measured on a B200 at G = 1
# and 3 (same values at both): GAT logits 1.82e-06, TemporalGNN logits 1.13e-06, TemporalGNN hidden 1.29e-06
REL_L2_VS_REFERENCE = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3])
def test_checkpointed_models_match_the_reference_and_the_fp64_oracle(emulate, G):
    gold = np.load(os.path.join(GOLDEN, "reference_models_golden.npz"))
    xc, eic = _graph_cached("golden_small")
    oracle = {}
    for name, cls, ck in (("gat", O.OracleGAT, "gat_ckpt.npz"), ("tgn", O.OracleTemporalGNN, "tgn_ckpt.npz")):
        m = load_ckpt(cls(165, 64, 1, num_layers=3), os.path.join(GOLDEN, ck)).eval().double()
        with torch.no_grad():
            kw = {"hidden_state": torch.zeros(xc.size(0), 64, dtype=torch.float64)} if name == "tgn" else {}
            r = m(xc.double(), eic, **kw)
        oracle[name] = r if isinstance(r, tuple) else (r,)
    gat, tgn = _checkpointed()
    res = _run(emulate(G, "auto"), [gat, tgn], xc.cuda(), eic.cuda())
    (lg,), (lt, ht) = _gather(res, 0), _gather(res, 1)
    errs = {"gat_logits": (lg, gold["gat_logits_f64"], oracle["gat"][0]),
            "tgn_logits": (lt, gold["tgn_logits_f64"], oracle["tgn"][0]),
            "tgn_hidden": (ht, gold["tgn_hidden_f64"], oracle["tgn"][1])}
    for name, (got, ref, orc) in errs.items():
        e_ref, e_orc = relerr(got, torch.from_numpy(ref)), relerr(got, orc)
        print(f"G={G} {name}: rel L2 vs reference fp64 {e_ref:.3g}, vs fp64 oracle {e_orc:.3g}")
        assert e_ref <= REL_L2_VS_REFERENCE and e_orc <= REL_L2_VS_REFERENCE, (name, e_ref, e_orc)


def _random_model(cls, in_channels, num_layers, residual, use_batch_norm, seed):
    torch.manual_seed(seed)
    m = cls(in_channels, 64, 1, num_layers=num_layers, residual=residual, use_batch_norm=use_batch_norm)
    if use_batch_norm:
        g = torch.Generator().manual_seed(seed + 1)
        for bn in m.batch_norms:            # trained-looking running statistics, so the folded affine is not the identity
            bn.running_mean.copy_(torch.randn(64, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(64, generator=g) + 0.5)
            bn.weight.data.copy_(torch.rand(64, generator=g) + 0.5)
            bn.bias.data.copy_(torch.randn(64, generator=g) * 0.1)
    return m.cuda().eval()


@pytest.mark.gpu
@pytest.mark.parametrize("in_channels,num_layers,residual,use_batch_norm", [
    (165, 1, True, True), (165, 2, True, True), (165, 5, True, True), (165, 3, False, True), (165, 3, True, False),
    (64, 2, True, True),        # a 64-wide input: the first layer's residual comes from the replicated input
])
def test_other_model_shapes_match_single_gpu(emulate, in_channels, num_layers, residual, use_batch_norm):
    x, ei = _graph_cached("hubs")
    x, ei = x[:, :in_channels].contiguous().cuda(), ei.cuda()
    ms = [_random_model(cls, in_channels, num_layers, residual, use_batch_norm, seed=20 + num_layers)
          for cls in (GAT, TemporalGNN)]
    res = _run(emulate(3, "auto"), ms, x, ei)
    for k, m in enumerate(ms):
        for name, a, b in zip(("logits", "hidden"), _gather(res, k), _single_gpu(m, x, ei)):
            assert maxabs(a, b) <= 1e-5, (k, name, maxabs(a, b))


@pytest.mark.gpu
def test_second_forward_through_the_same_buffers_equals_a_fresh_run(emulate):
    """A, then B (every weight changed), then A again through one partition: B equals B run on a fresh partition and the
    second A equals the first, bit for bit -- nothing of an earlier forward leaks through the exchange buffers."""
    x, ei = (t.cuda() for t in _graph_cached("hubs"))
    a, _ = _checkpointed()
    b, _ = _checkpointed()
    with torch.no_grad():
        for p in b.parameters():
            p.mul_(0.75)
    same = _run(emulate(3, "auto"), [a, b, a], x, ei)
    fresh = _run(emulate(3, "auto"), [b], x, ei)
    for r in range(3):
        (oa,), (ob,), (oa2,) = same[r]["outs"]
        assert not torch.equal(oa, ob) or same[r]["n_local"] == 0
        assert torch.equal(ob, fresh[r]["outs"][0][0]), (r, maxabs(ob, fresh[r]["outs"][0][0]))
        assert torch.equal(oa2, oa), (r, maxabs(oa2, oa))


# ------------------------------------------------------------------------------------------------
# refusals (checked before anything touches a device: no GPU needed)
# ------------------------------------------------------------------------------------------------
def _cpu_partition(N=50):
    ei = torch.randint(0, N, (2, 200), generator=torch.Generator().manual_seed(0))
    return InputSpaceModelPartition(DstRangePlan.build(ei, N, 2), 0, torch.device("cpu"))


def test_refuses_training_mode_other_widths_heads_inputs_and_classes(monkeypatch):
    part = _cpu_partition()
    x = torch.zeros(part.n_pos, 165)
    with pytest.raises(RuntimeError, match="inference only"):
        part.forward(GAT(165, 64, 1, num_layers=2).train(), x)
    for width in (32, 128):
        with pytest.raises(NotImplementedError, match="hidden_channels=64"):
            part.forward(TemporalGNN(165, width, 1, num_layers=2).eval(), x)
    with pytest.raises(NotImplementedError, match="in_channels <= 192"):
        part.forward(GAT(200, 64, 1, num_layers=2).eval(), torch.zeros(part.n_pos, 200))
    with pytest.raises(TypeError, match="GAT or TemporalGNN"):
        part.forward(torch.nn.Linear(165, 64).eval(), x)
    monkeypatch.setattr(models, "_HEADS", 4)
    with pytest.raises(NotImplementedError, match="8 heads"):
        part.forward(GAT(165, 64, 1, num_layers=2).eval(), x)
