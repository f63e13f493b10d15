"""Whole-model training across GPUs (``partition.InputSpaceModelTrainStep``) on ONE GPU: G emulated ranks run the real
``build`` / ``step`` in lockstep threads on cuda:0 (the harness of ``test_partition_model_infer_gpu``, extended with the
collectives training adds).  Symmetric buffers start as NaN: a row no rank stored, or a padding row that is read, shows up.

* G = 1 is bit-equal to one step of the single-GPU model (``gemm_algo=GEMM_INPUT`` on every layer, ``masked_bce_with_logits``,
  Adam), with dropout off and on;
* G > 1 matches the single-GPU model and the fp64 oracle -- with dropout on, fed each rank's attention masks put back in
  ``edge_index'`` order and the row-keyed feature masks;
* the peer exchange and the NCCL collectives give the same bits, and every rank ends with the same parameters;
* the BatchNorm tail that broadcasts its rows (``gnnfd_bn_relu_drop_res_fwd_bcast``) against the one that does not;
* the refusals, without a GPU; and the same comparisons on real ranks when the box has two GPUs or more.
"""
import copy
import ctypes as C
import functools
import os

import pytest
import torch
import torch.distributed
import torch.distributed as dist
import torch.multiprocessing as mp

from gnn_fraud_detection_b200 import GAT, TemporalGNN, _abi, fused, partition, synth
from gnn_fraud_detection_b200 import functional as Fn
from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE, _stream
from gnn_fraud_detection_b200.partition import DstRangePlan, InputSpaceModelPartition, InputSpaceModelTrainStep
from oracle import pyg_gatconv as O
from test_dropout_training_gpu import _errors, _oracle_step, _relu_decisions
from test_partition_model_infer_gpu import NAN, EmulatedWorld, _edges, _peer_table, _x_full
from util import maxabs, relerr

N_BIG, E_BIG, K = 20_000, 200_000, 166
SEED = 12345


class TrainWorld(EmulatedWorld):
    """The inference harness plus what a training step calls: ``reduce_scatter_tensor`` (summed in rank order, as
    ``gnnfd_peer_reduce`` does), ``broadcast``, ``all_reduce`` with a group, a non-None ``group.WORLD`` (the BatchNorm
    statistics are all-reduced only when a group is given), the peer exchange's side stream, and the backward on each rank's
    thread."""

    def all_reduce(self, t, op=torch.distributed.ReduceOp.SUM, group=None, async_op=False):
        super().all_reduce(t, op)

    def reduce_scatter_tensor(self, out, inp, async_op=False):
        ins = self._deposit(inp.clone())
        n = out.size(0)
        assert inp.size(0) == self.G * n
        acc = ins[0][self.rank * n:(self.rank + 1) * n].clone()
        for s in ins[1:]:
            acc = acc + s[self.rank * n:(self.rank + 1) * n]
        out.copy_(acc)
        self._finish()

    def broadcast(self, t, src=0, async_op=False):
        ins = self._deposit(t.clone())
        t.copy_(ins[src])
        self._finish()

    def module(self):
        m = super().module()
        m.all_reduce, m.reduce_scatter_tensor, m.broadcast = self.all_reduce, self.reduce_scatter_tensor, self.broadcast
        m.group = type("Group", (), {"WORLD": "emulated-world"})
        return m

    def run(self, fn):
        # the backward's collectives block each rank until all arrive: it must run on the rank's own thread, not on the
        # autograd engine's one worker thread for cuda:0, which every rank shares
        def on_own_thread(r):
            with torch.autograd.set_multithreading_enabled(False):
                return fn(r)
        return super().run(on_own_thread)

    def peer_exchange_class(self):
        base = super().peer_exchange_class()

        class FakePeerExchange(base):
            def __init__(self, *a, **kw):
                super().__init__(*a, **kw)
                self.side = torch.cuda.Stream()

        return FakePeerExchange


@pytest.fixture
def emulate(monkeypatch):
    def make(G, mode):
        monkeypatch.setenv("GNNFD_EXCHANGE", mode)
        world = TrainWorld(G)
        fake = world.module()
        monkeypatch.setattr(partition, "dist", fake)
        monkeypatch.setattr(fused, "dist", fake)
        monkeypatch.setattr(partition, "PeerExchange", world.peer_exchange_class())
        monkeypatch.setattr(partition, "symmetric_buffer", world.symmetric_buffer)
        return world
    return make


# ------------------------------------------------------------------------------------------------
# data, models, the single-GPU reference
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _data(graph):
    """(x [N,166], edge_index, y) on cpu: the 20K-node / 200K-edge power-law graph, or the same with a hub row (``hubs``)."""
    ei = synth.powerlaw_graph(N_BIG, E_BIG, seed=11) if graph == "powerlaw" else _edges("hubs")
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(N_BIG, K, generator=gen)
    y = (torch.rand(N_BIG, generator=gen) < 0.1).long()
    y[::7] = -1
    return x, ei.contiguous(), y


def _model(cls, num_layers, p):
    torch.manual_seed(20 + num_layers)
    return cls(K, 64, 1, num_layers=num_layers, dropout=p).train()


def _oracle_model(m):
    ref = (O.OracleGAT if isinstance(m, GAT) else O.OracleTemporalGNN)(K, 64, 1, num_layers=m.num_layers, dropout=m.dropout)
    ref.load_state_dict({k: v.detach().double().cpu() for k, v in m.state_dict().items()}, strict=True)
    return ref.double().train()


def _grads(m):
    return {n: q.grad.detach().clone() for n, q in m.named_parameters() if "lin_dst" not in n}


def _state(m):
    """Parameters after the step and the BatchNorm running statistics."""
    return {n: t.detach().clone() for n, t in m.state_dict().items() if "lin_dst" not in n and "num_batches" not in n}


def _single_gpu_step(base, x, ei, y, steps=1):
    """``steps`` steps of the single-GPU model, every layer with gemm_algo=GEMM_INPUT and the seeds the partitioned step
    uses; returns the last step's (logits, loss, grads, state after Adam)."""
    m = copy.deepcopy(base).to(x.device).train()
    N = x.size(0)
    g = GLOBAL_CSR_CACHE.get(ei, N, True, True)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=5e-4)
    for s in range(steps):
        opt.zero_grad(set_to_none=True)
        h = x
        for i, conv in enumerate(m.gat_layers):
            s_att, s_feat = InputSpaceModelTrainStep.dropout_seeds(SEED, s, i)
            z = Fn.gatconv(h, conv.lin_src.weight, conv.att_src, conv.att_dst, conv.bias, g, 8, 64, False,
                           conv.negative_slope, None, conv.dropout, torch.float32, _abi.GEMM_INPUT, seed=s_att)
            res = h if (m.residual and h.size(1) == z.size(1)) else None
            h = fused.bn_relu_dropout_residual(z, m.batch_norms[i], m.dropout, res, seed=s_feat)
        logits = fused.gru_head(h, m.gru, m.out)[0] if isinstance(m, TemporalGNN) else m.out(h)
        loss, _ = fused.masked_bce_with_logits(logits, y, 50.0)
        loss.backward()
        grads = _grads(m)
        opt.step()
    torch.cuda.synchronize()
    return logits.detach(), loss.detach(), grads, _state(m)


def _run(world, base, x, ei, y, steps=1):
    """Every rank builds the partition, its copy of ``base`` and the step, and runs ``steps`` steps."""
    N = x.size(0)

    def fn(r):
        dev = torch.device("cuda", 0)
        part = InputSpaceModelPartition.build(ei, N, r, world.G, dev)
        m = copy.deepcopy(base).cuda().train()
        step = InputSpaceModelTrainStep(part, m, _x_full(part, x), y, seed=SEED)
        for _ in range(steps):
            loss, _ = step.step()
        metrics = step.metrics()
        torch.cuda.synchronize()
        return dict(lo=step.lo, hi=step.hi, exchange=step.exchange, logits=step.logits.clone(), loss=loss.clone(),
                    grads=_grads(m), state=_state(m), metrics=metrics, n_edges=part.graph.n_edges,
                    local_ei=part.local_ei.clone(), plan=part.plan)

    return world.run(fn)


def _gather_logits(res):
    assert [rr["lo"] for rr in res[1:]] == [rr["hi"] for rr in res[:-1]] and res[0]["lo"] == 0
    return torch.cat([rr["logits"] for rr in res])


def _bit_equal_to(res, logits, loss, grads, state):
    got = _gather_logits(res)
    assert torch.equal(got, logits), ("logits", maxabs(got, logits))
    for rr in res:
        assert torch.equal(rr["loss"], loss), ("loss", float(rr["loss"]), float(loss))
        for n in grads:
            assert torch.equal(rr["grads"][n], grads[n]), (n, maxabs(rr["grads"][n], grads[n]))
        for n in state:
            assert torch.equal(rr["state"][n], state[n]), (n, maxabs(rr["state"][n], state[n]))


def _close_to(res, logits, loss, grads, state, what):
    """rel L2 <= 1e-5 for logits, loss, gradients and the BatchNorm running statistics (the conv biases feed a train-mode
    BatchNorm: their true gradient is zero, so max-abs there).  Not the parameters after the step: Adam's first update is
    +-lr wherever the gradient is far above its epsilon, so a gradient entry within rounding of zero flips the update by
    2 lr; the gradients themselves are compared, and the parameters bit for bit at one rank and across ranks."""
    errs = {"logits": relerr(_gather_logits(res), logits), "loss": relerr(res[0]["loss"].reshape(1), loss.reshape(1))}
    for n in grads:
        e = maxabs if (n.startswith("gat_layers.") and n.endswith(".bias")) else relerr
        errs["grad " + n] = max(e(rr["grads"][n], grads[n]) for rr in res)
    for n in state:
        if "running" in n:
            errs["state " + n] = max(relerr(rr["state"][n], state[n]) for rr in res)
    worst = max(errs.items(), key=lambda kv: kv[1])
    print(f"{what}: worst {worst[0]} {worst[1]:.3g}; logits {errs['logits']:.3g} loss {errs['loss']:.3g}")
    bad = {k: v for k, v in errs.items() if not v <= 1e-5}
    assert not bad, (what, bad)


CASES = [(cls, L) for cls in (GAT, TemporalGNN) for L in (1, 2, 3)]
IDS = [f"{cls.__name__}-L{L}" for cls, L in CASES]


# ------------------------------------------------------------------------------------------------
# 1. G = 1 is the single-GPU model, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("graph", ["powerlaw", "hubs"])
@pytest.mark.parametrize("cls,L", CASES, ids=IDS)
def test_one_rank_is_bit_equal_to_the_single_gpu_step(emulate, cls, L, graph, p):
    x, ei, y = (t.cuda() for t in _data(graph))
    base = _model(cls, L, p)
    ref = _single_gpu_step(base, x, ei, y)
    res = _run(emulate(1, "auto"), base, x, ei, y)
    assert res[0]["exchange"] == "none"
    _bit_equal_to(res, *ref)


# ------------------------------------------------------------------------------------------------
# 2. G > 1, dropout off: the single-GPU model and the fp64 oracle
# ------------------------------------------------------------------------------------------------
def _recording(monkeypatch):
    """Records, per rank (keyed on its first row), the input and output of every BatchNorm tail."""
    seen = {}
    real_bn = fused.bn_relu_dropout_residual

    def recording_bn(z, bn, p_drop=0.0, residual=None, seed=None, row_base=0, **kw):
        out = real_bn(z, bn, p_drop, residual, seed, row_base, **kw)
        seen.setdefault(row_base, []).append((z.detach().clone(), out.detach().clone()))
        return out

    monkeypatch.setattr(fused, "bn_relu_dropout_residual", recording_bn)
    return seen


def _leaky_from_inputs(base, ins, ei, dev):
    """The leaky-ReLU branch of every attention logit as the kernels take it: the sign of the fp32 a_src[j] + a_dst[i] from
    the logits kernel run again on the layer inputs the ranks saw (assembled in global row order; the logits of a row depend
    on that row alone), per edge of edge_index' and head."""
    N = ins[0].size(0)
    ei2 = O.rewrite_self_loops(ei.cpu(), N).to(dev)
    out = []
    for conv, h in zip(base.gat_layers, ins):
        W = conv.lin_src.weight.detach().to(dev).contiguous()
        a_s, a_d = (t.detach().reshape(-1).contiguous().to(dev) for t in (conv.att_src, conv.att_dst))
        prep = Fn._aligned_u8(Fn.in_sizes(N, h.size(1))[0], dev)
        a_src, a_dst = Fn.in_logits(Fn.in_pad_x(h), W, a_s, a_d, prep, torch.zeros(16, device=dev))
        out.append(((a_src[ei2[0]] + a_dst[ei2[1]]) > 0).cpu())
    return out


def _oracle_with_branches(res, seen, base, x, ei, y, att=None, feat=None, scale=None):
    """The fp64 oracle's step, taking the kernels' ReLU / leaky-ReLU branch where its pre-activation lies within 1e-5 of the
    kink (``test_dropout_training_gpu._oracle_step``)."""
    L, dev = base.num_layers, x.device
    zs = [torch.cat([seen[rr["lo"]][i][0] for rr in res]) for i in range(L)]
    hs = [torch.cat([seen[rr["lo"]][i][1] for rr in res]) for i in range(L)]
    follow = _relu_decisions(zs, copy.deepcopy(base.batch_norms).to(dev))      # the affine parameters before the update
    leaky = _leaky_from_inputs(base, [x] + hs[:-1], ei, dev)
    torch.set_num_threads(max(4, torch.get_num_threads()))
    lg, loss, grads, _, forced = _oracle_step(_oracle_model(base), x.double().cpu(), ei.cpu(), y.cpu(), att, feat, scale,
                                              relu_follow=follow, leaky_follow=leaky)
    print(f"({forced} branches at a kink taken from the kernels)")
    return lg, loss, grads


def _against_oracle(res, oracle, what):
    lg, loss, grads = oracle
    errs = _errors(_gather_logits(res).cpu(), float(res[0]["loss"]), {n: g.cpu() for n, g in res[0]["grads"].items()},
                   lg, loss, grads)
    print(what, "vs fp64 oracle:", {k: f"{e:.3g}" for k, (e, _) in errs.items()})
    bad = {k: e for k, (e, _) in errs.items() if not e <= 1e-5}
    assert not bad, (what, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["powerlaw", "hubs"])
@pytest.mark.parametrize("G", [2, 3, 4])
@pytest.mark.parametrize("cls,L", CASES, ids=IDS)
def test_ranks_match_the_single_gpu_step_and_the_fp64_oracle(emulate, monkeypatch, cls, L, G, graph):
    """Against the single-GPU step at every G and on both graphs; against the fp64 oracle at every G on the power-law graph
    (the hub graph's single-GPU step is checked against the oracle by the tests of the single-GPU model)."""
    x, ei, y = (t.cuda() for t in _data(graph))
    base = _model(cls, L, 0.0)
    ref = _single_gpu_step(base, x, ei, y)
    seen = _recording(monkeypatch)
    res = _run(emulate(G, "auto"), base, x, ei, y)
    assert all(rr["exchange"] == "peer" for rr in res)
    what = f"{cls.__name__} L={L} G={G} {graph}"
    _close_to(res, *ref, what=what)
    if graph == "powerlaw":
        _against_oracle(res, _oracle_with_branches(res, seen, base, x, ei, y), what)


# ------------------------------------------------------------------------------------------------
# 3. G > 1, dropout on: the fp64 oracle fed the ranks' masks
# ------------------------------------------------------------------------------------------------
def _global_attention_masks(res, ei, N, p, dev):
    """Per layer, the [E',8] attention keep-mask in edge_index' order (the surviving original edges, then one self-loop per
    node) assembled from every rank's mask over its local edge list: local position q of rank r is its q-th surviving
    original edge with a destination in r's range, or after those, the self-loop of node lo + (q - m_r)."""
    src, dst = ei[0].to(dev), ei[1].to(dev)
    surv = src != dst
    dst_s = dst[surv]
    E_s = int(surv.sum())
    pos_of = []
    for rr in res:
        mine = torch.nonzero((dst_s >= rr["lo"]) & (dst_s < rr["hi"])).view(-1)
        loops = E_s + torch.arange(rr["lo"], rr["hi"], device=dev)
        pos = torch.cat([mine, loops])
        assert pos.numel() == rr["n_edges"]
        pos_of.append(pos)
    masks = []
    for layer in range(res[0]["L"]):
        full = torch.full((E_s + N, 8), 255, dtype=torch.uint8, device=dev)
        for rr, pos in zip(res, pos_of):
            s_att, _ = InputSpaceModelTrainStep.dropout_seeds(SEED, 0, layer)
            full[pos] = Fn.dropout_mask(s_att, p, rr["n_edges"], 8, dev)[0]
        assert int((full == 255).sum()) == 0
        masks.append(full.cpu())
    return masks


def _feature_masks(L, p, N, dev):
    feat, scale = [], None
    for layer in range(L):
        _, s_feat = InputSpaceModelTrainStep.dropout_seeds(SEED, 0, layer)
        k, scale = Fn.dropout_mask(s_feat, p, N * 64, 1, dev)
        feat.append(k.view(N, 64).cpu())
    return feat, scale


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("cls", [GAT, TemporalGNN], ids=["GAT", "TemporalGNN"])
def test_dropout_ranks_match_the_fp64_oracle_given_the_ranks_masks(emulate, monkeypatch, cls, G):
    L, p = 3, 0.2
    x, ei, y = (t.cuda() for t in _data("powerlaw"))
    base = _model(cls, L, p)
    seen = _recording(monkeypatch)
    res = _run(emulate(G, "auto"), base, x, ei, y)
    for rr in res:
        rr["L"] = L
    att = _global_attention_masks(res, ei, x.size(0), p, x.device)
    feat, scale = _feature_masks(L, p, x.size(0), x.device)
    oracle = _oracle_with_branches(res, seen, base, x, ei, y, att, feat, scale)
    _against_oracle(res, oracle, f"{cls.__name__} p={p} G={G}")
    # negative control: every attention mask shifted by one edge must not pass
    wrong = [m.clone() for m in att]
    for m in wrong:
        m[:] = m.roll(1, 0)
    lg, loss, _ = _oracle_step(_oracle_model(base), x.double().cpu(), ei.cpu(), y.cpu(), wrong, feat, scale)[:3]
    assert relerr(_gather_logits(res).cpu(), lg) > 1e-4


# ------------------------------------------------------------------------------------------------
# 4. the exchange: peer == nccl, every rank ends with the same parameters
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("cls", [GAT, TemporalGNN], ids=["GAT", "TemporalGNN"])
def test_peer_exchange_equals_nccl_collectives_and_ranks_agree(emulate, cls, p):
    """Two steps at G = 3 (the second reuses every exchange buffer of the first)."""
    x, ei, y = (t.cuda() for t in _data("hubs"))
    base = _model(cls, 3, p)
    runs = {}
    for mode in ("auto", "nccl"):
        runs[mode] = _run(emulate(3, mode), base, x, ei, y, steps=2)
        assert all(rr["exchange"] == ("peer" if mode == "auto" else "nccl") for rr in runs[mode])
    a, b = runs["auto"], runs["nccl"]
    assert torch.equal(_gather_logits(a), _gather_logits(b))
    for r in range(3):
        assert torch.equal(a[r]["loss"], b[r]["loss"])
        assert a[r]["metrics"] == b[r]["metrics"] == a[0]["metrics"]
        for n in a[r]["grads"]:
            assert torch.equal(a[r]["grads"][n], b[r]["grads"][n]), (r, n, maxabs(a[r]["grads"][n], b[r]["grads"][n]))
            assert torch.equal(a[r]["grads"][n], a[0]["grads"][n]), (r, n)
        for n in a[r]["state"]:
            assert torch.equal(a[r]["state"][n], b[r]["state"][n]), (r, n)
            assert torch.equal(a[r]["state"][n], a[0]["state"][n]), (r, n)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_second_step_continues_the_single_gpu_training(emulate, p):
    """Two steps through the same buffers and optimizer at G = 1 are two single-GPU steps bit for bit (step-indexed seeds,
    Adam state, BatchNorm running statistics).  Not compared across G after the first step: Adam's first update is +-lr
    wherever a gradient is far above its epsilon, so an entry within rounding of zero (every conv bias entry: its true
    gradient is zero) takes either sign at G > 1, and the second step starts from parameters 2 lr apart there."""
    x, ei, y = (t.cuda() for t in _data("powerlaw"))
    base = _model(TemporalGNN, 3, p)
    _bit_equal_to(_run(emulate(1, "auto"), base, x, ei, y, steps=2), *_single_gpu_step(base, x, ei, y, steps=2))


# ------------------------------------------------------------------------------------------------
# 5. gnnfd_bn_relu_drop_res_fwd_bcast against gnnfd_bn_relu_drop_res_fwd
# ------------------------------------------------------------------------------------------------
def _bn_inputs(n, seed):
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(seed)
    z = (torch.randn(max(n, 1), 64, generator=gen) * 2 + 0.5).to(dev)[:n]
    mean, invstd = torch.randn(64, generator=gen).to(dev), (torch.rand(64, generator=gen) + 0.5).to(dev)
    gamma, beta = (torch.rand(64, generator=gen) + 0.5).to(dev), torch.randn(64, generator=gen).to(dev)
    res = torch.randn(max(n, 1), 64, generator=gen).to(dev)[:n]
    return z, mean, invstd, gamma, beta, res


def _bn_fwd(z, n, mean, invstd, gamma, beta, p, seed, row_base, res, out):
    return _abi.lib().gnnfd_bn_relu_drop_res_fwd(_abi.ptr(z), n, 64, mean.data_ptr(), invstd.data_ptr(), _abi.ptr(gamma),
                                                  _abi.ptr(beta), float(p), int(seed), int(row_base), _abi.ptr(res),
                                                  _abi.ptr(out), _stream())


def _bn_bcast(z, n, mean, invstd, gamma, beta, p, seed, row_base, res, peers, row_offset, mc, out):
    return _abi.lib().gnnfd_bn_relu_drop_res_fwd_bcast(_abi.ptr(z), n, 64, mean.data_ptr(), invstd.data_ptr(),
                                                        _abi.ptr(gamma), _abi.ptr(beta), float(p), int(seed), int(row_base),
                                                        _abi.ptr(res), C.byref(peers), int(row_offset), int(mc),
                                                        _abi.ptr(out), _stream())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 127, 129, 1000])
@pytest.mark.parametrize("G", [1, 3, 8])
def test_bn_bcast_stores_exactly_the_rows_of_bn_fwd_into_every_buffer(G, n):
    """Each "rank" r broadcasts the same n rows to rows [r*P, r*P + n) of G buffers (P = n + 5: padding rows between the
    ranges); every buffer gets exactly those rows, bit-equal to gnnfd_bn_relu_drop_res_fwd (dropout key, residual, affine
    included), and keeps its NaN sentinel everywhere else."""
    dev = torch.device("cuda", 0)
    P = n + 5
    z, mean, invstd, gamma, beta, res = _bn_inputs(n, seed=31 + n)
    for p, with_res, affine in ((0.0, False, True), (0.2, True, True), (0.5, True, False)):
        r_in = res if with_res else None
        g_in, b_in = (gamma, beta) if affine else (None, None)
        row_base = 1000 + 7 * n
        ref = torch.full((max(n, 1), 64), NAN, device=dev)
        assert _bn_fwd(z, n, mean, invstd, g_in, b_in, p, 99, row_base, r_in, ref) == 0
        bufs = [torch.full((G * P, 64), NAN, device=dev) for _ in range(G)]
        peers = _peer_table(bufs)
        want = torch.full((G * P, 64), NAN, device=dev)
        for r in range(G):
            own = torch.full((n + 1, 64), NAN, device=dev) if r % 2 == 0 else None      # out given on even ranks
            rc = _bn_bcast(z, n, mean, invstd, g_in, b_in, p, 99, row_base, r_in, peers, r * P, 0, own)
            torch.cuda.synchronize()
            assert rc == 0, (p, r, rc)
            want[r * P:r * P + n] = ref[:n]
            if own is not None:
                assert torch.equal(own[:n], ref[:n]), (p, r, maxabs(own[:n], ref[:n]))
                assert bool(torch.isnan(own[n:]).all()), (p, r, "out written beyond its n rows")
            for g, b in enumerate(bufs):
                assert torch.equal(b.view(torch.int32), want.view(torch.int32)), (p, r, g)


@pytest.mark.gpu
def test_bn_bcast_refuses_bad_peers_and_missing_multicast_before_launch():
    dev = torch.device("cuda", 0)
    n = 64
    z, mean, invstd, gamma, beta, res = _bn_inputs(n, seed=3)
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
            rc = _bn_bcast(z, rows, mean, invstd, gamma, beta, 0.0, 0, 0, res, p, 0, mc, out)
            torch.cuda.synchronize()
            assert rc == -1, (what, rows, rc)
            assert all(bool(torch.isnan(b).all()) for b in bufs) and bool(torch.isnan(out).all()), (what, "a buffer was written")
    assert _bn_bcast(z, 0, mean, invstd, gamma, beta, 0.0, 0, 0, res, _peer_table(bufs[:1]), 0, 0, None) == 0


# ------------------------------------------------------------------------------------------------
# 6. refusals (checked before anything touches a device: no GPU needed)
# ------------------------------------------------------------------------------------------------
def _cpu_partition(N=50):
    ei = torch.randint(0, N, (2, 200), generator=torch.Generator().manual_seed(0))
    return InputSpaceModelPartition(DstRangePlan.build(ei, N, 2), 0, torch.device("cpu"))


def test_train_step_refuses_what_it_does_not_compute(monkeypatch):
    from gnn_fraud_detection_b200 import models
    part = _cpu_partition()
    x, y = torch.zeros(part.n_pos, K), torch.zeros(50, dtype=torch.long)

    def make(m):
        return InputSpaceModelTrainStep(part, m, x, y)

    with pytest.raises(RuntimeError, match="model.train"):
        make(GAT(K, 64, 1, num_layers=2).eval())
    with pytest.raises(NotImplementedError, match="use_batch_norm"):
        make(GAT(K, 64, 1, num_layers=2, use_batch_norm=False))
    m = TemporalGNN(K, 64, 1, num_layers=2)
    m.fused_tail = False
    with pytest.raises(NotImplementedError, match="fused_tail"):
        make(m)
    for width in (32, 128):
        with pytest.raises(NotImplementedError, match="hidden_channels=64"):
            make(TemporalGNN(K, width, 1, num_layers=2))
    with pytest.raises(NotImplementedError, match="in_channels <= 192"):
        make(GAT(200, 64, 1, num_layers=2))
    with pytest.raises(NotImplementedError, match="add_self_loops"):
        make(GAT(K, 64, 1, num_layers=2, add_self_loops=False))
    with pytest.raises(TypeError, match="GAT or TemporalGNN"):
        make(torch.nn.Linear(K, 64))
    with pytest.raises(ValueError, match="x_full"):
        make(GAT(K, 64, 1, num_layers=2))                 # a CPU input
    monkeypatch.setattr(models, "_HEADS", 4)
    with pytest.raises(NotImplementedError, match="8 heads"):
        make(GAT(K, 64, 1, num_layers=2))


def test_source_pass_refuses_a_wrong_da_src_buffer():
    """``gat_bwd_src(da_src_out=)`` hands the buffer to the kernel as a raw pointer: anything but a contiguous float32
    [n_src, H] tensor on the edges' device is refused before a launch."""
    import types
    g = types.SimpleNamespace(n_src=10, n_edges=4)
    eg = torch.zeros(4, 16)
    good = torch.zeros(10, 8)
    for bad in (torch.zeros(9, 8), torch.zeros(10, 8, dtype=torch.float64), torch.zeros(8, 10).t(), torch.zeros(10, 4)):
        with pytest.raises(ValueError, match="da_src_out"):
            Fn.gat_bwd_src(g, eg[:, :8], eg[:, 8:], torch.zeros(10, 64), torch.zeros(512), torch.zeros(512), good, 8, 64,
                           False, da_src_out=bad)


# ------------------------------------------------------------------------------------------------
# 7. real ranks (>= 2 GPUs)
# ------------------------------------------------------------------------------------------------
def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        out = {}
        x, ei, y = (t.to(dev) for t in _data("hubs"))
        for cls in (GAT, TemporalGNN):
            base = _model(cls, 3, 0.0)
            lg_ref, loss_ref, grads_ref, state_ref = _single_gpu_step(base, x, ei, y)
            part = InputSpaceModelPartition.build(ei, x.size(0), rank, world, dev)
            m = copy.deepcopy(base).to(dev).train()
            step = InputSpaceModelTrainStep(part, m, _x_full(part, x), y, seed=SEED)
            loss, _ = step.step()
            torch.cuda.synchronize()
            errs = {"logits": relerr(step.logits, lg_ref[step.lo:step.hi]), "loss": relerr(loss.reshape(1), loss_ref.reshape(1))}
            for n, g in _grads(m).items():
                e = maxabs if (n.startswith("gat_layers.") and n.endswith(".bias")) else relerr
                errs["grad " + n] = e(g, grads_ref[n])
            state = _state(m)
            for n, t in state.items():
                if "running" in n:          # the parameters after Adam: see _close_to; compared across the ranks instead
                    errs["state " + n] = relerr(t, state_ref[n])
            out[cls.__name__] = (step.exchange, errs, {n: t.cpu() for n, t in state.items()})
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_real_ranks_match_the_single_gpu_step():
    """Check 2 on real ranks (NCCL, and the peer exchange where torch symmetric memory is available): logits, loss, gradients
    and BatchNorm running statistics within 1e-5 of the single-GPU step, and every rank's state after the step bit-identical."""
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, 29750 + os.getpid() % 1000, ret), nprocs=world, join=True)
    for r in range(world):
        for name, (exchange, errs, state) in ret[r].items():
            print(r, name, exchange, max(errs.values()))
            bad = {k: v for k, v in errs.items() if not v <= 1e-5}
            assert not bad, (r, name, bad)
            for n, t in state.items():         # parameters and running statistics after the step: the same bits on every rank
                assert torch.equal(t, ret[0][name][2][n]), (r, name, n)
