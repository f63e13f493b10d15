"""Neighbour sampler (csrc/sample.cu through NeighborSampler / NeighborLoader) against the oracle restatement of its
contract (oracle/neighbor_sampler.py): index work, so every comparison of a sample is bit-exact; then the sampled
subgraphs through the models (seed-set inference against the full graph, one training step against the fp64 oracle)."""
import ctypes as C
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from gnn_fraud_detection_b200 import GAT, NeighborLoader, NeighborSampler, TemporalGNN, _abi, synth
from oracle import neighbor_sampler as NS
from oracle import pyg_gatconv as O
from test_sampler import HAND_EI, HAND_N, hand_expected
from util import load_ckpt, maxabs, relerr

pytestmark = pytest.mark.gpu


def _check(sampler, ei_cpu, n, seeds, fanouts, seed, csr=None):
    """GPU sample == oracle sample, bit for bit; node_map is clean afterwards.  Returns the GPU sample."""
    out = sampler.sample(torch.as_tensor(seeds, dtype=torch.int64).cuda(), seed=seed)
    ref = NS.neighbor_sample(ei_cpu, n, seeds, fanouts, seed, csr=csr)
    assert np.array_equal(out.n_id.cpu().numpy(), ref.n_id)
    assert np.array_equal(out.edge_index.cpu().numpy(), ref.edge_index)
    assert np.array_equal(out.e_id.cpu().numpy(), ref.e_id)
    assert out.num_sampled_nodes == ref.num_sampled_nodes and out.num_sampled_edges == ref.num_sampled_edges
    assert out.batch_size == len(seeds)
    assert bool((sampler.node_map == -1).all())
    return out


def test_hand_built_graph_matches_hand_written_expectation():
    s = NeighborSampler(torch.from_numpy(HAND_EI).cuda(), HAND_N, [4, 3, 0])
    out = _check(s, HAND_EI, HAND_N, [0, 6], [4, 3, 0], seed=123)
    exp = hand_expected()
    assert out.n_id.tolist() == exp["n_id"] and out.edge_index.tolist() == exp["edge_index"]
    assert out.e_id.tolist() == exp["e_id"]
    for fan in ([2], [1, 1, 1], [-1, -1], [0]):                    # sub-sampled rows of the same graph
        s = NeighborSampler(torch.from_numpy(HAND_EI).cuda(), HAND_N, fan)
        for seed in range(5):
            _check(s, HAND_EI, HAND_N, [0, 5, 1], fan, seed)
    s = NeighborSampler(torch.from_numpy(HAND_EI).cuda(), HAND_N, [3, 3])
    _check(s, HAND_EI, HAND_N, [], [3, 3], seed=1)                  # empty seed set
    e0 = np.zeros((2, 0), dtype=np.int64)
    s = NeighborSampler(torch.from_numpy(e0).cuda(), 4, [-1, 5])    # no edges at all
    _check(s, e0, 4, [3, 0], [-1, 5], seed=1)


@pytest.mark.parametrize("fanouts", [[3, 5, 2], [-1, 2], [40, 50], [1]])
def test_random_graph_with_self_loops_matches_oracle(fanouts):
    n = 400 if fanouts != [40, 50] else 300
    ei = synth.random_graph(n, 30_000 if fanouts == [40, 50] else 2_000, seed=4, self_loops=True)
    assert bool((ei[0] == ei[1]).any())
    s = NeighborSampler(ei.cuda(), n, fanouts)
    csr = NS.raw_csr(ei.numpy(), n)
    rng = np.random.default_rng(0)
    for b in range(3):
        seeds = rng.choice(n, size=[1, 17, 60][b], replace=False)
        _check(s, ei.numpy(), n, seeds, fanouts, seed=b * 977 + 5, csr=csr)


def test_elliptic_shape_batches_match_oracle():
    _, ei, _ = synth.elliptic_synth(seed=0)
    n = synth.ELLIPTIC_NODES
    s = NeighborSampler(ei.cuda(), n, [10, 10, 10])
    csr = NS.raw_csr(ei.numpy(), n)
    starts = [0, 256, 512, (n // 256) * 256]                        # first three batches of 256 and the last partial one
    for i, st in enumerate(starts):
        seeds = np.arange(st, min(st + 256, n))
        out = _check(s, ei.numpy(), n, seeds, [10, 10, 10], seed=1000 + i, csr=csr)
        assert out.num_sampled_edges[0] > 0
    assert len(seeds) == n - (n // 256) * 256 < 256


@pytest.mark.parametrize("fanouts", [[10, 10], [-1, 2]])
def test_hub_of_in_degree_above_2_17(fanouts):
    g = torch.Generator().manual_seed(11)
    n, hub, deg = 200_000, 7, (1 << 17) + 8_000
    hub_edges = torch.stack([torch.randint(0, n, (deg,), generator=g), torch.full((deg,), hub)])
    background = torch.randint(0, n, (2, 60_000), generator=g)
    ei = torch.cat([hub_edges, background], 1)
    ei = ei[:, torch.randperm(ei.size(1), generator=g)].contiguous()
    s = NeighborSampler(ei.cuda(), n, fanouts)
    assert s.max_degree >= deg
    seeds = np.concatenate([[hub], np.random.default_rng(1).choice(np.arange(8, n), size=20, replace=False)])
    out = _check(s, ei.numpy(), n, seeds, fanouts, seed=99, csr=NS.raw_csr(ei.numpy(), n))
    assert out.num_sampled_edges[0] >= (deg if fanouts[0] == -1 else 10)


def test_determinism_and_independence_of_batch_and_hop():
    n = 2_000
    ei = synth.random_graph(n, 20_000, seed=8)
    s = NeighborSampler(ei.cuda(), n, [4, 4])
    seeds = torch.arange(0, 50, device="cuda")
    a, b, c = s.sample(seeds, seed=5), s.sample(seeds, seed=5), s.sample(seeds, seed=6)
    assert torch.equal(a.n_id, b.n_id) and torch.equal(a.edge_index, b.edge_index) and torch.equal(a.e_id, b.e_id)
    assert not torch.equal(a.e_id, c.e_id)
    torch.manual_seed(3)
    d = s.sample(seeds)
    torch.manual_seed(3)
    assert torch.equal(s.sample(seeds).e_id, d.e_id)                 # seed=None draws from torch's CPU generator

    def picks(out):
        """global node -> e_ids of its expansion, for every node expanded in this sample"""
        n_front = sum(out.num_sampled_nodes[:-1])
        dst, e = out.edge_index[1].cpu(), out.e_id.cpu()
        return {int(out.n_id[i]): sorted(e[dst == i].tolist()) for i in range(n_front)}

    # the nodes `a` expanded in hop 2 are the seeds (expanded in hop 1) of another batch
    pa = picks(a)
    hop1 = a.n_id[50:50 + a.num_sampled_nodes[1]]
    po = picks(s.sample(hop1, seed=5))
    common = set(pa) & set(po)
    assert len(common) >= hop1.numel() >= 50
    assert all(pa[v] == po[v] for v in common)


def _raw_call(s, seeds, fanouts, node_cap, edge_cap):
    lib = _abi.lib()
    L = len(fanouts)
    nb = C.c_size_t()
    _abi.check(lib.gnnfd_sample_workspace_bytes(node_cap, edge_cap, L, C.byref(nb)))
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    n_id = torch.empty(max(node_cap, 1), dtype=torch.int64, device="cuda")
    eo = torch.empty(2, max(edge_cap, 1), dtype=torch.int64, device="cuda")
    e_id = torch.empty(max(edge_cap, 1), dtype=torch.int64, device="cuda")
    counts = (C.c_int64 * (3 + 2 * L))()
    g = s.graph
    return lib.gnnfd_neighbor_sample(g.rowptr.data_ptr(), g.col.data_ptr(), g.perm.data_ptr(), s.num_nodes, seeds.data_ptr(),
                                     seeds.numel(), (C.c_int32 * L)(*fanouts), L, 3, s.node_map.data_ptr(), n_id.data_ptr(),
                                     node_cap, eo.data_ptr(), max(edge_cap, 1), e_id.data_ptr(), edge_cap, counts,
                                     ws.data_ptr(), nb.value, torch.cuda.current_stream().cuda_stream)


def test_errors_leave_node_map_clean():
    ei = torch.from_numpy(HAND_EI).cuda()
    s = NeighborSampler(ei, HAND_N, [2, 2])
    clean = lambda: bool((s.node_map == -1).all())                    # noqa: E731
    for bad in ([0, HAND_N], [-1, 2], [2, 10 ** 9]):
        with pytest.raises(_abi.GnnfdError, match="outside") as e:
            s.sample(torch.tensor(bad, device="cuda"), seed=1)
        assert e.value.code == -4 and clean()
    with pytest.raises(_abi.GnnfdError, match="duplicate") as e:
        s.sample(torch.tensor([1, 4, 0, 4], device="cuda"), seed=1)
    assert e.value.code == -1 and clean()
    s.sample(torch.tensor([1, 4, 0], device="cuda"), seed=1)           # and the sampler still works
    assert clean()
    seeds = torch.tensor([0], device="cuda")
    assert _raw_call(s, seeds, [-2], 4, 4) == -1 and b"< -1" in _abi.lib().gnnfd_last_error() and clean()
    # too small output capacities: refused without writing beyond them, node_map restored
    assert _raw_call(s, seeds, [-1], 8, 3) == -3 and clean()           # node 0 has 4 in-edges
    assert _raw_call(s, seeds, [-1], 2, 8) == -3 and clean()           # ... from 2 new nodes: 3 nodes in all
    assert _raw_call(s, seeds, [-1], 3, 4) == 0 and clean()
    with pytest.raises(ValueError):
        NeighborSampler(ei, HAND_N, [3, -2])
    with pytest.raises(RuntimeError, match="CUDA"):
        NeighborSampler(ei.cpu(), HAND_N, [2])
    with pytest.raises(RuntimeError, match="CUDA"):
        s.sample(torch.tensor([0]), seed=1)
    x = torch.randn(HAND_N, 3, device="cuda")
    with pytest.raises(RuntimeError, match="CUDA"):
        NeighborLoader(SimpleNamespace(x=x.cpu(), edge_index=ei.cpu()), [2])
    for opt in (dict(replace=True), dict(directed=False), dict(time_attr="t"), dict(disjoint=True)):
        with pytest.raises(NotImplementedError):
            NeighborLoader(SimpleNamespace(x=x, edge_index=ei), [2], **opt)


@pytest.mark.parametrize("shuffle", [False, True])
@pytest.mark.parametrize("drop_last", [False, True])
def test_loader_covers_input_nodes_once(shuffle, drop_last):
    x, ei, ts = synth.elliptic_synth(num_nodes=5_000, num_edges=9_000, num_feats=7, num_steps=5, seed=2)
    y = torch.randint(-1, 2, (x.size(0),), generator=torch.Generator().manual_seed(0))
    data = SimpleNamespace(x=x.cuda(), edge_index=ei.cuda(), y=y.cuda(), time_steps=ts.cuda())
    mask = torch.rand(x.size(0), generator=torch.Generator().manual_seed(1)) < 0.3
    for inp in (mask, torch.nonzero(mask).reshape(-1).cuda()):
        torch.manual_seed(0)
        loader = NeighborLoader(data, [10, 10, 10], input_nodes=inp, batch_size=256, shuffle=shuffle, drop_last=drop_last)
        n_in = int(mask.sum())
        assert len(loader) == (n_in // 256 if drop_last else -(-n_in // 256))
        seen = []
        for batch in loader:
            bs = batch.batch_size
            assert bs == 256 or (not drop_last and bs == n_in % 256)
            assert torch.equal(batch.n_id[:bs], loader.input_nodes[batch.input_id])
            assert torch.equal(batch.x, data.x[batch.n_id]) and torch.equal(batch.y, data.y[batch.n_id])
            assert torch.equal(batch.time_steps, data.time_steps[batch.n_id])
            assert torch.equal(batch.n_id[batch.edge_index], data.edge_index[:, batch.e_id])
            assert sum(batch.num_sampled_nodes) == batch.n_id.numel() and sum(batch.num_sampled_edges) == batch.e_id.numel()
            seen.append(batch.n_id[:bs].cpu())
        seen = torch.cat(seen)
        assert seen.numel() == (len(loader) * 256 if drop_last else n_in)
        assert seen.unique().numel() == seen.numel()
        assert set(seen.tolist()) <= set(torch.nonzero(mask).reshape(-1).tolist())
        if not shuffle:
            assert torch.equal(seen, torch.nonzero(mask).reshape(-1)[:seen.numel()])


def test_seed_set_inference_equals_full_graph(golden_dir):
    """[-1,-1,-1]: the seeds' 3-hop receptive field is complete and every row keeps its edge order, so a 3-layer model
    on the sampled subgraph gives the seeds the logits the whole graph gives them."""
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=50_000, num_feats=165, num_steps=4, seed=5)
    x, ei = x.cuda(), ei.cuda()
    seeds = torch.randperm(x.size(0), generator=torch.Generator().manual_seed(2))[:64].cuda()
    batch = NeighborSampler(ei, x.size(0), [-1, -1, -1]).sample(seeds, seed=0)
    assert batch.n_id.numel() > 10 * 64
    bs, xs = batch.batch_size, x[batch.n_id]
    for cls, ck in ((GAT, "gat_ckpt.npz"), (TemporalGNN, "tgn_ckpt.npz")):
        m = load_ckpt(cls(165, 64, 1, num_layers=3), os.path.join(golden_dir, ck)).cuda().eval()
        with torch.no_grad():
            full, sub = m(x, ei), m(xs, batch.edge_index)
        if cls is TemporalGNN:
            assert maxabs(sub[1][:bs], full[1][seeds]) <= 1e-5
            full, sub = full[0], sub[0]
        err = maxabs(sub[:bs], full[seeds])
        print(f"seed-set inference {cls.__name__}: max-abs {err:.3e}")
        assert err <= 1e-5


def test_training_step_on_sampled_batch_matches_oracle():
    """One mini-batch step (dropout 0, train-mode BatchNorm over the sampled nodes, loss over the seed rows) against the
    oracle wrappers evaluated in fp64 on the same subgraph."""
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    loader = NeighborLoader(SimpleNamespace(x=x.cuda(), edge_index=ei.cuda()), [10, 10, 10], batch_size=256, shuffle=True)
    torch.manual_seed(0)
    batch = next(iter(loader))
    bs = batch.batch_size
    ref = O.OracleGAT(166, 64, 1, num_layers=3, dropout=0.0).double()
    ours = GAT(166, 64, 1, num_layers=3, dropout=0.0)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    ours = ours.cuda()
    y = (torch.rand(batch.n_id.numel(), 1, generator=torch.Generator().manual_seed(1)) < 0.1).float()
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0))
    xr, er = batch.x.cpu().double(), batch.edge_index.cpu()
    logits_ref = ref(xr, er)
    lr = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0).double())(logits_ref[:bs], y[:bs].double())
    lr.backward()
    logits = ours(batch.x, batch.edge_index)
    lo = crit.cuda()(logits[:bs], y[:bs].cuda())
    lo.backward()
    dloss = abs(lr.item() - lo.item())
    print(f"sampled step: loss {dloss:.3e}, logits max-abs {maxabs(logits, logits_ref):.3e} "
          f"rel {relerr(logits, logits_ref):.3e}")
    bad = []
    for (n, p_ref), (_, p_our) in zip(ref.named_parameters(), ours.named_parameters()):
        ma, re = maxabs(p_our.grad, p_ref.grad), relerr(p_our.grad, p_ref.grad)
        print(f"  {n}: max-abs {ma:.3e} rel {re:.3e}")
        # (the pre-BatchNorm conv biases have an exactly-zero true gradient: no relative error for them)
        if ma > 1e-5 or (float(p_ref.grad.norm()) > 1e-6 and re > 1e-5):
            bad.append(n)
    assert dloss <= 1e-5
    assert maxabs(logits, logits_ref) <= 1e-5 and relerr(logits, logits_ref) <= 1e-5
    assert not bad, bad


def test_seed_count_beyond_one_thread_per_seed_grid():
    """More seeds than the capped seed-registration grid has threads (16 blocks of 256 per SM): every seed is registered."""
    cap = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256
    B = cap + 50_000
    n = B + 100_000
    ei = synth.random_graph(n, 2 * n, seed=12)
    s = NeighborSampler(ei.cuda(), n, [2])
    seeds = torch.randperm(n, generator=torch.Generator().manual_seed(3))[:B].numpy()
    out = _check(s, ei.numpy(), n, seeds, [2], seed=17)
    assert out.n_id[:B].cpu().numpy().tolist() == seeds.tolist()
