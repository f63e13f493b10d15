"""CPU checks of the neighbour-sampler oracle (oracle/neighbor_sampler.py), the bit-exact target of csrc/sample.cu:
a hand-worked graph, uniformity of the without-replacement draw, and the all-neighbours case against a BFS."""
import itertools

import numpy as np
import pytest
from scipy import stats

from oracle import neighbor_sampler as NS

# column: 0     1     2     3     4     5     6     7     8     9     10
# edge:   1->0  2->0  1->0  0->0  3->1  1->1  5->2  4->1  6->2  2->4  3->5
HAND_EI = np.array([[1, 2, 1, 0, 3, 1, 5, 4, 6, 2, 3],
                    [0, 0, 0, 0, 1, 1, 2, 1, 2, 4, 5]], dtype=np.int64)
HAND_N = 7


def hand_expected():
    """Seeds [0, 6] (6 has no in-edge), fanouts [4, 3, 0]: node 0 has d = 4 = k (duplicate 1->0 and self-loop 0->0 kept),
    node 1 has d = 3 = k (self-loop kept), node 2 has d = 2 < k, hop 3 has k = 0."""
    return dict(n_id=[0, 6, 1, 2, 3, 4, 5],
                edge_index=[[2, 3, 2, 0, 4, 2, 5, 6, 1],
                            [0, 0, 0, 0, 2, 2, 2, 3, 3]],
                e_id=[0, 1, 2, 3, 4, 5, 7, 6, 8],
                num_sampled_nodes=[2, 2, 3, 0], num_sampled_edges=[4, 5, 0])


def test_mix_is_splitmix64_finaliser():
    # splitmix64 sequence from state 0: next() = mix(state += 0x9E3779B97F4A7C15); first output is well known
    assert NS.mix(0x9E3779B97F4A7C15) == 0xE220A8397B1DCDAF
    assert NS.mix(0) == 0


def test_hand_built_graph():
    out = NS.neighbor_sample(HAND_EI, HAND_N, [0, 6], [4, 3, 0], seed=123)
    exp = hand_expected()
    assert out.n_id.tolist() == exp["n_id"]
    assert out.edge_index.tolist() == exp["edge_index"]
    assert out.e_id.tolist() == exp["e_id"]
    assert out.num_sampled_nodes == exp["num_sampled_nodes"] and out.num_sampled_edges == exp["num_sampled_edges"]
    assert out.batch_size == 2
    # the seed does not matter when every row is taken whole
    again = NS.neighbor_sample(HAND_EI, HAND_N, [0, 6], [4, 3, 0], seed=7)
    assert again.e_id.tolist() == exp["e_id"]


def test_hand_built_graph_subsampled_rows_and_errors():
    out = NS.neighbor_sample(HAND_EI, HAND_N, [0], [2], seed=5)       # node 0: 2 of its 4 in-edges
    assert out.num_sampled_edges == [2] and out.edge_index[1].tolist() == [0, 0]
    assert set(out.e_id.tolist()) <= {0, 1, 2, 3} and out.e_id.tolist() == sorted(out.e_id.tolist())
    empty = NS.neighbor_sample(HAND_EI, HAND_N, [], [3, 3], seed=5)
    assert empty.n_id.size == 0 and empty.num_sampled_nodes == [0, 0, 0] and empty.edge_index.shape == (2, 0)
    none = NS.neighbor_sample(np.zeros((2, 0), dtype=np.int64), 3, [2, 0], [-1, -1], seed=1)
    assert none.n_id.tolist() == [2, 0] and none.num_sampled_edges == [0, 0]
    with pytest.raises(IndexError):
        NS.neighbor_sample(HAND_EI, HAND_N, [7], [1], seed=0)
    with pytest.raises(ValueError):
        NS.neighbor_sample(HAND_EI, HAND_N, [1, 1], [1], seed=0)
    with pytest.raises(ValueError):
        NS.neighbor_sample(HAND_EI, HAND_N, [1], [-2], seed=0)


def test_selection_rules():
    assert NS.select_positions(9, 3, 5, -1) == [0, 1, 2, 3, 4]
    assert NS.select_positions(9, 3, 5, 5) == [0, 1, 2, 3, 4]
    assert NS.select_positions(9, 3, 5, 0) == []
    for seed in range(50):
        p = NS.select_positions(seed, 11, 40, 7)
        assert len(p) == 7 and len(set(p)) == 7 and p == sorted(p) and 0 <= p[0] and p[-1] < 40
    # a node's sample depends on (seed, v) only
    assert NS.select_positions(1, 2, 30, 4) == NS.select_positions(1, 2, 30, 4)
    assert any(NS.select_positions(1, v, 30, 4) != NS.select_positions(1, 2, 30, 4) for v in range(3, 8))


def test_uniform_without_replacement():
    """d = 6, k = 2: the 15 subsets are equally likely (chi-square over 3000 fixed seeds)."""
    subsets = {s: i for i, s in enumerate(itertools.combinations(range(6), 2))}
    counts = np.zeros(len(subsets))
    for seed in range(3000):
        counts[subsets[tuple(NS.select_positions(seed, 17, 6, 2))]] += 1
    assert stats.chisquare(counts).pvalue > 1e-3


def _bfs_in(ei, n, seeds, hops):
    """distance (in reversed edges) of every node within `hops` of the seeds"""
    dist = {int(s): 0 for s in seeds}
    front = list(dist)
    for h in range(1, hops + 1):
        nxt = []
        for v in front:
            for s in ei[0][ei[1] == v]:
                if int(s) not in dist:
                    dist[int(s)] = h
                    nxt.append(int(s))
        front = nxt
    return dist


@pytest.mark.parametrize("hops", [1, 2, 3])
def test_all_neighbours_is_the_bfs_neighbourhood(hops):
    rng = np.random.default_rng(hops)
    n = 300
    ei = rng.integers(0, n, size=(2, 900))
    seeds = rng.choice(n, size=12, replace=False)
    out = NS.neighbor_sample(ei, n, seeds, [-1] * hops, seed=3)
    dist = _bfs_in(ei, n, seeds, hops)
    assert out.n_id[:12].tolist() == seeds.tolist()
    assert set(out.n_id.tolist()) == set(dist) and len(out.n_id) == len(dist)
    inner = {v for v, d in dist.items() if d < hops}
    assert sorted(out.e_id.tolist()) == [e for e in range(ei.shape[1]) if int(ei[1, e]) in inner]
    # relabelled edges map back to the input edges; destinations are non-decreasing
    assert np.array_equal(out.n_id[out.edge_index], ei[:, out.e_id])
    assert np.all(np.diff(out.edge_index[1]) >= 0)
    # node groups: hop h's new nodes are exactly those at distance h
    start = 0
    for h, c in enumerate(out.num_sampled_nodes):
        assert {dist[int(v)] for v in out.n_id[start:start + c]} <= {h}
        start += c
