"""Neighbour-sampler timings (not the headline metric): NeighborSampler batches/s and sampled edges/s, and one mini-batch
training step through NeighborLoader (sampler + feature gather + 3-layer GAT forward/backward + Adam), on two workloads:

  elliptic  -- the Elliptic-shaped graph (203,769 nodes, 234,355 edges, 166 features), num_neighbors=[10,10,10], batch 256:
               the reference's --use_subgraph_sampling configuration (src/data/dataloader.py:42-66);
  powerlaw  -- the power-law family at 2M nodes / 20M edges, [10,10,10], batch 1024: the CSR alone (168 MB) exceeds the
               126 MB L2, so the sampler's row reads come from HBM.

Beside them, the oracle port of the same sampler (oracle/neighbor_sampler.py: pure Python, one host core) on the same
graphs -- a restatement of the contract, not pyg-lib, which is not installed.  One JSON line on stdout.
Run from the repository root: python scripts/bench_sampler.py [--steps K] [--warmup W] [--oracle-batches B]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from gnn_fraud_detection_b200 import GAT, NeighborLoader, NeighborSampler, _abi, synth  # noqa: E402
from oracle import neighbor_sampler as NS  # noqa: E402

FANOUTS = [10, 10, 10]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # the number is reported without it, labelled unknown
        q = f"unknown ({type(e).__name__})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def timed(fn, n):
    """(CUDA-event ms, host wall ms) per call over n calls; every call ends in a device synchronisation."""
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    return a.elapsed_time(b) / n, wall / n


def workload(name, x, ei, batch, args):
    N, E = x.size(0), ei.size(1)
    dev = torch.device("cuda")
    x, ei = x.to(dev), ei.to(dev)
    y = (torch.rand(N, generator=torch.Generator().manual_seed(1)) < 0.1).float().to(dev)
    res = {"graph": f"{name}: N={N} E={E} K={x.size(1)}", "num_neighbors": FANOUTS, "batch_size": batch}

    # sampler alone: consecutive batches of a fixed shuffled order of all nodes
    sampler = NeighborSampler(ei, N, FANOUTS)
    order = torch.randperm(N, generator=torch.Generator().manual_seed(0)).to(dev)
    n_batches = N // batch
    state = {"b": 0, "edges": 0, "nodes": 0}

    def one():
        b = state["b"] % n_batches
        s = sampler.sample(order[b * batch:(b + 1) * batch], seed=b)
        state["b"] += 1
        state["edges"] += s.e_id.numel()
        state["nodes"] += s.n_id.numel()

    for _ in range(args.warmup):
        one()
    state.update(edges=0, nodes=0)
    l0 = _abi.lib().gnnfd_launch_count()
    ev, wall = timed(one, args.steps)
    launches = (_abi.lib().gnnfd_launch_count() - l0) / args.steps
    edges, nodes = state["edges"] / args.steps, state["nodes"] / args.steps
    res["sampler"] = {"ms_per_batch_events": round(ev, 4), "ms_per_batch_wall": round(wall, 4),
                      "batches_per_s": round(1e3 / wall, 1), "sampled_edges_per_s": round(edges * 1e3 / wall, 1),
                      "mean_sampled_edges": round(edges, 1), "mean_sampled_nodes": round(nodes, 1),
                      "kernel_launches_per_batch": launches}

    # one mini-batch training step through the loader
    torch.manual_seed(0)
    model = GAT(x.size(1), 64, 1, num_layers=3).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-4)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, device=dev))
    loader = NeighborLoader(SimpleNamespace(x=x, edge_index=ei, y=y), FANOUTS, batch_size=batch, shuffle=True)
    it = {"it": iter(loader)}

    def step():
        try:
            bt = next(it["it"])
        except StopIteration:
            it["it"] = iter(loader)
            bt = next(it["it"])
        opt.zero_grad(set_to_none=True)
        loss = crit(model(bt.x, bt.edge_index)[:bt.batch_size, 0], bt.y[:bt.batch_size])
        loss.backward()
        opt.step()
        return loss

    for _ in range(args.warmup):
        step()
    ev, wall = timed(step, args.steps)
    res["train_step"] = {"what": "NeighborLoader batch (sampler + x/y gather) + GAT(3 layers, 8 heads x 64) fwd/bwd + Adam",
                         "ms_per_step_events": round(ev, 4), "ms_per_step_wall": round(wall, 4)}

    # the oracle port on the host
    csr = NS.raw_csr(ei.cpu().numpy(), N)
    order_cpu = order.cpu().numpy()
    t0 = time.perf_counter()
    o_edges = 0
    for b in range(args.oracle_batches):
        o = NS.neighbor_sample(None, N, order_cpu[b * batch:(b + 1) * batch], FANOUTS, b, csr=csr)
        o_edges += o.e_id.size
    dt = time.perf_counter() - t0
    res["oracle_port_host"] = {"kind": "oracle port (pure Python, one host core), not pyg-lib",
                               "host_cores_available": os.cpu_count(), "batches": args.oracle_batches,
                               "ms_per_batch": round(dt * 1e3 / args.oracle_batches, 2),
                               "batches_per_s": round(args.oracle_batches / dt, 3),
                               "sampled_edges_per_s": round(o_edges / dt, 1)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--oracle-batches", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampler.py measures the CUDA sampler: no CUDA device")
    torch.cuda.set_device(0)
    out = {"metric": "neighbor_sampler", "card": card(), "workloads": {}}
    x, ei, _ = synth.elliptic_synth(seed=0)
    out["workloads"]["elliptic"] = workload("elliptic_synth", x, ei, 256, args)
    del x, ei
    n, e = 2_000_000, 20_000_000
    ei = synth.powerlaw_graph(n, e, seed=1234, device="cuda")
    x = torch.randn(n, synth.ELLIPTIC_FEATS, generator=torch.Generator(device="cuda").manual_seed(0), device="cuda")
    out["workloads"]["powerlaw_20m"] = workload("powerlaw_graph", x, ei, 1024, args)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
