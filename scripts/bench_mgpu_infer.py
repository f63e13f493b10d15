"""Whole-model inference across GPUs: a 3-layer GAT (eval, no_grad) on the 200M-edge power-law graph (N = 20M, K = 166)
through ``partition.InputSpaceModelPartition``, one process per GPU:

    torchrun --nproc_per_node G scripts/bench_mgpu_infer.py [--out FILE]      (G = 1 also runs without torchrun)

Per layer the time is split with CUDA events into logits + exchange (``in_logits_bcast``, barrier, xmax reduce,
``in_prepare``), aggregation (``in_fwd``) and output GEMM + broadcast (``in_out_bcast``, barrier); the forward's wall time is
the slowest rank's.  At G = 1 the single-GPU ``model.eval()`` forward is timed beside it, default and with
``gemm_algo=GEMM_INPUT`` on every layer.  Before the timed region every rank checks its rows of a 200K-node graph against the
single-GPU model (GEMM_INPUT on every layer).  Prints one JSON line (rank 0), with the card's name and power limit read in
the same run; ``--out`` also writes it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gnn_fraud_detection_b200 import GAT, _abi, functional as Fn, synth  # noqa: E402
from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE  # noqa: E402
from gnn_fraud_detection_b200.partition import InputSpaceModelPartition  # noqa: E402

STAGES = ("logits_exchange", "aggregate", "out_gemm_bcast")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return {"name": torch.cuda.get_device_name(), "power_limit_and_max_sm_clock": q}


def x_full(part, x16):
    """x (padded rows) replicated in padded position space, with the same padded row layout."""
    K = x16.size(1)
    pos = part.plan.to_pos(torch.arange(x16.size(0), device=x16.device))
    xf = torch.zeros(part.n_pos, Fn.in_sizes(0, K)[3], device=x16.device)
    xf[pos, :K] = x16
    return xf[:, :K]


def graph(N, E, K, dev):
    ei = synth.powerlaw_graph(N, E, seed=1234, device=dev)
    x = torch.randn(N, K, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    return ei, Fn.in_pad_x(x)


def model(K, L, dev):
    torch.manual_seed(0)
    m = GAT(K, 64, 1, num_layers=L).eval()
    g = torch.Generator().manual_seed(1)
    for bn in m.batch_norms:          # trained-looking running statistics
        bn.running_mean.copy_(torch.randn(64, generator=g) * 0.1)
        bn.running_var.copy_(torch.rand(64, generator=g) + 0.5)
    return m.to(dev)


def single_gpu(m, x, ei, algo):
    old = [c.gemm_algo for c in m.gat_layers]
    for c in m.gat_layers:
        c.gemm_algo = algo if algo is not None else c.gemm_algo
    try:
        with torch.no_grad():
            return m(x, ei)
    finally:
        for c, a in zip(m.gat_layers, old):
            c.gemm_algo = a


def barrier(G):
    if G > 1:
        dist.barrier()


def wall_max(t, G, dev):
    if G == 1:
        return t
    v = torch.tensor([t], device=dev)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return float(v.item())


def selfcheck(args, rank, G, dev):
    N = args.check_nodes
    ei, x16 = graph(N, 10 * N, args.feats, dev)
    m = model(args.feats, args.layers, dev)
    ref = single_gpu(m, x16, ei, _abi.GEMM_INPUT)
    part = InputSpaceModelPartition.build(ei, N, rank, G, dev)
    (out, (lo, hi)) = part.forward(m, x_full(part, x16))
    err = wall_max(float((out - ref[lo:hi]).abs().max()) if hi > lo else 0.0, G, dev)
    del part
    GLOBAL_CSR_CACHE.clear()
    return err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=20_000_000)
    ap.add_argument("--edges", type=int, default=200_000_000)
    ap.add_argument("--feats", type=int, default=166)
    ap.add_argument("--layers", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check-nodes", type=int, default=200_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    G = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if G > 1:
        dist.init_process_group("nccl", device_id=dev)
    res = {"what": f"{args.layers}-layer GAT eval forward, power-law graph N={args.nodes} E={args.edges} K={args.feats}",
           "gpus": G, "card": card()}
    res["selfcheck_maxabs_vs_1gpu"] = selfcheck(args, rank, G, dev)
    torch.cuda.empty_cache()

    N, L = args.nodes, args.layers
    ei, x16 = graph(N, args.edges, args.feats, dev)
    m = model(args.feats, L, dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    part = InputSpaceModelPartition.build(ei, N, rank, G, dev)
    xf = x16 if G == 1 else x_full(part, x16)      # at G = 1 position space is the id space
    if G > 1:
        del x16
    torch.cuda.synchronize()
    res["partition_build_s"] = time.perf_counter() - t0
    marks = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(L)]
    for _ in range(args.warmup):
        part.forward(m, xf)
    torch.cuda.synchronize()
    barrier(G)
    stage_ms = [[0.0] * 3 for _ in range(L)]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        part.forward(m, xf, marks=marks)
        torch.cuda.synchronize()
        for i in range(L):
            for s in range(3):
                stage_ms[i][s] += marks[i][s].elapsed_time(marks[i][s + 1]) / args.steps
    res["forward_ms"] = wall_max((time.perf_counter() - t0) / args.steps * 1e3, G, dev)
    res["exchange"] = part.exchange
    res["rank0_rows"] = part.n_local
    res["rank0_stage_ms"] = [dict(zip(STAGES, s)) for s in stage_ms]
    # NVLink bytes a rank sends per forward: its h rows (256 B) and a_src rows (32 B) to every other rank, every layer
    res["nvlink_bytes_sent_per_rank"] = L * part.n_local * (64 + 8) * 4 * (G - 1)
    res["peak_mem_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
    del part
    torch.cuda.empty_cache()
    if G == 1:
        for name, algo in (("single_gpu_default_ms", None), ("single_gpu_gemm_input_ms", _abi.GEMM_INPUT)):
            for _ in range(args.warmup):
                single_gpu(m, xf, ei, algo)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                single_gpu(m, xf, ei, algo)
            torch.cuda.synchronize()
            res[name] = (time.perf_counter() - t0) / args.steps * 1e3
    else:
        res["single_gpu"] = "timed in the G = 1 run"
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if G > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
