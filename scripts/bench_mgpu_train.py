"""Whole-model training across GPUs: one full-batch step (forward, masked BCE, backward, gradient all-reduce, Adam) of a
3-layer GAT (dropout 0.2) on a power-law graph (K = 166) through ``partition.InputSpaceModelTrainStep``, one process per GPU:

    torchrun --nproc_per_node G scripts/bench_mgpu_train.py [--nodes N --edges E] [--out FILE]   (G = 1 runs without torchrun)

Reports the milliseconds per step (CUDA events around each step after warm-up; the slowest rank's), rank 0's per-layer split
(forward: logits + exchange, aggregation, output GEMM + BatchNorm + broadcast; backward: edge pass, source pass (dxw_part /
da_src_part), parameter gradients with the da_src exchange, dx GEMM + reduce), the span from the head to the end of Adam
(which contains the whole backward), and the peak memory per rank.  At G = 1 the
single-GPU model (``gemm_algo=GEMM_INPUT`` on every layer, eager, Adam) is timed beside it, and the backward's last stage is
the dx GEMM over all n_pos positions alone.  A graph that does not fit is reported as such (``out_of_memory``).  Before the
timed region every rank checks the step's loss on a 200K-node graph against the single-GPU model at dropout 0.  Prints one
JSON line (rank 0), with the card's name and power limit read in the same run; ``--out`` also writes it.
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
from gnn_fraud_detection_b200 import GAT, _abi, fused, functional as Fn, synth  # noqa: E402
from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE  # noqa: E402
from gnn_fraud_detection_b200.partition import InputSpaceModelPartition, InputSpaceModelTrainStep  # noqa: E402

FWD = ("logits_exchange", "aggregate", "out_gemm_bn_bcast")
BWD = ("bwd_edges", "bwd_src_pass", "params_da_exchange", "dx_gemm_reduce")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return {"name": torch.cuda.get_device_name(), "power_limit_and_max_sm_clock": q}


def data(N, E, K, dev):
    ei = synth.powerlaw_graph(N, E, seed=1234, device=dev)
    x = torch.randn(N, K, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    y = (torch.rand(N, generator=torch.Generator(device=dev).manual_seed(6), device=dev) < 0.1).long()
    y[::7] = -1
    return ei, Fn.in_pad_x(x), y


def x_full(part, x16):
    K = x16.size(1)
    pos = part.plan.to_pos(torch.arange(x16.size(0), device=x16.device))
    xf = torch.zeros(part.n_pos, Fn.in_sizes(0, K)[3], device=x16.device)
    xf[pos, :K] = x16
    return xf[:, :K]


def model(K, L, p, dev):
    torch.manual_seed(0)
    return GAT(K, 64, 1, num_layers=L, dropout=p).to(dev).train()


def single_gpu_step(m, opt, x, ei, y):
    opt.zero_grad(set_to_none=True)
    loss, _ = fused.masked_bce_with_logits(m(x, ei), y, 50.0)
    loss.backward()
    opt.step()
    return loss.detach()


def wall_max(t, G, dev):
    if G == 1:
        return t
    v = torch.tensor([t], device=dev)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return float(v.item())


def selfcheck(args, rank, G, dev):
    N = args.check_nodes
    ei, x16, y = data(N, 10 * N, args.feats, dev)
    m = model(args.feats, args.layers, 0.0, dev)
    ref = model(args.feats, args.layers, 0.0, dev)
    for c in ref.gat_layers:
        c.gemm_algo = _abi.GEMM_INPUT
    loss_ref = single_gpu_step(ref, torch.optim.Adam(ref.parameters(), lr=1e-3, weight_decay=5e-4), x16, ei, y)
    part = InputSpaceModelPartition.build(ei, N, rank, G, dev)
    loss, _ = InputSpaceModelTrainStep(part, m, x_full(part, x16), y).step()
    err = wall_max(float((loss - loss_ref).abs() / loss_ref.abs()), G, dev)
    del part
    GLOBAL_CSR_CACHE.clear()
    return err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=20_000_000)
    ap.add_argument("--edges", type=int, default=200_000_000)
    ap.add_argument("--feats", type=int, default=166)
    ap.add_argument("--layers", type=int, default=3)
    ap.add_argument("--dropout", type=float, default=0.2)
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
    N, L = args.nodes, args.layers
    res = {"what": f"{L}-layer GAT training step (dropout {args.dropout}, Adam), power-law graph N={N} E={args.edges} "
                   f"K={args.feats}", "gpus": G, "card": card()}
    res["selfcheck_loss_rel_vs_1gpu"] = selfcheck(args, rank, G, dev)
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    ei, x16, y = data(N, args.edges, args.feats, dev)
    m = model(args.feats, L, args.dropout, dev)
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        part = InputSpaceModelPartition.build(ei, N, rank, G, dev)
        xf = x16 if part.n_pos == N else x_full(part, x16)     # one range, no padding: position space is the id space
        step = InputSpaceModelTrainStep(part, m, xf, y)
        torch.cuda.synchronize()
        res["partition_build_s"] = time.perf_counter() - t0
        marks = [[torch.cuda.Event(enable_timing=True) for _ in range(9)] for _ in range(L)]
        marks.append([torch.cuda.Event(enable_timing=True) for _ in range(2)])
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.warmup):
            step.step()
        torch.cuda.synchronize()
        if G > 1:
            dist.barrier()
        fwd = [[0.0] * 3 for _ in range(L)]
        bwd = [[0.0] * 4 for _ in range(L)]
        head, total = 0.0, 0.0
        for _ in range(args.steps):
            ends[0].record()
            step.step(marks=marks)
            ends[1].record()
            torch.cuda.synchronize()
            total += ends[0].elapsed_time(ends[1]) / args.steps
            for i in range(L):
                for s in range(3):
                    fwd[i][s] += marks[i][s].elapsed_time(marks[i][s + 1]) / args.steps
                for s in range(4):
                    bwd[i][s] += marks[i][4 + s].elapsed_time(marks[i][5 + s]) / args.steps
            head += marks[L][0].elapsed_time(marks[L][1]) / args.steps
        res["step_ms"] = wall_max(total, G, dev)
        res["exchange"] = step.exchange
        res["rank0_rows"] = part.n_local
        res["rank0_layer_ms"] = [dict(zip(FWD + BWD, f + b)) for f, b in zip(fwd, bwd)]
        res["rank0_head_to_adam_ms"] = head          # head, loss, the whole backward (the stages above), all-reduce, Adam
        res["peak_mem_gb_per_rank"] = wall_max(torch.cuda.max_memory_allocated(dev) / 1e9, G, dev)
        # transient per hidden layer and rank: dxw_part [n_pos, 512] fp32; the dx GEMM covers all n_pos rows at every G
        res["dxw_part_gb_per_hidden_layer"] = part.n_pos * 512 * 4 / 1e9
        del step, part
    except torch.OutOfMemoryError as e:
        res["out_of_memory"] = str(e).splitlines()[0]
        res["peak_mem_gb_per_rank"] = torch.cuda.max_memory_allocated(dev) / 1e9
    torch.cuda.empty_cache()
    if G == 1 and "out_of_memory" not in res:
        for c in m.gat_layers:
            c.gemm_algo = _abi.GEMM_INPUT
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=5e-4)
        try:
            for _ in range(args.warmup):
                single_gpu_step(m, opt, x16, ei, y)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                single_gpu_step(m, opt, x16, ei, y)
            torch.cuda.synchronize()
            res["single_gpu_gemm_input_step_ms"] = (time.perf_counter() - t0) / args.steps * 1e3
        except torch.OutOfMemoryError as e:
            res["single_gpu_gemm_input_step_ms"] = "out of memory: " + str(e).splitlines()[0]
    elif G > 1:
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
