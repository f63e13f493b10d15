"""Per-kernel device time of the layer backward (or, with --stage fwd, of the layer's gat_fwd) on the headline graph
(20M nodes / 200M edges, H=8, C=64, head mean).

Runs warm-up steps of the single-GPU layer as bench.py does (project_fwd, gat_fwd, gat_bwd, project_bwd), one step for
max_memory_allocated / max_memory_reserved, then one step whose gat_bwd call (the dst and src passes) or gat_fwd call
runs under torch.profiler with CUDA activity, and prints one JSON line: the device time of every kernel that call
launched, by kernel name.  Run it in a process of its own (tracing slows the host; the times are device times of single
launches).

  python scripts/prof_bwd.py [--stage bwd|fwd] [--workload powerlaw_200m] [--out profiles/prof_bwd_TAG.json]

GNNFD_B200_LIB selects the library build, as for bench.py."""
import argparse
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from gnn_fraud_detection_b200 import GATConv, build_csr, functional as Fn  # noqa: E402


def short(name: str) -> str:
    """demangled kernel name without namespace, parameters and the template's argument list"""
    m = re.search(r"(?:gnnfd::)?(\w+)<", name) or re.search(r"(?:gnnfd::)?(\w+)\(", name)
    return m.group(1) if m else name


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="powerlaw_200m", choices=["powerlaw_200m", "powerlaw_20m"])
    ap.add_argument("--stage", default="bwd", choices=["bwd", "fwd"], help="the call that runs under the profiler")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    H, C = bench.H, bench.C
    N, E, K = bench.WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ei = bench.make_edges(args.workload, N, E, dev)
    g = build_csr(ei, N)
    del ei
    torch.manual_seed(1)
    conv = GATConv(K, C, heads=H, concat=False, dropout=0.0).to(dev)
    W = conv.lin_src.weight.detach()
    a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
    x = torch.randn(N, K, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    d_out = torch.full((N, C), 1.0 / N, device=dev)

    def step(prof_stage: str = ""):
        prof = None

        def window(stage):             # only the profiled call runs inside the window
            nonlocal prof
            torch.cuda.synchronize()
            if prof_stage == stage:
                prof = profile(activities=[ProfilerActivity.CUDA])
                prof.__enter__()

        def close(stage):
            torch.cuda.synchronize()
            if prof_stage == stage:
                prof.__exit__(None, None, None)

        xw, a_src, a_dst = Fn.project_fwd(x, W, a_s, a_d, H, C)
        window("fwd")
        out, rowmax, rowsum = Fn.gat_fwd(g, xw, a_src, a_dst, conv.bias.detach(), H, C, 0.2, False)
        close("fwd")
        del out
        window("bwd")
        dxw, da_src, da_dst = Fn.gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C, 0.2, False)
        close("bwd")
        Fn.project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C, C, False)
        torch.cuda.synchronize()
        return prof

    for _ in range(args.warmup):
        step()
    torch.cuda.reset_peak_memory_stats(dev)
    step()
    peak = torch.cuda.max_memory_allocated(dev)
    peak_reserved = torch.cuda.max_memory_reserved(dev)
    prof = step(prof_stage=args.stage)
    kern = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or e.name.startswith(("Memcpy", "Memset")):
            continue
        k = short(e.name)
        kern[k] = kern.get(k, 0.0) + e.time_range.elapsed_us() / 1e3
    per = {k: round(v, 3) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])}
    line = {
        "workload": args.workload, "gpu": torch.cuda.get_device_name(dev),
        "lib": os.environ.get("GNNFD_B200_LIB", "gnn_fraud_detection_b200/libgnnfd_b200.so"),
        f"{args.stage}_kernel_ms": per, f"{args.stage}_total_ms": round(sum(per.values()), 3),
        "max_memory_allocated_gb": round(peak / 1e9, 2), "max_memory_reserved_gb": round(peak_reserved / 1e9, 2),
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
