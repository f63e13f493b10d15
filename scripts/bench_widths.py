"""One GATConv layer (8 heads, head mean) forward + backward at out_channels 32, 64 and 128, per stage.

For every width the layer runs twice: as a first layer (K = 166 input features, no gradient w.r.t. x) and as a hidden
layer (K = C, with dx).  Every stage (project_fwd, gat_fwd, gat_bwd = dst + src pass, project_bwd) is timed with CUDA
events over --steps steps after --warmup steps, and set against its algorithmic bytes (roofline.stage_bytes with the
width's C) over the device-to-device copy rate measured in the same run.  The default graph, a 4M-node / 40M-edge
power law, is far larger than L2 and fits all three widths: at C = 128 xw and dxw take 4 KB per node each, so the
200M-edge headline graph (20M nodes) does not fit one GPU.

  python scripts/bench_widths.py [--nodes 4000000 --edges 40000000] [--steps 10 --warmup 3] [--out FILE]
  python scripts/bench_widths.py --profile [--out FILE]     # per-kernel device times of one step, torch.profiler

Prints one JSON line (and writes it to --out): the card name and power limit read in the same run, the copy rate, and
per (width, layer) the per-stage times, bytes and their ratio to the copy rate."""
import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from gnn_fraud_detection_b200 import GATConv, build_csr, functional as Fn, roofline, synth  # noqa: E402

H = 8
STAGES = ("project_fwd", "gat_fwd", "gat_bwd", "project_bwd")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return {"name": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": q}


def copy_rate_gbs(dev, nbytes=4 << 30, reps=20):
    """device-to-device copy of nbytes (read + write counted), best of reps"""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device=dev).fill_(1.0)
    b = torch.empty_like(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * nbytes / (best * 1e-3) / 1e9


class Layer:
    """inputs and parameters of one layer at width C and fan-in K"""

    def __init__(self, g, N, K, C, need_dx, dev):
        torch.manual_seed(1)
        conv = GATConv(K, C, heads=H, concat=False, dropout=0.0).to(dev)
        self.g, self.N, self.K, self.C, self.need_dx = g, N, K, C, need_dx
        self.W = conv.lin_src.weight.detach()
        self.a_s = conv.att_src.detach().view(-1).contiguous()
        self.a_d = conv.att_dst.detach().view(-1).contiguous()
        self.bias = conv.bias.detach()
        self.x = torch.randn(N, K, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
        self.d_out = torch.full((N, C), 1.0 / N, device=dev)

    def step(self, ev=None):
        """one fwd + bwd; ev: dict stage -> (start, end) events recorded around each stage"""
        def mark(stage, i):
            if ev is not None:
                ev[stage][i].record()
        C, g = self.C, self.g
        mark("project_fwd", 0)
        xw, a_src, a_dst = Fn.project_fwd(self.x, self.W, self.a_s, self.a_d, H, C)
        mark("project_fwd", 1)
        mark("gat_fwd", 0)
        out, rowmax, rowsum = Fn.gat_fwd(g, xw, a_src, a_dst, self.bias, H, C, 0.2, False)
        mark("gat_fwd", 1)
        mark("gat_bwd", 0)
        dxw, da_src, da_dst = Fn.gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, self.d_out, self.a_s, self.a_d, H, C, 0.2,
                                         False)
        mark("gat_bwd", 1)
        mark("project_bwd", 0)
        Fn.project_bwd(self.x, self.W, dxw, xw, da_src, da_dst, self.d_out, H, C, C, self.need_dx)
        mark("project_bwd", 1)
        return out


def short(name):
    m = re.search(r"(?:gnnfd::)?(?:tc::)?(\w+)<", name) or re.search(r"(?:gnnfd::)?(\w+)\(", name)
    return m.group(1) if m else name


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=4_000_000)
    ap.add_argument("--edges", type=int, default=40_000_000)
    ap.add_argument("--widths", default="32,64,128")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="per-kernel device times of one step (torch.profiler)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_widths.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    N = args.nodes
    ei = synth.powerlaw_graph(N, args.edges, seed=1234, device=dev)
    g = build_csr(ei, N)
    del ei
    Ep = g.n_edges
    res = {"metric": "gatconv_layer_stage_ms_by_width", "graph": f"powerlaw N={N} E={args.edges} E'={Ep}", "heads": H,
           "gpu": card(), "runs": []}
    if not args.profile:
        res["copy_gbs"] = copy_rate_gbs(dev)
    for C in [int(c) for c in args.widths.split(",")]:
        for kind, K, need_dx in (("first", 166, False), ("hidden", C, True)):
            lay = Layer(g, N, K, C, need_dx, dev)
            for _ in range(args.warmup):
                lay.step()
            torch.cuda.synchronize()
            run = {"C": C, "layer": kind, "K": K, "dx": need_dx}
            if args.profile:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    lay.step()
                    torch.cuda.synchronize()
                kern = {}
                for e in prof.events():
                    if e.device_type.name == "CUDA":
                        k = short(e.name)
                        kern[k] = kern.get(k, 0.0) + e.device_time / 1e3
                run["kernel_ms"] = {k: round(v, 4) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])}
            else:
                ms = {s: 0.0 for s in STAGES}
                for _ in range(args.steps):
                    ev = {s: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for s in STAGES}
                    lay.step(ev)
                    torch.cuda.synchronize()
                    for s in STAGES:
                        ms[s] += ev[s][0].elapsed_time(ev[s][1]) / args.steps
                b = roofline.stage_bytes(N, Ep, K, H=H, C=C, need_dx=need_dx)
                b["gat_bwd"] = b["gat_bwd_dst"] + b["gat_bwd_src"]
                run["stages"] = {s: {"ms": round(ms[s], 4), "bytes": b[s],
                                     "gbs": round(b[s] / (ms[s] * 1e-3) / 1e9, 1),
                                     "frac_of_copy": round(b[s] / (ms[s] * 1e-3) / 1e9 / res["copy_gbs"], 3)}
                                 for s in STAGES}
                run["step_ms"] = round(sum(ms.values()), 4)
            res["runs"].append(run)
            del lay
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
