"""Training-step time of a 3-layer GAT(166, 64, 1) on one GPU: the projected-feature path (GEMM_AUTO) against the input-space
formulation on every layer (GEMM_INPUT; the hidden layers get dx through the source-major pass and the dx GEMM).

A step is DeviceTrainStep's: forward, masked BCEWithLogitsLoss(pos_weight=50), backward and capturable Adam, replayed from one
CUDA graph (reference training configuration: dropout 0.2, train-mode BatchNorm, residual).  Per workload the two arms are
alternated --rounds times in this one process; each arm is built, captured, timed over --steps replays (CUDA events) and freed
before the other is built, so max_memory_allocated is the arm's own.  The relative L2 difference of the two arms' parameter
gradients comes from one eager step with dropout 0 from the same initial weights on the timed graph.

  --workloads  powerlaw_20m (N = 2M, E = 20M), elliptic (N = 203,769, E = 234,355: latency-bound), and powerlaw_max: the
               first of --max-edges (descending) at which both arms fit.
  --profile    instead: one eager step per arm under torch.profiler on the 20M-edge graph, the hidden layers' backward split
               into edge pass, source-major pass, dx GEMM and parameter gradients (device time of the kernels each stage
               launches).  Run it separately: tracing slows the host.

Prints one JSON line and writes it to --out, with the card name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from gnn_fraud_detection_b200 import GAT, _abi, functional as Fn, synth  # noqa: E402
from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE  # noqa: E402
from gnn_fraud_detection_b200.train_step import DeviceTrainStep  # noqa: E402

ARMS = {"auto": _abi.GEMM_AUTO, "input": _abi.GEMM_INPUT}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return {"name": torch.cuda.get_device_name(), "power_limit_and_max_sm_clock": q}


def data(n, e):
    dev = torch.device("cuda")
    if n is None:
        x, ei, _ = synth.elliptic_synth(seed=0, device=dev)
    else:
        ei = synth.powerlaw_graph(n, e, seed=1234, device=dev)
        x = torch.randn(n, 166, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    y = (torch.rand(x.size(0), device=dev, generator=torch.Generator(device=dev).manual_seed(1)) < 0.1).long()
    y[::7] = -1
    return x, ei, y


def model(algo, dropout):
    torch.manual_seed(0)
    return GAT(166, 64, 1, num_layers=3, dropout=dropout, gemm_algo=algo).cuda().train()


def free():
    GLOBAL_CSR_CACHE.clear()
    Fn.GLOBAL_XIMAGE_CACHE.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def time_arm(algo, x, ei, y, steps):
    """(ms per replayed step, bytes of max_memory_allocated above what was resident before the arm was built)."""
    free()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    tr = DeviceTrainStep(model(algo, 0.2), x, ei, y)
    for _ in range(3):
        tr.step()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        tr.step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    peak = torch.cuda.max_memory_allocated() - base
    tr.close()
    del tr
    return ms, peak


def grads(algo, x, ei, y):
    m = model(algo, 0.0)
    mask = y != -1
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, device="cuda"))
    crit(m(x, ei)[mask].squeeze(1), y[mask].float()).backward()
    g = torch.cat([p.grad.reshape(-1).double().cpu() for n, p in m.named_parameters()
                   if not (n.startswith("gat_layers.") and n.endswith(".bias"))])   # conv biases: true gradient 0 (BatchNorm)
    del m
    free()
    return g


def bench(name, n, e, steps, rounds):
    x, ei, y = data(n, e)
    r = {"workload": name, "nodes": int(x.size(0)), "edges": int(ei.size(1)), "steps": steps, "rounds": rounds}
    for arm in ARMS:
        r[f"{arm}_ms"], r[f"{arm}_max_memory_allocated_bytes"] = [], 0
    for _ in range(rounds):
        for arm, algo in ARMS.items():
            ms, peak = time_arm(algo, x, ei, y, steps)
            r[f"{arm}_ms"].append(round(ms, 3))
            r[f"{arm}_max_memory_allocated_bytes"] = max(r[f"{arm}_max_memory_allocated_bytes"], peak)
    ga, gi = grads(ARMS["auto"], x, ei, y), grads(ARMS["input"], x, ei, y)
    r["grad_rel_l2_input_vs_auto"] = float((gi - ga).norm() / ga.norm())
    for arm in ARMS:
        r[f"{arm}_ms_median"] = sorted(r[f"{arm}_ms"])[len(r[f"{arm}_ms"]) // 2]
    del x, ei, y
    free()
    return r


def profile(n, e):
    """Device time per backward stage of the hidden layers (K = 64), one eager step per arm."""
    from torch.profiler import ProfilerActivity, profile as tprof, record_function
    stages = {"in_bwd_edges": "edge_pass", "gat_bwd_src": "src_pass", "project_dx": "dx_gemm", "in_bwd_params": "params"}
    orig = {f: getattr(Fn, f) for f in stages}

    xarg = {"in_bwd_edges": 1, "in_bwd_params": 2}    # position of the layer input x; the other two run for hidden layers only

    def wrap(f):
        def call(*a, **kw):
            hidden = f not in xarg or a[xarg[f]].size(1) == 64
            with record_function(f"hidden/{stages[f]}" if hidden else f"first/{stages[f]}"):
                return orig[f](*a, **kw)
        return call

    x, ei, y = data(n, e)
    out = {"workload": f"powerlaw N={n} E={e}", "nodes": int(x.size(0)), "edges": int(ei.size(1))}
    for f in stages:
        setattr(Fn, f, wrap(f))
    try:
        for arm, algo in ARMS.items():
            grads(algo, x, ei, y)               # warm-up: modules, CSR, workspaces
            torch.cuda.synchronize()
            with tprof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as p:
                grads(algo, x, ei, y)
                torch.cuda.synchronize()
            ev = p.key_averages()
            labels = ("hidden/", "first/")      # the stage ranges above also appear as device events: not kernels
            kern = sorted(((k.key, k.device_time_total / 1e3) for k in ev if k.device_type == torch.autograd.DeviceType.CUDA
                           and k.device_time_total > 0 and not k.key.startswith(labels)), key=lambda t: -t[1])
            # (the projected path calls gat_bwd_src for every layer: its stage labels mean something for the input arm only)
            split = {k.key: round(k.device_time_total / 1e3, 3) for k in ev if k.key.startswith(labels)}
            out[arm] = {"stages_ms_summed_over_layers": split if arm == "input" else None,
                        "kernels_ms": [(k, round(t, 3)) for k, t in kern[:40]],
                        "device_ms_total": round(sum(t for _, t in kern), 3)}
    finally:
        for f, fn in orig.items():
            setattr(Fn, f, fn)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="powerlaw_20m,elliptic,powerlaw_max")
    ap.add_argument("--max-edges", default="100000000,60000000,40000000")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_input_space.py needs a CUDA device")
    res = {"card": card(), "model": "GAT(166, 64, 1, num_layers=3)"}

    def emit():                                 # after every workload: a later out-of-memory attempt cannot lose results
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")

    if args.profile:
        res["profile"] = profile(2_000_000, 20_000_000)
        emit()
        return
    res["results"] = []
    for w in args.workloads.split(","):
        if w == "powerlaw_20m":
            res["results"].append(bench(w, 2_000_000, 20_000_000, args.steps, args.rounds))
        elif w == "elliptic":
            res["results"].append(bench(w, None, None, args.steps, args.rounds))
        elif w == "powerlaw_max":
            res["powerlaw_max_did_not_fit_edges"] = []
            for e in (int(float(v)) for v in args.max_edges.split(",")):
                try:
                    res["results"].append(bench(w, e // 10, e, args.steps, args.rounds))
                    break
                except torch.OutOfMemoryError:
                    res["powerlaw_max_did_not_fit_edges"].append(e)
                    free()
        else:
            raise SystemExit(f"unknown workload {w}")
        emit()


if __name__ == "__main__":
    main()
