#!/usr/bin/env python
"""Headline benchmark: GAT layer fwd+bwd edges/sec (BASELINE.json metric) + achieved HBM GB/s vs peak.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload powerlaw_200m|elliptic|skew] [--impl reference]
                  [--dump-outputs DIR]

A "step" is one GATConv layer (H=8, C=64, concat=False, bias, dropout off) forward + backward over the
whole synthetic graph, CSR cached (its build is reported separately).  Default workload at N=1 is the
configuration the metric's target is quoted on: the 200M-edge / 20M-node power-law graph, K=166
(BASELINE.json configs[3], "powerlaw_200m"); it fits one B200 (~125 GB).  One JSON line on stdout (rank 0).

`--impl reference` times the reference formulation (PyG GATConv semantics: the CPU oracle port, since
torch_geometric is not installable in this image) on the host cores, on a bounded sample of the same
workload family.

`--dump-outputs DIR` writes what the timed path computed in its last timed step -- the layer output and the parameter
gradients (the TGN workload: loss, logits and parameter gradients) -- as DIR/<name>.npy in float32 / float64.  Of an
output with more than 65,536 rows, a fixed seeded sample of 65,536 rows is written.  The inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "gat_layer_fwd_bwd_edges_per_sec"
UNIT = "edges/s"
H, C = 8, 64

WORKLOADS = {
    # name: (N, E, K)
    "powerlaw_200m": (20_000_000, 200_000_000, 166),
    "powerlaw_20m": (2_000_000, 20_000_000, 166),
    "elliptic": (203_769, 234_355, 166),
    "skew": (1_000_000, 5_000_000 + 16 * 131_072 + 64_000, 166),
    # BASELINE.json configs[2]: TemporalGNN over the 49 time-step snapshots, sharded by time step (model-level step)
    "tgn_snapshots": (203_769, 234_355, 166),
}
CPU_SAMPLE = (200_000, 2_000_000, 166)   # 1/100-scale power-law graph for the CPU arm (bounded sample, BASELINE.md section 3)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


DUMP_ROWS = 65_536
DUMP_LIMIT_BYTES = 64 << 20


def output_sample(arrays: dict) -> dict:
    """Host float32 / float64 copies of ``arrays``; of a tensor with more than DUMP_ROWS rows, the rows of a fixed
    seeded sample (the same rows in every run)."""
    res = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.dim() and t.size(0) > DUMP_ROWS:
            rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
            t = t[rows.to(t.device)]
        res[name] = (t if t.dtype == torch.float64 else t.float()).cpu().numpy()
    return res


def write_outputs(path: str, arrays: dict) -> None:
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def make_edges(workload: str, N: int, E: int, device):
    from gnn_fraud_detection_b200 import synth
    if workload.startswith("powerlaw"):
        return synth.powerlaw_graph(N, E, seed=1234, device=device)
    if workload == "elliptic":
        return synth.elliptic_synth(N, E, 1, seed=0, device=device)[1]
    if workload == "skew":
        return synth.fraud_ring_skew(num_nodes=N, seed=7, device=device)
    raise ValueError(workload)


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (pynvml; nvidia-smi fallback)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self._h is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm (reference formulation = oracle port)
# ------------------------------------------------------------------------------------------------
def cpu_sample_for(workload: str):
    """(N, E, K, same_config): the Elliptic-shaped workload runs at FULL size on the host (BASELINE.json configs[0]/[1]);
    the power-law / skew workloads cannot (PyG's [E',8,64] message tensor alone is 450 GB at 200M edges), so the CPU arm
    runs the 1/100-scale graph of the same family."""
    if workload == "elliptic":
        return WORKLOADS["elliptic"] + (True,)
    return CPU_SAMPLE + (False,)


def cpu_reference_step_fn(workload, threads):
    """Returns (step_fn, kind, description, E, same_config).  Only bench.py's cpu_baseline / --impl reference legs use the
    oracle."""
    from gnn_fraud_detection_b200 import synth
    from oracle import pyg_gatconv as O
    torch.set_num_threads(threads)
    kind = "port"
    N, E, K, same = cpu_sample_for(workload)
    if workload == "elliptic":
        ei = synth.elliptic_synth(N, E, 1, seed=0, device="cpu")[1]
        what = f"Elliptic-shaped graph N={N} E={E} K={K} at FULL size (same config as the GPU arm)"
    else:
        ei = synth.powerlaw_graph(N, E, seed=1234, device="cpu")
        what = f"power-law graph N={N} E={E} K={K} (1/{200_000_000 // E}-scale powerlaw_200m)"
    E = ei.size(1)
    x = torch.randn(N, K, generator=torch.Generator().manual_seed(0))
    torch.manual_seed(1)
    conv = O.OracleGATConv(K, C, heads=H, concat=False, dropout=0.0)
    if O.real_pyg_available():      # never true in this image; kept so the arm uses the real thing if it appears
        from torch_geometric.nn import GATConv as PygGATConv
        conv = PygGATConv(K, C, heads=H, concat=False, dropout=0.0)
        kind = "reference"
    d_out = torch.ones(N, C) / N

    def step():
        for p in conv.parameters():
            p.grad = None
        out = conv(x, ei)
        out.backward(d_out)
        return {"out": out.detach(), **{f"grad.{n}": p.grad for n, p in conv.named_parameters()}}

    return step, kind, what + ", one GATConv fwd+bwd", E, same


def cpu_tgn_step_fn(threads):
    """The reference's TemporalGNN training step (oracle port of the PyG formulation) on the full Elliptic-shaped graph."""
    from gnn_fraud_detection_b200 import synth
    from oracle import pyg_gatconv as O
    torch.set_num_threads(threads)
    N, E, K = WORKLOADS["tgn_snapshots"]
    x, ei, _ = synth.elliptic_synth(N, E, K, seed=0, device="cpu")
    y = (torch.rand(N, generator=torch.Generator().manual_seed(3)) < 0.1).long()
    y[torch.rand(N, generator=torch.Generator().manual_seed(4)) < 0.77] = -1
    torch.manual_seed(1)
    ref = O.OracleTemporalGNN(K, 64, 1, num_layers=2, dropout=0.0).train()
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0))

    def step():
        for p in ref.parameters():
            p.grad = None
        lg, _ = ref(x, ei)
        m = y != -1
        loss = crit(lg[m].squeeze(1), y[m].float())
        loss.backward()
        return {"loss": loss.detach(), "logits": lg.detach(), **{f"grad.{n}": p.grad for n, p in ref.named_parameters()}}

    return step, "port", (f"Elliptic-shaped graph N={N} E={E} K={K}, 49 time steps, at FULL size: one TemporalGNN (2 layers) "
                          f"training step, fwd + loss + bwd"), E, True


def run_reference_arm(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    if args.workload == "tgn_snapshots":
        step, kind, sample, E, same = cpu_tgn_step_fn(threads)
    else:
        step, kind, sample, E, same = cpu_reference_step_fn(args.workload, threads)
    K = WORKLOADS[args.workload][2]
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outputs = step()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        write_outputs(args.dump_outputs, output_sample(outputs))
    val = E / dt
    line = {
        "impl": "reference", "metric": "tgn_train_step_edges_per_sec" if args.workload == "tgn_snapshots" else METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "reference_sample": sample, "same_config": same, "H": H, "C": C, "K": K,
                   "note": "reference = PyG GATConv formulation on host cores; torch_geometric is absent from "
                           "this image so the CPU oracle port (oracle/pyg_gatconv.py) is what runs"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def run_gpu_arm(args):
    import torch.distributed as dist
    from gnn_fraud_detection_b200 import GATConv, _abi, build_csr, functional as Fn, roofline, synth
    from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback); use --impl reference "
                         "for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from gnn_fraud_detection_b200 import partition
    L = _abi.lib()

    workload = args.workload
    N, E, K = WORKLOADS[workload]
    free_b, total_b = torch.cuda.mem_get_info()
    note = None
    if workload == "powerlaw_200m" and world == 1 and free_b < 140e9:
        workload, note = "powerlaw_20m", f"only {free_b / 1e9:.0f} GB free: fell back from powerlaw_200m"
        N, E, K = WORKLOADS[workload]

    # ---- inputs, resident in HBM before the timed region ------------------------------------------
    t_gen = time.perf_counter()
    ei = make_edges(workload, N, E, dev)
    E = ei.size(1)
    gen = torch.Generator(device=dev).manual_seed(0)
    torch.manual_seed(1)
    conv = GATConv(K, C, heads=H, concat=False, dropout=0.0, gemm_algo=args.algo,
                   feature_dtype=torch.bfloat16 if args.bf16 else torch.float32).to(dev)
    W = conv.lin_src.weight.detach()
    a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
    bias = conv.bias.detach()
    xw_dtype = conv.feature_dtype

    if world == 1:
        x = torch.randn(N, K, device=dev, generator=gen)
        g = build_csr(ei, N)            # cold build: module load, allocator growth
        torch.cuda.synchronize()
        del g
        t0 = time.perf_counter()
        g = build_csr(ei, N)            # warm build: what every e2e step pays
        torch.cuda.synchronize()
        csr_ms = (time.perf_counter() - t0) * 1e3
        Ep = g.n_edges
        d_out = torch.full((N, C), 1.0 / N, device=dev)      # timing only (SURVEY 8(d)); parity runs use randn/N
        n_local, part = N, None
    else:
        Part = {"input": partition.InputSpacePartition, "replicate": partition.ReplicatedInputPartition,
                "allgather": partition.DstRangePartition}[args.mgpu]
        part = Part.build(ei, N, rank, world, dev)
        del ei
        g, Ep, n_local = part.graph, part.graph.n_edges, part.n_local
        csr_ms = part.build_ms
        if args.mgpu == "input":       # replicated input in the padded-row layout of the input-space kernels
            x = torch.zeros(part.n_pos, Fn.in_sizes(0, K)[3], device=dev)
            x[:, :K] = torch.randn(part.n_pos, K, device=dev, generator=gen)
            x = x[:, :K]
        elif args.mgpu == "replicate":   # the layer input is resident on every GPU (same seed => identical copies)
            x = torch.randn(part.n_pos, K, device=dev, generator=gen)
        else:                          # this rank's rows of x
            x = torch.randn(part.rows_padded, K, device=dev, generator=gen)
        d_out = torch.full((n_local, C), 1.0 / N, device=dev)
    gen_s = time.perf_counter() - t_gen

    input_space = (args.algo == _abi.GEMM_INPUT) if world == 1 else (args.mgpu == "input")
    if input_space:
        stages = ["in_logits", "in_fwd_edges", "in_out_gemm", "in_bwd_gd_edges", "in_bwd_dasrc", "in_bwd_params"]
        if world == 1:
            in_prep = Fn._aligned_u8(Fn.in_sizes(n_local, K)[0], dev)
            x = Fn.in_pad_x(x)            # static first-layer input: padded once, like the CSR
            in_xmax = torch.zeros(16, device=dev)
    else:
        stages = ["project_fwd", "gat_fwd", "gat_bwd_dst_src", "project_bwd"]
    ximg, ximg_ms = None, None
    if world == 1 and not input_space and Fn.image_projection_applies(x, H, C, xw_dtype, args.algo):
        t0 = time.perf_counter()
        ximg = Fn.XImage(x)
        torch.cuda.synchronize()
        ximg_ms = (time.perf_counter() - t0) * 1e3
    ev = {}

    def step(timed: bool):
        """One layer fwd+bwd through the C ABI stage calls (exactly what GATConvFunction issues)."""
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(len(stages) + 1)] if timed else None
        if timed:
            marks[0].record()
        if part is None and input_space:
            in_xmax.zero_()
            a_src, a_dst = Fn.in_logits(x, W, a_s, a_d, in_prep, in_xmax)
            Fn.in_prepare(W, K, in_xmax, in_prep)
            if timed: marks[1].record()
            zimg, att = Fn.in_fwd(g, x, a_src, a_dst, 0.2, in_prep)
            if timed: marks[2].record()
            out = Fn.in_out(zimg, N, K, in_prep, bias)
            if timed: marks[3].record()
            dz, da_dst = Fn.in_bwd_edges(g, x, att, d_out, in_prep, 0.2)
            if timed: marks[4].record()
            da_src = Fn.in_dasrc(g, dz)
            if timed: marks[5].record()
            grads = Fn.in_bwd_params(zimg, d_out, x, W, a_s, a_d, da_src, da_dst, in_prep)
            if timed: marks[6].record()
            del zimg, dz
        elif part is None:
            if ximg is not None:       # static first-layer input: its tensor-core image is built once, like the CSR
                xw, a_src, a_dst = Fn.project_fwd_image(ximg, W, a_s, a_d)
            else:
                xw, a_src, a_dst = Fn.project_fwd(x, W, a_s, a_d, H, C, xw_dtype, args.algo)
            if timed: marks[1].record()
            out, rowmax, rowsum = Fn.gat_fwd(g, xw, a_src, a_dst, bias, H, C, 0.2, False)
            if timed: marks[2].record()
            dxw, da_src, da_dst = Fn.gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C, 0.2, False)
            if timed: marks[3].record()
            grads = Fn.project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C, C, False, args.algo)
            if timed: marks[4].record()
        else:
            out, grads = part.layer_fwd_bwd(x, W, a_s, a_d, bias, d_out, H, C, xw_dtype, args.algo, marks)
        return out, grads, marks

    for _ in range(max(args.warmup, 3)):
        step(False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    L.gnnfd_launch_count_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    all_marks = []
    t_host = time.perf_counter()
    e_start.record()
    for i in range(args.steps):
        out, grads, marks = step(True)
        all_marks.append(marks)
        if i + 1 < args.steps:
            del out, grads          # only the last step's outputs are kept
    e_end.record()
    host_enqueue_ms = (time.perf_counter() - t_host) * 1e3 / args.steps       # host time to ENQUEUE one step
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    launches = int(L.gnnfd_launch_count())
    out_names = ("out", "dW", "datt_src", "datt_dst", "dbias")
    dumped = output_sample(dict(zip(out_names, (out,) + tuple(grads)))) if args.dump_outputs and rank == 0 else None
    del out, grads
    total_ms = e_start.elapsed_time(e_end)
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    eager_ms_per_step, graph_note = ms_per_step, None
    use_graph = args.graph == "on" or (args.graph == "auto" and world > 1)
    if use_graph:
        # The step launches ~50 kernels and 3 collectives.  Replaying it from a CUDA graph removes the host from the loop:
        # across 8 ranks the slowest host thread otherwise delays everybody at the first collective of the step.  Same
        # kernels, same collectives, same data; K replays timed exactly like the eager loop (whose per-stage split stays
        # in roofline.stages_ms).
        try:
            torch.cuda.synchronize()
            cg = torch.cuda.CUDAGraph()
            cs = torch.cuda.Stream(device=dev)
            cs.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(cs):
                step(False)
                cs.synchronize()
                with torch.cuda.graph(cg, stream=cs):
                    g_out, g_grads, _ = step(False)
            torch.cuda.current_stream().wait_stream(cs)
            for _ in range(3):
                cg.replay()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(args.steps):
                cg.replay()
            g1.record()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()
            g_ms = g0.elapsed_time(g1)
            if world > 1:
                t = torch.tensor([g_ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                g_ms = float(t.item())
            ms_per_step = g_ms / args.steps
            graph_note = "timed as K replays of ONE CUDA graph of the whole step (kernels + collectives)"
            if dumped is not None:
                dumped = output_sample(dict(zip(out_names, (g_out,) + tuple(g_grads))))
            del cg, g_out, g_grads
        except Exception as ex:     # capture not possible on this stack: keep the eager number
            graph_note = f"CUDA graph capture failed ({type(ex).__name__}: {str(ex)[:120]}); eager timing reported"
            ms_per_step = eager_ms_per_step
    selfcheck = None
    if world > 1 and not args.no_selfcheck:
        selfcheck = multi_gpu_selfcheck(type(part), rank, world, dev, K, H, C)
    clocks = sampler.stop()
    stage_ms = {s: statistics.mean(m[i].elapsed_time(m[i + 1]) for m in all_marks) for i, s in enumerate(stages)}
    if os.environ.get("GNNFD_BENCH_DEBUG"):
        print(f"[rank {rank}] n_local={n_local} Ep={Ep} host_enqueue_ms={host_enqueue_ms:.2f} eager_ms={eager_ms_per_step:.2f} "
              f"ms={ms_per_step:.2f} stages_ms={ {k: round(v, 2) for k, v in stage_ms.items()} } {graph_note}",
              file=sys.stderr, flush=True)

    # ---- roofline ------------------------------------------------------------------------------------
    peak, peak_src = load_peaks()
    s_bytes = 2 if args.bf16 else 4
    E_total = E
    if world > 1:
        te = torch.tensor([float(Ep)], device=dev)
        dist.all_reduce(te)
        Ep_total = int(te.item())
    else:
        Ep_total = Ep
    # SURVEY.md 8(d) byte model (projected-feature formulation): the figure `layer` is quoted against, whichever
    # formulation ran.  `own` = the byte model of the formulation that actually ran on this rank.
    bmodel = roofline.stage_bytes(N, Ep_total, K, H, C, False, s_bytes, need_dx=False)
    if input_space:
        own = roofline.stage_bytes_input_space(n_local, Ep, K, H, C, n_src=(N if world > 1 else None))
        stage_b = {"in_logits": own["in_logits"], "in_fwd_edges": own["in_fwd_edges"], "in_out_gemm": own["in_out_gemm"],
                   "in_bwd_gd_edges": own["in_bwd_gd"] + own["in_bwd_edges"], "in_bwd_dasrc": own["in_bwd_dasrc"],
                   "in_bwd_params": own["in_bwd_params"]}
        kernels = {"in_logits": "in_logits_kernel", "in_fwd_edges": "in_alpha_items + gat_in_fwd_items (+hub chunks/merge)",
                   "in_out_gemm": "in_out_gemm (tcgen05 kind::f16, bulk-fed)",
                   "in_bwd_gd_edges": "in_proj_gemm<false> (Gd, tcgen05 kind::f16) + gat_in_bwd_items (+hub)",
                   "in_bwd_dasrc": "in_dasrc_kernel",
                   "in_bwd_params": "in_dw_gemm (tcgen05 kind::f16, MN-major) + dax_partial"}
    else:
        own = roofline.stage_bytes(n_local, Ep, K, H, C, False, s_bytes, need_dx=False, n_src=(N if world > 1 else None))
        stage_b = {"project_fwd": own["project_fwd"], "gat_fwd": own["gat_fwd"],
                   "gat_bwd_dst_src": own["gat_bwd_dst"] + own["gat_bwd_src"], "project_bwd": own["project_bwd"]}
        kernels = {"project_fwd": "in_proj_gemm (tcgen05 kind::f16 from the cached image of x)" if ximg is not None else "tc::gemm_tc_ws2", "gat_fwd": "gat_fwd_items_pack (+hub chunks/merge)",
                   "gat_bwd_dst_src": "gat_bwd_dst_items_pack (+hub) + gat_bwd_src_rows", "project_bwd": "tc::dw_tc2 + dax_partial"}
    # dominant stage = the one with the largest measured time on this rank
    dom = max(stages, key=lambda k: stage_ms[k])
    dom_bytes, dom_ms = stage_b[dom], stage_ms[dom]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    own_total = sum(stage_b.values())
    traffic = None
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            traffic = json.load(open(traffic_file)).get(workload, {}).get(dom)
        except Exception:
            traffic = None
    roof = {"bound": "hbm", "kernel": kernels[dom], "stage": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": dom_bytes, "ms_per_launch": dom_ms,
            "formulation": "input-space (csrc/in_common.cuh)" if input_space else "projected-feature (PyG order of operations)",
            "layer": {"algorithmic_bytes": bmodel["total"], "achieved": bmodel["total"] / (ms_per_step * 1e-3) / 1e9 / world,
                      "frac": bmodel["total"] / (ms_per_step * 1e-3) / 1e9 / world / peak,
                      "byte_model": "SURVEY.md 8(d), projected-feature formulation"},
            "layer_own_model": {"algorithmic_bytes": own_total, "achieved": own_total / (ms_per_step * 1e-3) / 1e9,
                                "frac": own_total / (ms_per_step * 1e-3) / 1e9 / peak,
                                "byte_model": "bytes of the formulation that ran, this rank"},
            "stages_ms": stage_ms,
            "stages_gbs": {k: stage_b[k] / stage_ms[k] / 1e6 for k in stages}}

    value = E_total / (ms_per_step * 1e-3)

    # ---- e2e: public API (GATConv module) with HOST buffers, copies inside the timed region ----------
    e2e = None
    if not args.no_e2e:
        if world == 1:
            # stage the inputs in pinned host memory, then release the device-resident copies
            x_host = torch.empty(x.shape, dtype=x.dtype, pin_memory=True).copy_(x)
            ei_host = torch.empty(ei.shape, dtype=ei.dtype, pin_memory=True).copy_(ei)
            torch.cuda.synchronize()
            del x, ei, g, d_out, all_marks
            ximg = None
            Fn.GLOBAL_XIMAGE_CACHE.clear()
            GLOBAL_CSR_CACHE.clear()
            torch.cuda.empty_cache()
            e2e = run_e2e(args, conv, x_host, ei_host, N, E_total, dev)
        else:
            e2e = part.e2e(args, conv, x, N, E_total, K, dev)

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) -------------------------------------------
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu:
        threads = os.cpu_count() or 1
        cstep, kind, sample, ce, same = cpu_reference_step_fn(workload, threads)
        cstep()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            cstep()
        cdt = (time.perf_counter() - t0) / reps
        cpu = {"value": ce / cdt, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample, "same_config": same,
               "ms_per_step": cdt * 1e3}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16-storage/f32-accum" if args.bf16 else "f32", "data": "synthetic",
            "config": {"workload": workload, "nodes": N, "edges": E_total, "edges_after_self_loop_rewrite": Ep_total,
                       "in_features": K, "heads": H, "out_channels": C, "concat": False,
                       "l2": "inputs larger than L2 (xw %.1f GB per pass)" % (N * H * C * s_bytes / 1e9),
                       "parallelism": "1 GPU" if world == 1 else {
                           "input": f"dst-range x{world}: replicated input, input-space aggregation, all-gather / "
                                    f"reduce-scatter of [N,H] logit vectors only",
                           "replicate": f"dst-range x{world}: replicated input + redundant projection, all-to-all of "
                                        f"per-edge grads, all-gather of dOut",
                           "allgather": f"dst-range x{world}: NCCL all-gather of projected features, reduce-scatter of dxw",
                       }[args.mgpu],
                       "formulation": "input-space" if input_space else "projected-feature",
                       "exchange": (None if part is None else {
                           "multicast": "fused into the kernels: multimem.st / multimem.ld_reduce through the NVSwitch "
                                        "(symmetric memory), no collective call on the data path",
                           "peer": "fused into the kernels: NVLink stores / loads on peer memory (symmetric memory)",
                       }.get(getattr(part, "exchange", "nccl"), "NCCL all-gather / reduce-scatter")),
                       "csr_build_ms": csr_ms, "x_image_build_ms": ximg_ms, "setup_s": gen_s,
                       "gemm_algo": args.algo, "note": note},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "timing": {"eager_ms_per_step": eager_ms_per_step, "host_enqueue_ms_per_step": host_enqueue_ms, "cuda_graph": graph_note},
            "selfcheck": selfcheck,
        }
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[2]: TemporalGNN over 49 snapshots, sharded by time step (no data-path collective)
# ------------------------------------------------------------------------------------------------
def multi_gpu_selfcheck(partition_cls, rank, world, dev, K, H, C):
    """Every multi-GPU run checks itself (outside the timed region): the SAME partition class on a 200K-node / 2M-edge graph
    of the same family, against the single-GPU projected-feature layer computed redundantly on every rank.  Returns the
    worst relative L2 error over the ranks of (out rows, dW, datt_src, dbias)."""
    import torch.distributed as dist
    from gnn_fraud_detection_b200 import GATConv, build_csr, functional as Fn, partition, synth
    n, e = 200_000, 2_000_000
    ei = synth.powerlaw_graph(n, e, seed=5, device=dev)
    x = torch.randn(n, K, device=dev, generator=torch.Generator(device=dev).manual_seed(10))
    torch.manual_seed(11)
    conv = GATConv(K, C, heads=H, concat=False).to(dev)
    W, bias = conv.lin_src.weight.detach(), conv.bias.detach()
    a_s, a_d = conv.att_src.detach().view(-1).contiguous(), conv.att_dst.detach().view(-1).contiguous()
    d_out = torch.randn(n, C, device=dev, generator=torch.Generator(device=dev).manual_seed(12)) / n
    g = build_csr(ei, n)
    xw, a_src, a_dst = Fn.project_fwd(x, W, a_s, a_d, H, C)
    out, rowmax, rowsum = Fn.gat_fwd(g, xw, a_src, a_dst, bias, H, C, 0.2, False)
    dxw, da_src, da_dst = Fn.gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C, 0.2, False)
    dW, datt_s, _, dbias, _ = Fn.project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C, C, False)
    part = partition_cls.build(ei, n, rank, world, dev)
    lo, hi = int(part.plan.start[rank]), int(part.plan.start[rank + 1])
    if isinstance(part, partition.InputSpacePartition):
        xp = torch.zeros(part.n_pos, Fn.in_sizes(0, K)[3], device=dev)
        xp[part.plan.to_pos(torch.arange(n, device=dev)), :K] = x
        xp = xp[:, :K]
    elif isinstance(part, partition.ReplicatedInputPartition):
        xp = torch.zeros(part.n_pos, K, device=dev)
        xp[part.plan.to_pos(torch.arange(n, device=dev))] = x
    else:
        xp = torch.zeros(part.rows_padded, K, device=dev)
        xp[:hi - lo] = x[lo:hi]
    o2, (dW2, ds2, _, db2) = part.layer_fwd_bwd(xp, W, a_s, a_d, bias, d_out[lo:hi].contiguous(), H, C, torch.float32, 0)
    rel = lambda a, b: float((a - b).norm() / b.norm().clamp_min(1e-30))
    errs = torch.tensor([rel(o2, out[lo:hi]), rel(dW2, dW), rel(ds2, datt_s), rel(db2, dbias)], device=dev)
    dist.all_reduce(errs, op=dist.ReduceOp.MAX)
    names = ["out", "dW", "datt_src", "dbias"]
    res = {k: float(v) for k, v in zip(names, errs.tolist())}
    res["graph"] = f"powerlaw N={n} E={e}"
    res["against"] = "single-GPU projected-feature layer on every rank"
    res["ok"] = bool(max(errs.tolist()) <= 3e-5)
    return res


def run_tgn_snapshots(args):
    """A step = one full-batch TRAINING step of the reference's TemporalGNN (2 GAT layers + BatchNorm/ReLU/residual tail +
    GRU head, src/models/tgn.py) with the reference's loss (masked BCE, pos_weight 50) over all 49 snapshots: every rank
    runs forward + backward on the block-diagonal batch of ITS snapshots (LPT-dealt; no edge crosses a time step, so the
    GAT layers need no communication), BatchNorm statistics are all-reduced (full-batch semantics, 2 x 64 doubles per
    layer) and the weight gradients are all-reduced once.  Metric: input edges of the whole graph per second."""
    import torch.distributed as dist
    from gnn_fraud_detection_b200 import TemporalGNN, _abi, fused, roofline, synth
    from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE
    from gnn_fraud_detection_b200.partition import snapshot_batches

    world, rank, local_rank = env_int("WORLD_SIZE", 1), env_int("RANK", 0), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _abi.lib()
    N, E, K = WORKLOADS["tgn_snapshots"]
    x, ei, ts = synth.elliptic_synth(N, E, K, seed=0, device=dev)
    y = (torch.rand(N, device=dev, generator=torch.Generator(device=dev).manual_seed(3)) < 0.1).long()
    y[torch.rand(N, device=dev, generator=torch.Generator(device=dev).manual_seed(4)) < 0.77] = -1     # ~23 % labelled
    torch.manual_seed(1)
    model = TemporalGNN(K, 64, 1, num_layers=2, dropout=0.0).to(dev).train()
    t0 = time.perf_counter()
    if world > 1:
        xl, el, ids = snapshot_batches(x, ei, ts, rank, world)
        xl, yl = xl.contiguous(), y[ids].contiguous()
        model.bn_group, model.bn_rows = dist.group.WORLD, N
    else:
        xl, el, yl = x, ei, y
    GLOBAL_CSR_CACHE.get(el, xl.size(0), True, True)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3
    params = [p for p in model.parameters()]
    n_lab = torch.tensor([float((yl != -1).sum())], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(n_lab)
    w_lab = float((yl != -1).sum()) / max(float(n_lab.item()), 1.0)        # this rank's share of the labelled nodes

    def step():
        for p in params:
            p.grad = None
        logits, _ = model(xl, el)
        loss, stats = fused.masked_bce_with_logits(logits, yl, 50.0)
        (loss * w_lab).backward()                        # global mean over labelled nodes = share-weighted local means
        flat = None
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in params])
            dist.all_reduce(flat)
        return loss, logits, flat

    def outputs(res):
        """What a caller of the step receives: the loss, the logits and the (all-reduced) parameter gradients."""
        loss, logits, flat = res
        names = [n for n, _ in model.named_parameters()]
        grads = [p.grad for p in params] if flat is None else flat.split([p.numel() for p in params])
        return output_sample({"loss": loss, "logits": logits,
                              **{f"grad.{n}": g.view(p.shape) for n, g, p in zip(names, grads, params)}})

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    L.gnnfd_launch_count_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    torch.cuda.synchronize()
    launches = int(L.gnnfd_launch_count())
    eager_ms = e0.elapsed_time(e1) / args.steps
    dumped = outputs(res) if args.dump_outputs and rank == 0 else None
    del res
    ms, graph_note = eager_ms, None
    if args.graph != "off":
        try:
            cg, cs = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=dev)
            cs.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(cs):
                step()
                cs.synchronize()
                with torch.cuda.graph(cg, stream=cs):
                    g_res = step()
            torch.cuda.current_stream().wait_stream(cs)
            for _ in range(3):
                cg.replay()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0.record()
            for _ in range(args.steps):
                cg.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            graph_note = "timed as K replays of ONE CUDA graph of the whole training step (launch-bound at this size)"
            if dumped is not None:
                dumped = outputs(g_res)
            del cg, g_res   # a live graph with captured collectives stalls destroy_process_group
            torch.cuda.synchronize()
        except Exception as ex:
            graph_note = f"CUDA graph capture failed ({type(ex).__name__}: {str(ex)[:120]}); eager timing reported"
    if world > 1:
        t = torch.tensor([ms, eager_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, eager_ms = float(t[0]), float(t[1])
    clocks = sampler.stop()
    peak, peak_src = load_peaks()
    Ep = E + N
    b1 = roofline.stage_bytes(N, Ep, K, H, C, False, 4, need_dx=False)["total"]
    b2 = roofline.stage_bytes(N, Ep, 64, H, C, False, 4, need_dx=True)["total"]
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu:
        threads = os.cpu_count() or 1
        cstep, _, _, _, _ = cpu_tgn_step_fn(threads)
        cstep()
        tc = time.perf_counter()
        cstep()
        cdt = time.perf_counter() - tc
        cpu = {"value": E / cdt, "unit": UNIT, "cores": threads, "kind": "port", "same_config": True, "ms_per_step": cdt * 1e3,
               "sample": "the same 203,769-node / 234,355-edge graph, TemporalGNN training step (oracle port of the reference's "
                         "PyG formulation)"}
    if rank == 0:
        line = {
            "metric": "tgn_train_step_edges_per_sec", "value": E / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "tgn_snapshots", "nodes": N, "edges": E, "in_features": K, "time_steps": 49, "layers": 2,
                       "l2": "working set (~0.7 GB) is L2-resident on purpose: this is the reference's real dataset size; the "
                             "headline HBM numbers are the powerlaw_200m workload",
                       "parallelism": "1 GPU" if world == 1 else f"time-step sharding x{world} (LPT on n_t + e_t): no data-path "
                                      f"collective; BatchNorm sums and weight gradients all-reduced",
                       "local_nodes": int(xl.size(0)), "local_edges": int(el.size(1)), "csr_build_ms": build_ms},
            "roofline": {"bound": "latency", "kernel": "whole training step (~90 launches)", "achieved": (b1 + b2) / (ms * 1e-3) / 1e9 / world,
                         "peak": peak, "unit": "GB/s", "frac": (b1 + b2) / (ms * 1e-3) / 1e9 / world / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes": b1 + b2,
                         "note": "two GAT layers' algorithmic bytes over the step time; at 4 GB per step the step is launch- and "
                                 "latency-bound, not HBM-bound"},
            "cpu_baseline": cpu, "e2e": None, "gpu_launches": launches, "clocks": clocks,
            "timing": {"eager_ms_per_step": eager_ms, "cuda_graph": graph_note},
        }
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_e2e(args, conv, x_host, ei_host, N, E_total, dev):
    """Same metric through the drop-in module with pinned HOST inputs: every step copies x and edge_index to
    the device (src/train.py:105 `batch.to(device)`), rebuilds the CSR (a fresh edge_index tensor, exactly as
    the reference's per-call self-loop rewrite), runs forward + backward, and reads the loss and the
    parameter gradients back (src/train.py:146-149)."""
    from gnn_fraud_detection_b200.graph import GLOBAL_CSR_CACHE
    steps = max(1, min(args.steps, args.e2e_steps))
    w_scale = 1.0 / N

    copy_stream = torch.cuda.Stream(device=dev)

    def one():
        GLOBAL_CSR_CACHE.clear()
        main = torch.cuda.current_stream()
        ed = ei_host.to(dev, non_blocking=True)
        # the feature copy (13 GB on the headline workload) rides the copy engine on its own stream while the
        # CSR/CSC build of the freshly arrived edge list runs on the SMs; GATConv accepts the prebuilt GraphCSR
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            xd = x_host.to(dev, non_blocking=True)
        g = GLOBAL_CSR_CACHE.get(ed, N, True, True)
        main.wait_stream(copy_stream)
        xd.record_stream(main)
        for p in conv.parameters():
            p.grad = None
        out = conv(xd, g)
        loss = out.sum() * w_scale
        loss.backward()
        res = [loss.detach().cpu()] + [p.grad.cpu() for p in conv.parameters()]
        return res

    one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = one()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    GLOBAL_CSR_CACHE.clear()
    h2d = x_host.numel() * x_host.element_size() + ei_host.numel() * ei_host.element_size()
    d2h = sum(t.numel() * t.element_size() for t in res)
    return {"value": E_total / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
            "ms_per_step": dt * 1e3, "includes": "H2D of x+edge_index (x copy overlapped with the CSR/CSC rebuild), fwd+bwd, D2H of loss+grads"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="powerlaw_200m", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", type=int, default=0, help="0 auto, 1 fp32 SIMT projection, 2 tensor-core projection, "
                    "3 input-space formulation (first layer)")
    ap.add_argument("--bf16", action="store_true", help="bf16 storage of projected features")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true", help="skip the multi-GPU parity self-check (outside the timed region)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="time the step as replays of one CUDA graph (auto: multi-GPU only)")
    ap.add_argument("--mgpu", default="input", choices=["input", "replicate", "allgather"],
                    help="multi-GPU variant of the destination-range partition (see partition.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "tgn_snapshots":
        return run_tgn_snapshots(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
