"""Algorithmic-byte model of one GATConv layer (SURVEY.md section 8(d); restated in DESIGN.md).

Gather traffic is charged per edge (no credit for cache reuse); indices are int32 (i = 4 B); logits,
row statistics, gradients are fp32; ``s`` is the storage size of a projected feature element (4 fp32 /
2 bf16); ``Co`` = C (head mean) or H*C (concat).  ``Ep`` is E' (edges after the self-loop rewrite).
The ``gat_fwd`` and ``gat_bwd_dst`` terms describe the kernels that run: for the head mean on one node set
(``n_src`` not given) the source-major forms (forward: attention pass, source-major messages, row sums; backward:
d_alpha computed source-major, then a dst pass that reads no features), otherwise the gather passes (the backward's
two-pass form also runs for a head-mean partition with ``n_src``).
"""
from __future__ import annotations


def stage_bytes(N: int, Ep: int, K: int, H: int = 8, C: int = 64, concat: bool = False, s: int = 4,
                need_dx: bool = False, n_src: int | None = None) -> dict:
    D, i = H * C, 4
    Co = D if concat else C
    Ns = N if n_src is None else n_src
    b = {}
    # x read, xw write, a_src/a_dst write, W read
    b["project_fwd"] = N * (K * 4 + D * s + 8 * H) + K * D * 4
    if concat or n_src is not None:
        # gather pass -- per edge: xw[src] row, col, a_src[src]; per row: a_dst, out, (max,sum), rowptr
        b["gat_fwd"] = Ep * (D * s + i + 4 * H) + N * (4 * H + 4 * Co + 8 * H + i)
    else:
        # head mean, three passes (DESIGN 4.3).  Attention -- per edge: col, a_src[src], alpha_used write; per row:
        # a_dst, (max,sum), rowptr.  Messages -- per edge: csc_eid, alpha_used[eid], v write; per source row: xw row,
        # colptr.  Sums -- per edge: v read; per row: out, rowptr
        b["gat_fwd"] = (Ep * (i + 4 * H + 4 * H) + N * (4 * H + 8 * H + i)
                        + Ep * (i + 4 * H + 4 * C) + Ns * (D * s + i)
                        + Ep * 4 * C + N * (4 * Co + i))
    if concat:
        # one gather pass -- per edge: xw[src] row, col, a_src[src], dz write (alpha write is not charged, as in
        # SURVEY 8(d)); per row: dOut, (a_dst,max,sum), da_dst, rowptr
        b["gat_bwd_dst"] = Ep * (D * s + i + 4 * H + 4 * H) + N * (4 * Co + 8 * H + 4 * H + i)
    else:
        # head mean, two passes (DESIGN 4.4).  Source-major d_alpha stream -- per edge: csc_row, csc_eid, dOut[dst]
        # row, record {d_alpha, a_src[src]} write (CSR position); per source row: xw row, a_src, colptr.  Dst pass --
        # per edge: record read, csr2csc, (alpha_used, dz) write; per row: (a_dst,max,sum), da_dst, rowptr.  The record
        # costs 4H B more per edge than a bare d_alpha and saves the col read, but it turns the dst pass's one random
        # gather (a_src[col[e]]) into a contiguous stream
        b["gat_bwd_dst"] = (Ep * (2 * i + 4 * Co + 8 * H) + Ns * (D * s + 4 * H + i)
                            + Ep * (8 * H + i + 8 * H) + N * (12 * H + 4 * H + i))
    # per edge: dOut[dst] row, (csc_row, csc_eid), alpha, dz; per source row: dxw write, da_src write, colptr
    b["gat_bwd_src"] = Ep * (4 * Co + 2 * i + 4 * H + 4 * H) + Ns * (D * 4 + 4 * H + i)
    # GEMM-bwd: read dxw, xw, x (+ dx write), da_src/da_dst; W read + dW write
    b["project_bwd"] = Ns * (D * 4 + D * s + K * 4 + (K * 4 if need_dx else 0) + 8 * H) + 2 * K * D * 4
    b["fwd"] = b["project_fwd"] + b["gat_fwd"]
    b["bwd"] = b["gat_bwd_dst"] + b["gat_bwd_src"] + b["project_bwd"]
    b["total"] = b["fwd"] + b["bwd"]
    return b


def stage_flops(N: int, Ep: int, K: int, H: int = 8, C: int = 64, need_dx: bool = False) -> dict:
    D = H * C
    return {
        "project_fwd": 2 * N * K * D,
        "project_bwd": 2 * N * K * D * (2 if need_dx else 1),
        "gat_fwd": Ep * H * (2 * C + 10),
        "gat_bwd": Ep * H * (4 * C + 20),
    }


def stage_bytes_input_space(N: int, Ep: int, K: int, H: int = 8, C: int = 64, n_src: int | None = None) -> dict:
    """Algorithmic bytes of the input-space formulation of the first layer (csrc/in_common.cuh): per-edge gathers are
    x rows (K*4 B) instead of projected rows (H*C*4 B); the aggregated input Z [N, H*KP] (fp16 pair = 4 B/element) is
    written once and read by the two tensor-core GEMMs; Gd [N, H*KP] fp32 is written and read once.  Same charging
    rules as ``stage_bytes`` (gathers per edge, no credit for cache reuse)."""
    i = 4
    KP = (K + 7) // 8 * 8
    F = H * KP
    Ns = N if n_src is None else n_src
    b = {}
    b["in_logits"] = N * (K * 4 + 8 * H)
    # per edge: x[src] row, col, a_src[src]; per row: a_dst, (max,sum), rowptr, Z row
    b["in_fwd_edges"] = Ep * (K * 4 + i + 4 * H) + N * (4 * H + 8 * H + i + F * 4)
    b["in_out_gemm"] = N * (F * 4 + 4 * C) + F * C * 4
    b["in_bwd_gd"] = N * (4 * C + F * 4)
    # per edge: x[src] row, col, a_src[src], csr2csc, dz write; per row: Gd row, (a_dst,max,sum), da_dst, rowptr
    b["in_bwd_edges"] = Ep * (K * 4 + i + 4 * H + i + 4 * H) + N * (F * 4 + 12 * H + 4 * H + i)
    b["in_bwd_dasrc"] = Ep * 4 * H + Ns * (4 * H + i)
    # dW GEMM reads Z and dOut; da^T x reads x and the logit gradients; dbias reads dOut
    b["in_bwd_params"] = N * (F * 4 + 4 * C + K * 4 + 8 * H + 4 * C) + 2 * K * H * C * 4
    b["fwd"] = b["in_logits"] + b["in_fwd_edges"] + b["in_out_gemm"]
    b["bwd"] = b["in_bwd_gd"] + b["in_bwd_edges"] + b["in_bwd_dasrc"] + b["in_bwd_params"]
    b["total"] = b["fwd"] + b["bwd"]
    return b
