"""ctypes binding of ``libgnnfd_b200.so`` (the C ABI declared in ``include/gnnfd_b200.h``).

There is no fallback: if the shared library is missing or fails to load, importing the product path
raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` (or ``make -C
gnn_fraud_detection_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GNNFD_B200_LIB") or os.path.join(_HERE, "libgnnfd_b200.so")   # override: A/B runs of two builds

# enums (mirror include/gnnfd_b200.h)
ADD_SELF_LOOPS, BUILD_CSC, ORDER_DST_SRC = 1, 2, 4
F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_ELU = 0, 1, 2
GEMM_AUTO, GEMM_SIMT, GEMM_TC, GEMM_INPUT = 0, 1, 2, 3
HUB_THRESHOLD, HUB_CHUNK = 512, 512
ABI_VERSION = 22

_i32p = C.POINTER(C.c_int32)


class HubPlan(C.Structure):
    _fields_ = [("n_hub", C.c_int32), ("n_chunk", C.c_int32), ("threshold", C.c_int32), ("chunk", C.c_int32),
                ("hub_row", C.c_void_p), ("hub_chunk_ptr", C.c_void_p), ("chunk_hub", C.c_void_p)]


class ItemPlan(C.Structure):
    _fields_ = [("n_items", C.c_int32), ("target", C.c_int32), ("item_start", C.c_void_p)]


MAX_PEERS = 16


class Peers(C.Structure):
    """gnnfd_peers_t: the addresses of one symmetric buffer on every rank (+ its multicast mapping)."""
    _fields_ = [("n_peers", C.c_int32), ("rank", C.c_int32), ("ptr", C.c_void_p * MAX_PEERS), ("multicast", C.c_void_p)]


class Graph(C.Structure):
    _fields_ = [("n_dst", C.c_int64), ("n_src", C.c_int64), ("n_edges", C.c_int64),
                ("rowptr", C.c_void_p), ("col", C.c_void_p), ("perm", C.c_void_p),
                ("colptr", C.c_void_p), ("csc_row", C.c_void_p), ("csc_eid", C.c_void_p), ("csr2csc", C.c_void_p),
                ("hub_dst", HubPlan), ("hub_src", HubPlan), ("items_dst", ItemPlan), ("items_src", ItemPlan),
                ("edge_grads_indirect", C.c_int32), ("reserved_", C.c_int32)]


# name -> (restype, argtypes); every symbol include/gnnfd_b200.h declares
_vp, _sz, _i64, _i, _f, _u64 = C.c_void_p, C.c_size_t, C.c_int64, C.c_int, C.c_float, C.c_uint64
_szp, _i64p, _gp = C.POINTER(C.c_size_t), C.POINTER(C.c_int64), C.POINTER(Graph)
SIGNATURES = {
    "gnnfd_last_error": (C.c_char_p, []),
    "gnnfd_abi_version": (_i, []),
    "gnnfd_sizeof_graph": (_sz, []),
    "gnnfd_sizeof_hub_plan": (_sz, []),
    "gnnfd_sizeof_item_plan": (_sz, []),
    "gnnfd_item_plan": (_i, [_vp, _i64, _i64, C.c_int32, C.c_int32, _vp, _vp]),
    "gnnfd_invert_perm": (_i, [_vp, _i64, _vp, _vp]),
    "gnnfd_subgraph_workspace_bytes": (_i, [_i64, _i64, _szp]),
    "gnnfd_subgraph_build": (_i, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i64p, _vp, _sz, _vp]),
    "gnnfd_launch_count": (_i64, []),
    "gnnfd_launch_count_reset": (None, []),
    "gnnfd_shutdown": (_i, []),
    "gnnfd_csr_workspace_bytes": (_i, [_i64, _i64, _i, _szp]),
    "gnnfd_csr_build": (_i, [_vp, _i64, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i64p, _vp, _sz, _vp]),
    "gnnfd_hub_plan_workspace_bytes": (_i, [_i64, _szp]),
    "gnnfd_hub_plan": (_i, [_vp, _i64, C.c_int32, C.c_int32, _vp, _vp, _vp, _i64, _i64, _i64p, _vp, _sz, _vp]),
    "gnnfd_project_workspace_bytes": (_i, [_i64, _i64, _i, _i, _i, _szp]),
    "gnnfd_project_fwd": (_i, [_vp, _i64, _vp, _vp, _vp, _i64, _i64, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_project_image_bytes": (_i, [_i64, _i64, _szp, _szp]),
    "gnnfd_project_image_build": (_i, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "gnnfd_project_fwd_image": (_i, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_gat_fwd_workspace_bytes": (_i, [_gp, _i, _i, _szp]),
    "gnnfd_dropout_mask": (_i, [_u64, _f, _i64, _i, _vp, C.POINTER(C.c_float), _vp]),
    "gnnfd_set_dropout_seed_source": (None, [_vp]),
    "gnnfd_gat_fwd": (_i, [_gp, _vp, _i, _vp, _vp, _vp, _i, _i, _f, _i, _i, _vp, _f, _u64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_gat_fwd_fused": (_i, [_gp, _vp, _i, _vp, _vp, _vp, _i, _i, _f, _i, _i, _vp, _f, _u64, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _sz, _vp]),
    "gnnfd_gat_alpha": (_i, [_gp, _vp, _vp, _vp, _vp, _i, _f, _vp, _vp]),
    "gnnfd_gat_bwd_workspace_bytes": (_i, [_gp, _i, _i, _szp]),
    "gnnfd_gat_bwd_dst": (_i, [_gp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp, _f, _u64, _vp, _vp, _vp, _vp,
                               _sz, _vp]),
    "gnnfd_gat_bwd_src": (_i, [_gp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_project_bwd_workspace_bytes": (_i, [_i64, _i64, _i, _i, _i, _szp]),
    "gnnfd_project_bwd": (_i, [_vp, _i64, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i64, _i64, _i, _i, _i, _i, _vp, _vp,
                               _vp, _vp, _vp, _i64, _vp, _sz, _vp]),
    "gnnfd_project_dx_workspace_bytes": (_i, [_i64, _i64, _i, _i, _szp]),
    "gnnfd_project_dx": (_i, [_vp, _vp, _i64, _i64, _i, _i, _vp, _i64, _vp, _sz, _vp]),
    # input-space formulation
    "gnnfd_in_supported": (_i, [_i64, _i, _i, _i]),
    "gnnfd_in_sizes": (_i, [_i64, _i64, _szp, _szp, _i64p, _i64p]),
    "gnnfd_in_pad_x": (_i, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "gnnfd_in_logits": (_i, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gnnfd_in_logits_bcast": (_i, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, C.POINTER(Peers), _i64, _i, _vp, _vp, _vp, _vp]),
    "gnnfd_peer_reduce": (_i, [C.POINTER(Peers), _i64, _i64, _i, _i, _vp, _vp]),
    "gnnfd_in_prepare": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "gnnfd_in_fwd_workspace_bytes": (_i, [_gp, _szp]),
    "gnnfd_in_fwd": (_i, [_gp, _vp, _i64, _i64, _vp, _vp, _f, _vp, _f, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_in_out": (_i, [_vp, _i64, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "gnnfd_in_out_bcast": (_i, [_vp, _i64, _i64, _vp, _vp, _i, _vp, _vp, _vp, C.POINTER(Peers), _i64, _i, _vp, _vp]),
    "gnnfd_in_bwd_gd_workspace_bytes": (_i, [_i64, _szp]),
    "gnnfd_in_bwd_gd": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "gnnfd_in_bwd_edges_workspace_bytes": (_i, [_gp, _szp]),
    "gnnfd_in_bwd_edges": (_i, [_gp, _vp, _i64, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _f, _vp, _f,
                                _u64, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "gnnfd_in_bwd_dasrc": (_i, [_gp, _vp, _vp, _vp]),
    "gnnfd_in_bwd_params_workspace_bytes": (_i, [_i64, _i64, _szp]),
    "gnnfd_in_bwd_params": (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                 _i, _vp]),
    # model-level fused operators
    "gnnfd_model_ops_workspace_bytes": (_i, [_i64, _szp]),
    "gnnfd_bn_sums": (_i, [_vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "gnnfd_bn_finalize": (_i, [_vp, C.c_double, _i, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    "gnnfd_bn_relu_drop_res_fwd": (_i, [_vp, _i64, _i, _vp, _vp, _vp, _vp, _f, _u64, _i64, _vp, _vp, _vp]),
    "gnnfd_bn_relu_drop_res_fwd_bcast": (_i, [_vp, _i64, _i, _vp, _vp, _vp, _vp, _f, _u64, _i64, _vp, C.POINTER(Peers), _i64, _i,
                                             _vp, _vp]),
    "gnnfd_bn_bwd_sums": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp, _f, _u64, _i64, _vp, _vp, _sz, _vp]),
    "gnnfd_bn_bwd_apply": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp, _f, _u64, _i64, _vp, C.c_double, _vp, _vp, _vp, _vp]),
    "gnnfd_gru_head_fwd": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gnnfd_gru_head_bwd": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _sz, _vp]),
    "gnnfd_bce_masked": (_i, [_vp, _vp, _i64, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    # neighbour sampling
    "gnnfd_sample_workspace_bytes": (_i, [_i64, _i64, C.c_int32, _szp]),
    "gnnfd_neighbor_sample": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i32p, C.c_int32, _u64, _vp, _vp, _i64, _vp, _i64, _vp,
                                   _i64, _i64p, _vp, _sz, _vp]),
}


class GnnfdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libgnnfd_b200 error {code}: {msg}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """Load (once) and type the shared library.  Raises if it is missing -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is required (no CPU/PyTorch fallback). "
            "Build it with `python -c 'import __graft_entry__ as g; g.build()'`.")
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(l, name)  # AttributeError => a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if l.gnnfd_abi_version() != ABI_VERSION:
        raise ImportError(f"libgnnfd_b200 ABI {l.gnnfd_abi_version()} != binding {ABI_VERSION}; rebuild")
    if (l.gnnfd_sizeof_graph() != C.sizeof(Graph) or l.gnnfd_sizeof_hub_plan() != C.sizeof(HubPlan)
            or l.gnnfd_sizeof_item_plan() != C.sizeof(ItemPlan)):
        raise ImportError("gnnfd_graph_t layout mismatch between header and ctypes binding")
    _lib = l
    return l


def check(rc: int) -> None:
    if rc != 0:
        raise GnnfdError(rc, lib().gnnfd_last_error().decode("utf-8", "replace"))


def ptr(t) -> int:
    """data_ptr of a tensor or 0 for None."""
    return 0 if t is None else t.data_ptr()
