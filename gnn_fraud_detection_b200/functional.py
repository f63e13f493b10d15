"""``torch.autograd.Function`` over the C ABI: one GATConv layer, forward and backward.

PyTorch is used here for device memory, streams and autograd bookkeeping only; every arithmetic step
of the layer runs in ``libgnnfd_b200.so``.  Mirrors ``GATConv.forward`` as called at
``src/models/gat.py:80`` / ``src/models/tgn.py:94`` and its autograd backward (``src/train.py:142``).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _abi
from .graph import GraphCSR, _stream

_DT = {torch.float32: _abi.F32, torch.bfloat16: _abi.BF16}


def _ws(nbytes: int, device) -> Optional[torch.Tensor]:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _aligned_u8(nbytes: int, device, align: int = 1024) -> torch.Tensor:
    """uint8 buffer whose data_ptr is ``align``-byte aligned (torch guarantees only 512)."""
    raw = torch.empty(int(nbytes) + align, dtype=torch.uint8, device=device)
    off = (-raw.data_ptr()) % align
    return raw[off: off + int(nbytes)]


def _require_f32_cuda(name: str, t: torch.Tensor):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the B200 path has no CPU fallback")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")


def project_fwd(x, W, att_src, att_dst, H, C_, xw_dtype=torch.float32, algo=_abi.GEMM_AUTO, out=None):
    """xw [N,H*C] (xw_dtype), a_src [N,H], a_dst [N,H] = gnnfd_project_fwd(x, W, att).

    ``out=(xw, a_src, a_dst)`` writes into caller-provided contiguous buffers (e.g. this rank's slice of an
    all-gather buffer)."""
    L = _abi.lib()
    N, K = x.shape
    dev = x.device
    if out is not None:
        xw, a_src, a_dst = out
        assert xw.is_contiguous() and a_src.is_contiguous() and a_dst.is_contiguous() and xw.dtype == xw_dtype
        assert xw.shape == (N, H * C_) and a_src.shape == (N, H) and a_dst.shape == (N, H)
    else:
        xw = torch.empty(N, H * C_, dtype=xw_dtype, device=dev)
        a_src = torch.empty(N, H, dtype=torch.float32, device=dev)
        a_dst = torch.empty(N, H, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_project_workspace_bytes(N, K, H, C_, algo, C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_project_fwd(x.data_ptr(), x.stride(0), W.data_ptr(), att_src.data_ptr(), att_dst.data_ptr(),
                                   N, K, H, C_, _DT[xw_dtype], algo, xw.data_ptr(), a_src.data_ptr(),
                                   a_dst.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    return xw, a_src, a_dst


class XImage:
    """The fp16-pair tensor-core image of a static layer input (``gnnfd_project_image_build``) + its per-row scales."""

    def __init__(self, x: torch.Tensor):
        N, K = x.shape
        ib, _ = C.c_size_t(), None
        wb = C.c_size_t()
        _abi.check(_abi.lib().gnnfd_project_image_bytes(N, K, C.byref(ib), C.byref(wb)))
        self.N, self.K, self.ws_bytes = N, K, wb.value
        self.img = _aligned_u8(ib.value, x.device)
        self.row_scale = torch.empty(max(N, 1), dtype=torch.float32, device=x.device)
        xc = x if x.stride(1) == 1 else x.contiguous()
        with torch.cuda.device(x.device):
            _abi.check(_abi.lib().gnnfd_project_image_build(xc.data_ptr(), xc.stride(0), N, K, self.img.data_ptr(),
                                                            self.row_scale.data_ptr(), _stream()))


class XImageCache:
    """Images of STATIC inputs, keyed on the identity of ``x`` (data_ptr, shape, strides, version) like the CSR cache; an
    entry dies with its tensor.  The image is built the SECOND time the same tensor is seen: a fresh ``x`` every step (the
    reference's ``batch.to(device)``, ``src/train.py:105``) never pays the extra pass and the extra 768 B per row -- it takes
    the register-staged GEMM -- while a resident input is projected from its image from the second step on."""

    def __init__(self, capacity: int = 4):
        import weakref
        from collections import OrderedDict
        self._weakref, self.capacity, self._d = weakref, capacity, OrderedDict()

    def get(self, x: torch.Tensor):
        """The cached image of ``x``, or ``None`` when ``x`` is seen for the first time (or cannot be tracked)."""
        if x.is_inference():
            return None
        key = (x.data_ptr(), tuple(x.shape), tuple(x.stride()), x._version, x.device.index)
        hit = self._d.get(key)
        if hit is not None and hit[1]() is x:
            self._d.move_to_end(key)
            if hit[0] is None:                          # second sight: the input is static, build its image now
                hit = (XImage(x), hit[1])
                self._d[key] = hit
            return hit[0]
        self._weakref.finalize(x, self._d.pop, key, None)
        self._d[key] = (None, self._weakref.ref(x))
        while len(self._d) > self.capacity:
            self._d.popitem(last=False)
        return None

    def clear(self):
        self._d.clear()


GLOBAL_XIMAGE_CACHE = XImageCache()
IMAGE_PROJECTION = True       # first-layer projection from the cached image (False: always stage x inside the GEMM)


def image_projection_applies(x, H, C_, xw_dtype, algo) -> bool:
    return (IMAGE_PROJECTION and algo in (_abi.GEMM_AUTO, _abi.GEMM_TC) and xw_dtype == torch.float32 and H == 8 and C_ == 64
            and 64 < x.size(1) <= 192 and x.size(0) > 0 and torch.cuda.get_device_capability(x.device)[0] == 10)


def project_fwd_image(img: XImage, W, att_src, att_dst, out=None):
    """xw [N,512] fp32, a_src / a_dst [N,8] from the cached image of x (same results as ``project_fwd``)."""
    N, dev = img.N, img.img.device
    if out is not None:
        xw, a_src, a_dst = out
    else:
        xw = torch.empty(N, 512, dtype=torch.float32, device=dev)
        a_src = torch.empty(N, 8, dtype=torch.float32, device=dev)
        a_dst = torch.empty(N, 8, dtype=torch.float32, device=dev)
    ws = _aligned_u8(img.ws_bytes, dev)
    _abi.check(_abi.lib().gnnfd_project_fwd_image(img.img.data_ptr(), img.row_scale.data_ptr(), N, img.K, W.data_ptr(),
                                                  att_src.data_ptr(), att_dst.data_ptr(), xw.data_ptr(), a_src.data_ptr(),
                                                  a_dst.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    return xw, a_src, a_dst


def gat_fwd(g: GraphCSR, xw, a_src, a_dst, bias, H, C_, negative_slope, concat, act=_abi.ACT_NONE, keep_mask=None,
            p_drop=0.0, post_scale=None, post_shift=None, residual=None, seed=0):
    """Fused softmax/aggregation.  ``post_scale``/``post_shift`` [Co] (folded eval-mode BatchNorm), ``act`` and
    ``residual`` [n_dst,Co] are applied in the row epilogue: ``act((mean+bias)*scale+shift) + residual``."""
    L = _abi.lib()
    dev = xw.device
    Co = H * C_ if concat else C_
    out = torch.empty(g.n_dst, Co, dtype=torch.float32, device=dev)
    rowmax = torch.empty(g.n_dst, H, dtype=torch.float32, device=dev)
    rowsum = torch.empty(g.n_dst, H, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_gat_fwd_workspace_bytes(g.ref(), H, C_, C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_gat_fwd_fused(g.ref(), xw.data_ptr(), _DT[xw.dtype], a_src.data_ptr(), a_dst.data_ptr(),
                                     _abi.ptr(bias), H, C_, float(negative_slope), int(concat), int(act),
                                     _abi.ptr(keep_mask), float(p_drop), int(seed), _abi.ptr(post_scale), _abi.ptr(post_shift),
                                     _abi.ptr(residual), out.data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(),
                                     ws.data_ptr(), ws.numel(), _stream()))
    return out, rowmax, rowsum


def dropout_mask(seed: int, p_drop: float, n_edges: int, H: int, device):
    """The keep bits the kernels derive from ``seed`` (counter-based RNG), as a [E',H] uint8 mask in edge_index' order,
    and the survivor scale.  Test hook: the kernels never materialise this tensor."""
    keep = torch.empty(n_edges, H, dtype=torch.uint8, device=device)
    scale = C.c_float()
    with torch.cuda.device(device):
        _abi.check(_abi.lib().gnnfd_dropout_mask(int(seed), float(p_drop), int(n_edges), int(H), keep.data_ptr(),
                                                 C.byref(scale), _stream()))
    return keep, scale.value


def gat_alpha(g: GraphCSR, a_src, a_dst, rowmax, rowsum, H, negative_slope):
    """alpha [E',H] in CSR (dst-sorted) order."""
    L = _abi.lib()
    alpha = torch.empty(g.n_edges, H, dtype=torch.float32, device=a_src.device)
    _abi.check(L.gnnfd_gat_alpha(g.ref(), a_src.data_ptr(), a_dst.data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(),
                                 H, float(negative_slope), alpha.data_ptr(), _stream()))
    return alpha


def gat_bwd(g: GraphCSR, xw, a_src, a_dst, rowmax, rowsum, d_out, att_src, att_dst, H, C_, negative_slope, concat,
            keep_mask=None, p_drop=0.0, da_dst_full="same", da_dst_view=None, seed=0):
    """dst-major + src-major backward passes.  Returns dxw [n_src,H*C], da_src [n_src,H], da_dst [n_dst,H].

    For a destination-range partition ``da_dst_full`` is a zero ``[n_src,H]`` buffer in source-position space
    and ``da_dst_view=(lo, n)`` says where this rank's ``da_dst`` rows belong in it."""
    alpha_used, dz, da_dst = gat_bwd_dst(g, xw, a_src, a_dst, rowmax, rowsum, d_out, H, C_, negative_slope, concat,
                                         keep_mask, p_drop, seed)
    full = da_dst if isinstance(da_dst_full, str) else da_dst_full
    if da_dst_view is not None:
        lo, n = da_dst_view
        full[lo:lo + n].copy_(da_dst)
    dxw, da_src = gat_bwd_src(g, alpha_used, dz, d_out, att_src, att_dst, full, H, C_, concat)
    return dxw, da_src, da_dst


def gat_bwd_dst(g: GraphCSR, xw, a_src, a_dst, rowmax, rowsum, d_out, H, C_, negative_slope, concat, keep_mask=None,
                p_drop=0.0, seed=0):
    """dst-major pass: alpha_used [E',H], dz [E',H] (views of one interleaved [E',2H] buffer, rows in source-major
    order) and da_dst [n_dst,H]."""
    L = _abi.lib()
    dev = xw.device
    # one interleaved [E', 2H] buffer: row = (alpha_used[0..H), dz[0..H)) of an edge, 64 contiguous bytes; the
    # library recognises the layout from dz == alpha_used + H
    eg = torch.empty(g.n_edges, 2 * H, dtype=torch.float32, device=dev)
    alpha_used, dz = eg[:, :H], eg[:, H:]
    da_dst = torch.empty(g.n_dst, H, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_gat_bwd_workspace_bytes(g.ref(), H, C_, C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_gat_bwd_dst(g.ref(), xw.data_ptr(), _DT[xw.dtype], a_src.data_ptr(), a_dst.data_ptr(),
                                   rowmax.data_ptr(), rowsum.data_ptr(), d_out.data_ptr(), H, C_,
                                   float(negative_slope), int(concat), _abi.ptr(keep_mask), float(p_drop), int(seed),
                                   alpha_used.data_ptr(), dz.data_ptr(), da_dst.data_ptr(), ws.data_ptr(),
                                   ws.numel(), _stream()))
    return alpha_used, dz, da_dst


def gat_bwd_src(g: GraphCSR, alpha_used, dz, d_out, att_src, att_dst, da_dst_full, H, C_, concat, da_src_out=None):
    """src-major pass over g's CSC: dxw [n_src,H*C] and da_src [n_src,H] (written into ``da_src_out`` if given)."""
    L = _abi.lib()
    dev = alpha_used.device
    dxw = torch.empty(g.n_src, H * C_, dtype=torch.float32, device=dev)
    if da_src_out is not None and (tuple(da_src_out.shape) != (g.n_src, H) or da_src_out.dtype != torch.float32
                                   or not da_src_out.is_contiguous() or da_src_out.device != dev):
        raise ValueError(f"da_src_out must be a contiguous float32 [{g.n_src},{H}] tensor on {dev}")
    da_src = da_src_out if da_src_out is not None else torch.empty(g.n_src, H, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_gat_bwd_workspace_bytes(g.ref(), H, C_, C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_gat_bwd_src(g.ref(), alpha_used.data_ptr(), dz.data_ptr(), d_out.data_ptr(),
                                   att_src.data_ptr(), att_dst.data_ptr(), _abi.ptr(da_dst_full), H, C_, int(concat),
                                   dxw.data_ptr(), da_src.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    return dxw, da_src


def project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C_, Co, need_dx, algo=_abi.GEMM_AUTO):
    L = _abi.lib()
    N, K = x.shape
    dev = x.device
    dW = torch.empty(H * C_, K, dtype=torch.float32, device=dev)
    datt_src = torch.empty(H * C_, dtype=torch.float32, device=dev)
    datt_dst = torch.empty(H * C_, dtype=torch.float32, device=dev)
    dbias = torch.empty(Co, dtype=torch.float32, device=dev)
    dx = torch.empty(N, K, dtype=torch.float32, device=dev) if need_dx else None
    nb = C.c_size_t()
    _abi.check(L.gnnfd_project_bwd_workspace_bytes(N, K, H, C_, algo, C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_project_bwd(x.data_ptr(), x.stride(0), W.data_ptr(), dxw.data_ptr(), xw.data_ptr(),
                                   _DT[xw.dtype], da_src.data_ptr(), da_dst.data_ptr(), d_out.data_ptr(), N, K, H, C_,
                                   Co, algo, dW.data_ptr(), datt_src.data_ptr(), datt_dst.data_ptr(),
                                   dbias.data_ptr(), _abi.ptr(dx), K, ws.data_ptr(), ws.numel(), _stream()))
    return dW, datt_src, datt_dst, dbias, dx


def project_dx(dxw, W, H, C_, out=None):
    """dx [N,K] = dxw [N,H*C] W: the dx GEMM of ``project_bwd`` alone (for a layer that has no xw).  ``out``: an [N,K] view
    with unit column stride to write into (e.g. a symmetric buffer the ranks reduce from)."""
    L = _abi.lib()
    N, K = dxw.size(0), W.size(1)
    if out is not None and (tuple(out.shape) != (N, K) or out.stride(1) != 1 or out.dtype != torch.float32):
        raise ValueError(f"out must be float32 [{N},{K}] with unit column stride")
    dx = out if out is not None else torch.empty(N, K, dtype=torch.float32, device=dxw.device)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_project_dx_workspace_bytes(N, K, H, C_, C.byref(nb)))
    ws = _ws(nb.value, dxw.device)
    _abi.check(L.gnnfd_project_dx(dxw.data_ptr(), W.data_ptr(), N, K, H, C_, dx.data_ptr(), dx.stride(0), ws.data_ptr(),
                                  ws.numel(), _stream()))
    return dx


# ------------------------------------------------------------------------------------------------
# input-space formulation (include/gnnfd_b200.h section (5), csrc/in_common.cuh)
# ------------------------------------------------------------------------------------------------
def in_supported(K: int, H: int, C_: int, concat: bool) -> bool:
    return bool(_abi.lib().gnnfd_in_supported(int(K), int(H), int(C_), int(bool(concat))))


def in_sizes(n_dst: int, K: int):
    """(prep bytes, image bytes, leading dimension of Gd, leading dimension of the padded x)."""
    pb, zb, ld, xld = C.c_size_t(), C.c_size_t(), C.c_int64(), C.c_int64()
    _abi.check(_abi.lib().gnnfd_in_sizes(int(n_dst), int(K), C.byref(pb), C.byref(zb), C.byref(ld), C.byref(xld)))
    return pb.value, zb.value, ld.value, xld.value


def in_pad_x(x: torch.Tensor) -> torch.Tensor:
    """x [N,K] -> view [N,K] of a zero-padded [N, round_up(K,8)] copy (16-byte aligned rows for the bulk-copy gathers);
    returns ``x`` itself when it already has that layout."""
    N, K = x.shape
    xld = in_sizes(0, K)[3]
    if x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.stride(0) >= xld and x.data_ptr() % 16 == 0:
        return x
    if x.stride(1) != 1:
        x = x.contiguous()
    x16 = torch.empty(N, xld, dtype=torch.float32, device=x.device)
    _abi.check(_abi.lib().gnnfd_in_pad_x(x.data_ptr(), x.stride(0), N, K, x16.data_ptr(), _stream()))
    return x16[:, :K]


def in_logits(x, W, att_src, att_dst, prep, xmax, n_rows=None):
    """a_src, a_dst [n,H] straight from the rows of ``x``; accumulates max|x| into ``xmax`` (a zeroed 1-element tensor)."""
    N, K = x.shape if n_rows is None else (n_rows, x.size(1))
    a_src = torch.empty(N, 8, dtype=torch.float32, device=x.device)
    a_dst = torch.empty(N, 8, dtype=torch.float32, device=x.device)
    _abi.check(_abi.lib().gnnfd_in_logits(x.data_ptr(), x.stride(0), N, K, W.data_ptr(), att_src.data_ptr(),
                                          att_dst.data_ptr(), a_src.data_ptr(), a_dst.data_ptr(), xmax.data_ptr(),
                                          prep.data_ptr(), _stream()))
    return a_src, a_dst


def in_logits_bcast(x, W, att_src, att_dst, prep, xmax, peers, row_offset, use_multicast=False):
    """``in_logits`` fused with the all-gather of ``a_src``: the rows go to ``row_offset ..`` of the symmetric buffer described
    by ``peers`` (``_abi.Peers``) on EVERY rank; returns the local ``a_dst``."""
    N, K = x.shape
    a_dst = torch.empty(N, 8, dtype=torch.float32, device=x.device)
    _abi.check(_abi.lib().gnnfd_in_logits_bcast(x.data_ptr(), x.stride(0), N, K, W.data_ptr(), att_src.data_ptr(),
                                                att_dst.data_ptr(), C.byref(peers), int(row_offset), int(use_multicast),
                                                a_dst.data_ptr(), xmax.data_ptr(), prep.data_ptr(), _stream()))
    return a_dst


def peer_reduce(peers, offset, n, out, op="sum", use_multicast=False):
    """``out[:n]`` = sum / max over ranks of the symmetric buffer's elements ``offset .. offset+n`` (peer loads, or the
    in-switch ``multimem.ld_reduce``)."""
    _abi.check(_abi.lib().gnnfd_peer_reduce(C.byref(peers), int(offset), int(n), 0 if op == "sum" else 1, int(use_multicast),
                                            out.data_ptr(), _stream()))
    return out


def in_prepare(W, K, xmax, prep):
    _abi.check(_abi.lib().gnnfd_in_prepare(W.data_ptr(), int(K), xmax.data_ptr(), prep.data_ptr(), _stream()))


class InAttention:
    """What the input-space forward saves for the backward: ``alpha [E',H]`` (CSR order, normalised, before dropout; sign bit =
    LeakyReLU negative region), ``jflag [E']`` (source id | row-end flag), ``rowmax`` / ``rowsum [n_dst,H]``."""
    __slots__ = ("alpha", "jflag", "rowmax", "rowsum")

    def __init__(self, alpha, jflag, rowmax, rowsum):
        self.alpha, self.jflag, self.rowmax, self.rowsum = alpha, jflag, rowmax, rowsum


def in_fwd(g: GraphCSR, x, a_src, a_dst, negative_slope, prep, keep_mask=None, p_drop=0.0, seed=0):
    """Aggregation in input space -> (zimg, InAttention)."""
    L = _abi.lib()
    dev, K = x.device, x.size(1)
    zb = in_sizes(g.n_dst, K)[1]
    zimg = _aligned_u8(zb, dev)
    rowmax = torch.empty(g.n_dst, 8, dtype=torch.float32, device=dev)
    rowsum = torch.empty(g.n_dst, 8, dtype=torch.float32, device=dev)
    alpha = torch.empty(max(g.n_edges, 1), 8, dtype=torch.float32, device=dev)
    jflag = torch.empty(max(g.n_edges, 1), dtype=torch.int32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_in_fwd_workspace_bytes(g.ref(), C.byref(nb)))
    ws = _ws(nb.value, dev)
    _abi.check(L.gnnfd_in_fwd(g.ref(), x.data_ptr(), x.stride(0), K, a_src.data_ptr(), a_dst.data_ptr(),
                              float(negative_slope), _abi.ptr(keep_mask), float(p_drop), int(seed), prep.data_ptr(),
                              zimg.data_ptr(), rowmax.data_ptr(), rowsum.data_ptr(), alpha.data_ptr(), jflag.data_ptr(),
                              ws.data_ptr(), ws.numel(), _stream()))
    return zimg, InAttention(alpha, jflag, rowmax, rowsum)


def in_out(zimg, n, K, prep, bias, act=_abi.ACT_NONE, post_scale=None, post_shift=None, residual=None, out=None):
    if out is None:
        out = torch.empty(n, 64, dtype=torch.float32, device=zimg.device)
    _abi.check(_abi.lib().gnnfd_in_out(zimg.data_ptr(), int(n), int(K), prep.data_ptr(), _abi.ptr(bias), int(act),
                                       _abi.ptr(post_scale), _abi.ptr(post_shift), _abi.ptr(residual), out.data_ptr(),
                                       _stream()))
    return out


def in_out_bcast(zimg, n, K, prep, bias, peers, row_offset, use_multicast=False, act=_abi.ACT_NONE, post_scale=None,
                 post_shift=None, residual=None, out=None):
    """``in_out`` fused with the all-gather of its rows: row ``r`` also goes to row ``row_offset + r`` of the symmetric
    ``[n_pos, 64]`` buffer described by ``peers`` (``_abi.Peers``) on EVERY rank.  ``out`` (the own rows) is optional;
    returns it."""
    _abi.check(_abi.lib().gnnfd_in_out_bcast(zimg.data_ptr(), int(n), int(K), prep.data_ptr(), _abi.ptr(bias), int(act),
                                             _abi.ptr(post_scale), _abi.ptr(post_shift), _abi.ptr(residual), C.byref(peers),
                                             int(row_offset), int(use_multicast), _abi.ptr(out), _stream()))
    return out


IN_GD_BLOCK_BYTES = 8 << 30     # upper bound of the Gd buffer of the backward edge pass (rows are processed in blocks)


def in_bwd_edges(g: GraphCSR, x, att: "InAttention", d_out, prep, negative_slope, keep_mask=None, p_drop=0.0,
                 n_blocks=None, seed=0, records=False):
    """Gd GEMM + backward edge pass, in blocks of destination rows.  Returns dz [E',H] (source-major) and da_dst.

    ``records=True`` (K = 64): returns alpha_used, dz, da_dst, where alpha_used and dz are the halves of one interleaved
    [E',2H] buffer, the slot records ``gat_bwd_src`` reads (what ``gat_bwd_dst`` returns on the projected path)."""
    L = _abi.lib()
    dev, K = x.device, x.size(1)
    F = in_sizes(g.n_dst, K)[2]
    if records:
        eg = torch.empty(g.n_edges, 16, dtype=torch.float32, device=dev)
        alpha_used, dz = eg[:, :8], eg[:, 8:]
    else:
        alpha_used, dz = None, torch.empty(g.n_edges, 8, dtype=torch.float32, device=dev)
    da_dst = torch.empty(g.n_dst, 8, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_in_bwd_edges_workspace_bytes(g.ref(), C.byref(nb)))
    ws = _ws(nb.value, dev)
    if n_blocks is None:
        n_blocks = max(1, -(-g.n_dst * F * 4 // IN_GD_BLOCK_BYTES))
    blocks = g.item_blocks(n_blocks)
    max_rows = max(hi - lo for _, _, lo, hi in blocks)
    gd = torch.empty(max_rows, F, dtype=torch.float32, device=dev)
    gb = C.c_size_t()
    _abi.check(L.gnnfd_in_bwd_gd_workspace_bytes(max_rows, C.byref(gb)))
    gws = _aligned_u8(gb.value, dev)
    for bi, (i_lo, i_hi, r_lo, r_hi) in enumerate(blocks):
        if r_hi > r_lo:
            _abi.check(L.gnnfd_in_bwd_gd(d_out[r_lo:r_hi].data_ptr(), r_hi - r_lo, K, prep.data_ptr(), gd.data_ptr(),
                                         gws.data_ptr(), gws.numel(), _stream()))
        phase = 1 | (2 if bi == len(blocks) - 1 else 0)
        _abi.check(L.gnnfd_in_bwd_edges(g.ref(), x.data_ptr(), x.stride(0), K, att.alpha.data_ptr(), att.jflag.data_ptr(),
                                        gd.data_ptr(), r_lo, i_lo, i_hi, r_lo, r_hi,
                                        float(negative_slope), _abi.ptr(keep_mask), float(p_drop), int(seed),
                                        _abi.ptr(alpha_used), dz.data_ptr(), da_dst.data_ptr(), ws.data_ptr(), ws.numel(),
                                        phase, _stream()))
    return (alpha_used, dz, da_dst) if records else (dz, da_dst)


def in_dasrc(g: GraphCSR, dz, out=None):
    da_src = out if out is not None else torch.empty(g.n_src, 8, dtype=torch.float32, device=dz.device)
    _abi.check(_abi.lib().gnnfd_in_bwd_dasrc(g.ref(), dz.data_ptr(), da_src.data_ptr(), _stream()))
    return da_src


def in_bwd_params(zimg, d_out, x, W, att_src, att_dst, da_src, da_dst, prep):
    """dW, datt_src, datt_dst, dbias from the saved image and the logit gradients of x's rows."""
    return in_bwd_params_split(zimg, d_out, x, W, att_src, att_dst, prep, _phase=3, _da=(da_src, da_dst))


def in_bwd_params_split(zimg, d_out, x, W, att_src, att_dst, prep, _phase=1, _da=None):
    """The same in two steps: this call enqueues the tensor-core reduction ``dO^T Z`` (which needs no logit gradients) and
    returns ``finish(da_src, da_dst) -> (dW, datt_src, datt_dst, dbias)`` -- across GPUs the first step runs while ``da_src``
    is still being exchanged on another stream."""
    L = _abi.lib()
    n, K = x.shape
    dev = x.device
    dW = torch.empty(512, K, dtype=torch.float32, device=dev)
    datt_src = torch.empty(512, dtype=torch.float32, device=dev)
    datt_dst = torch.empty(512, dtype=torch.float32, device=dev)
    dbias = torch.empty(64, dtype=torch.float32, device=dev)
    nb = C.c_size_t()
    _abi.check(L.gnnfd_in_bwd_params_workspace_bytes(n, K, C.byref(nb)))
    ws = _ws(nb.value, dev) if _phase == 3 else torch.empty(nb.value, dtype=torch.uint8, device=dev)

    def call(phase, da_src, da_dst):
        _abi.check(L.gnnfd_in_bwd_params(zimg.data_ptr(), d_out.data_ptr(), x.data_ptr(), x.stride(0), n, K, W.data_ptr(),
                                         att_src.data_ptr(), att_dst.data_ptr(), _abi.ptr(da_src), _abi.ptr(da_dst),
                                         prep.data_ptr(), dW.data_ptr(), datt_src.data_ptr(), datt_dst.data_ptr(),
                                         dbias.data_ptr(), ws.data_ptr(), ws.numel(), phase, _stream()))

    if _phase == 3:
        call(3, *_da)
        return dW, datt_src, datt_dst, dbias
    call(1, None, None)

    def finish(da_src, da_dst):
        call(2, da_src, da_dst)
        return dW, datt_src, datt_dst, dbias
    return finish


class GATConvInputSpaceFunction(torch.autograd.Function):
    """GATConv (concat=False, H=8, C=64) in the input-space formulation.  The gradient w.r.t. x (a hidden layer, K=64) goes
    through the projected path's source-major pass and dx GEMM: dx = dxw W with dxw from the (alpha_used, dz) records."""

    @staticmethod
    def forward(ctx, x, W, att_src, att_dst, bias, g: GraphCSR, negative_slope, keep_mask, p_drop, want_stats, seed=0):
        _require_f32_cuda("x", x)
        _require_f32_cuda("lin_src.weight", W)
        if x.dim() != 2 or x.size(1) != W.size(1):
            raise ValueError(f"x must be [N,{W.size(1)}], got {tuple(x.shape)}")
        if x.size(0) != g.n_src:
            raise ValueError(f"x has {x.size(0)} rows but the graph has {g.n_src} source nodes")
        W = W.contiguous()
        a_s, a_d = att_src.contiguous().view(-1), att_dst.contiguous().view(-1)
        K = x.size(1)
        with torch.cuda.device(x.device):
            pb = in_sizes(g.n_dst, K)[0]
            x = in_pad_x(x)
            prep = _aligned_u8(pb, x.device)
            xmax = torch.zeros(16, dtype=torch.float32, device=x.device)
            a_src, a_dst = in_logits(x, W, a_s, a_d, prep, xmax)
            in_prepare(W, K, xmax, prep)
            zimg, att = in_fwd(g, x, a_src, a_dst, negative_slope, prep, keep_mask, p_drop, seed)
            out = in_out(zimg, g.n_dst, K, prep, bias)
        rowmax, rowsum = att.rowmax, att.rowsum
        # the backward needs neither logits nor row statistics: alpha / jflag carry everything (see gnnfd_in_fwd)
        ctx.save_for_backward(x, W, a_s, a_d, rowmax, rowsum, att.alpha, att.jflag, keep_mask, zimg, prep)
        ctx.g, ctx.slope, ctx.p, ctx.seed = g, negative_slope, p_drop, seed
        ctx.has_bias = bias is not None
        ctx.att_shape = att_src.shape
        if want_stats:
            ctx.mark_non_differentiable(a_src, a_dst, rowmax, rowsum)
            return out, a_src, a_dst, rowmax, rowsum
        return out

    @staticmethod
    def backward(ctx, d_out, *unused):
        x, W, a_s, a_d, rowmax, rowsum, alpha, jflag, keep_mask, zimg, prep = ctx.saved_tensors
        g = ctx.g
        if not g.has_csc:
            raise RuntimeError("backward needs the CSC twin; build the graph with build_csc=True")
        d_out = d_out.contiguous().float()
        dx = None
        with torch.cuda.device(x.device):
            att = InAttention(alpha, jflag, rowmax, rowsum)
            if ctx.needs_input_grad[0]:
                alpha_used, dz, da_dst = in_bwd_edges(g, x, att, d_out, prep, ctx.slope, keep_mask, ctx.p, seed=ctx.seed,
                                                      records=True)
                dxw, da_src = gat_bwd_src(g, alpha_used, dz, d_out, a_s, a_d, da_dst, 8, 64, False)
                dW, datt_src, datt_dst, dbias = in_bwd_params(zimg, d_out, x, W, a_s, a_d, da_src, da_dst, prep)
                dx = project_dx(dxw, W, 8, 64)
            else:
                dz, da_dst = in_bwd_edges(g, x, att, d_out, prep, ctx.slope, keep_mask, ctx.p, seed=ctx.seed)
                da_src = in_dasrc(g, dz)
                dW, datt_src, datt_dst, dbias = in_bwd_params(zimg, d_out, x, W, a_s, a_d, da_src, da_dst, prep)
        return (dx, dW, datt_src.view(ctx.att_shape), datt_dst.view(ctx.att_shape), dbias if ctx.has_bias else None,
                None, None, None, None, None, None)


class GATConvFunction(torch.autograd.Function):
    """out = GATConv(x, edge_index') with every stage in the CUDA library."""

    @staticmethod
    def forward(ctx, x, W, att_src, att_dst, bias, g: GraphCSR, H, C_, concat, negative_slope, keep_mask, p_drop,
                xw_dtype, algo, want_stats, seed=0):
        _require_f32_cuda("x", x)
        _require_f32_cuda("lin_src.weight", W)
        if x.dim() != 2 or x.size(1) != W.size(1):
            raise ValueError(f"x must be [N,{W.size(1)}], got {tuple(x.shape)}")
        if x.size(0) != g.n_src:
            raise ValueError(f"x has {x.size(0)} rows but the graph has {g.n_src} source nodes")
        if x.stride(1) != 1:
            x = x.contiguous()
        W = W.contiguous()
        a_s, a_d = att_src.contiguous().view(-1), att_dst.contiguous().view(-1)
        with torch.cuda.device(x.device):
            img = None
            if image_projection_applies(x, H, C_, xw_dtype, algo) and not x.requires_grad:
                img = GLOBAL_XIMAGE_CACHE.get(x)        # None the first time this tensor is seen
            if img is not None:
                # first layer (x is data, static across steps): projection from the cached fp16-pair image of x
                xw, a_src, a_dst = project_fwd_image(img, W, a_s, a_d)
            else:
                xw, a_src, a_dst = project_fwd(x, W, a_s, a_d, H, C_, xw_dtype, algo)
            out, rowmax, rowsum = gat_fwd(g, xw, a_src, a_dst, bias, H, C_, negative_slope, concat, _abi.ACT_NONE,
                                          keep_mask, p_drop, seed=seed)
        ctx.save_for_backward(x, W, a_s, a_d, xw, a_src, a_dst, rowmax, rowsum, keep_mask)
        ctx.g, ctx.H, ctx.C, ctx.concat, ctx.slope, ctx.p, ctx.algo = g, H, C_, concat, negative_slope, p_drop, algo
        ctx.seed = seed
        ctx.has_bias = bias is not None
        ctx.att_shape = att_src.shape
        if want_stats:
            ctx.mark_non_differentiable(a_src, a_dst, rowmax, rowsum)
            return out, a_src, a_dst, rowmax, rowsum
        return out

    @staticmethod
    def backward(ctx, d_out, *unused):
        x, W, a_s, a_d, xw, a_src, a_dst, rowmax, rowsum, keep_mask = ctx.saved_tensors
        g, H, C_, concat = ctx.g, ctx.H, ctx.C, ctx.concat
        if not g.has_csc:
            raise RuntimeError("backward needs the CSC twin; build the graph with build_csc=True")
        d_out = d_out.contiguous().float()
        need_dx = ctx.needs_input_grad[0]
        Co = H * C_ if concat else C_
        with torch.cuda.device(x.device):
            dxw, da_src, da_dst = gat_bwd(g, xw, a_src, a_dst, rowmax, rowsum, d_out, a_s, a_d, H, C_, ctx.slope,
                                          concat, keep_mask, ctx.p, seed=ctx.seed)
            dW, datt_src, datt_dst, dbias, dx = project_bwd(x, W, dxw, xw, da_src, da_dst, d_out, H, C_, Co, need_dx,
                                                            ctx.algo)
        return (dx, dW, datt_src.view(ctx.att_shape), datt_dst.view(ctx.att_shape),
                dbias if ctx.has_bias else None, None, None, None, None, None, None, None, None, None, None, None)


def gatconv(x, W, att_src, att_dst, bias, g: GraphCSR, heads, out_channels, concat=False, negative_slope=0.2,
            keep_mask=None, p_drop=0.0, xw_dtype=torch.float32, algo=_abi.GEMM_AUTO, want_stats=False, seed=0):
    """``p_drop > 0`` with ``keep_mask=None`` selects the in-kernel counter-based dropout RNG keyed on ``seed``."""
    if algo == _abi.GEMM_INPUT:
        need_dx = x.requires_grad and torch.is_grad_enabled()
        if ((need_dx and x.size(1) != 64) or xw_dtype != torch.float32 or not in_supported(x.size(1), heads, out_channels, concat)
                or p_drop > 0.9):
            raise _abi.GnnfdError(-5, "input-space formulation: needs concat=False, heads=8, out_channels=64, "
                                      "in_channels <= 192 (exactly 64 when x needs a gradient), fp32 features, dropout <= 0.9")
        return GATConvInputSpaceFunction.apply(x, W, att_src, att_dst, bias, g, negative_slope, keep_mask, p_drop,
                                               want_stats, seed)
    return GATConvFunction.apply(x, W, att_src, att_dst, bias, g, heads, out_channels, concat, negative_slope,
                                 keep_mask, p_drop, xw_dtype, algo, want_stats, seed)
