"""Drop-in for HAC's `arithmetic` CUDA extension (HAC/submodules/arithmetic.zip!arithmetic/arithmetic.cpp:4-49): the same three
functions with the same arguments and results, on libgpcgc.so's attribute-coder kernels (csrc/attr_ac.cu), plus the two fused
entry points the B200 path uses (`gaussian_encode` / `gaussian_decode`: no lower[N][Lp] table), the same for HAC++'s mixture of
K <= 4 Gaussians (`mixture_encode` / `mixture_decode`) and for a table whose rows are all one row (`row_encode` / `row_decode`,
the Bernoulli mask coder).

There is no CPU fallback: tensors must be CUDA tensors and the library must be built.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _check_cuda(*ts):
    for t in ts:
        if not t.is_cuda:
            raise RuntimeError("gauspcc_b200.arithmetic: tensors must be CUDA tensors (there is no CPU path)")
        if not t.is_contiguous():
            raise RuntimeError("gauspcc_b200.arithmetic: tensors must be contiguous")      # CHECK_INPUT, include/utils.h:3-5


def _workspace(n, chunk_size, dev):
    lib = _lib.load()
    return torch.empty(int(lib.gpc_attr_workspace_bytes(n, chunk_size)), dtype=torch.uint8, device=dev)


def calculate_cdf(mean, scale, Q, min_value, max_value):
    """arithmetic.calculate_cdf: lower[N, max - min + 2] float32 (arithmetic_kernel.cu:11-55)."""
    _check_cuda(mean, scale, Q)
    lib = _lib.load()
    mn, mx = int(min_value), int(max_value)
    n = mean.shape[0]
    lower = torch.empty((n, mx - mn + 2), dtype=torch.float32, device=mean.device)
    _lib.check(lib.gpc_attr_calculate_cdf(_ptr(mean), _ptr(scale), _ptr(Q), n, mn, mx, _ptr(lower), _stream(mean.device)), "calculate_cdf")
    return lower


def _finish_encode(ws, n, chunk_size, cnt, offsets, dev):
    lib = _lib.load()
    total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.uint8, device=dev)
    _lib.check(lib.gpc_attr_merge_chunks(_ptr(ws), n, chunk_size, _ptr(offsets), _ptr(out), _stream(dev)), "merge_chunks")
    return out, cnt


def arithmetic_encode(sym, cdf, chunk_size, N, Lp):
    """arithmetic.arithmetic_encode -> (byte stream uint8[total], bytes per chunk int32[chunks]) (arithmetic_kernel.cu:186-232)."""
    _check_cuda(sym, cdf)
    if sym.dim() != 1 or cdf.dim() != 2:
        raise RuntimeError("Expected sym to have 1 dimension and cdf to have 2")
    if sym.dtype != torch.int16 or cdf.dtype != torch.float32:
        raise RuntimeError("sym must be int16 and cdf float32")
    lib = _lib.load()
    dev = sym.device
    chunks = (N + chunk_size - 1) // chunk_size
    cnt = torch.zeros(chunks, dtype=torch.int32, device=dev)
    offsets = torch.zeros(chunks + 1, dtype=torch.int32, device=dev)
    ws = _workspace(N, chunk_size, dev)
    _lib.check(lib.gpc_attr_encode_table(_ptr(sym), _ptr(cdf), N, Lp, chunk_size, _ptr(cnt), _ptr(offsets), _ptr(ws), ws.numel(),
                                         _stream(dev)), "arithmetic_encode")
    return _finish_encode(ws, N, chunk_size, cnt, offsets, dev)


def arithmetic_decode(cdf, in_cache_all, in_cnt_all, chunk_size, N, Lp):
    """arithmetic.arithmetic_decode -> int16[N] (arithmetic_kernel.cu:365-407)."""
    _check_cuda(cdf, in_cache_all, in_cnt_all)
    lib = _lib.load()
    dev = cdf.device
    sym = torch.zeros(N, dtype=torch.int16, device=dev)
    ws = _workspace(N, chunk_size, dev)
    _lib.check(lib.gpc_attr_decode_table(_ptr(cdf), _ptr(in_cache_all), _ptr(in_cnt_all.to(torch.int32)), N, Lp, chunk_size, _ptr(sym),
                                         _ptr(ws), ws.numel(), _stream(dev)), "arithmetic_decode")
    return sym


def gaussian_encode(sym, mean, scale, Q, min_value, max_value, chunk_size):
    """calculate_cdf + arithmetic_encode in one pass over the symbols: the same bytes, no table."""
    _check_cuda(sym, mean, scale, Q)
    lib = _lib.load()
    dev = sym.device
    n = sym.shape[0]
    chunks = (n + chunk_size - 1) // chunk_size
    cnt = torch.zeros(chunks, dtype=torch.int32, device=dev)
    offsets = torch.zeros(chunks + 1, dtype=torch.int32, device=dev)
    ws = _workspace(n, chunk_size, dev)
    _lib.check(lib.gpc_attr_encode_gaussian(_ptr(sym), _ptr(mean), _ptr(scale), _ptr(Q), n, int(min_value), int(max_value), chunk_size,
                                            _ptr(cnt), _ptr(offsets), _ptr(ws), ws.numel(), _stream(dev)), "gaussian_encode")
    return _finish_encode(ws, n, chunk_size, cnt, offsets, dev)


def gaussian_decode(mean, scale, Q, in_cache_all, in_cnt_all, min_value, max_value, chunk_size):
    """calculate_cdf + arithmetic_decode without the table -> int16[N]."""
    _check_cuda(mean, scale, Q, in_cache_all, in_cnt_all)
    lib = _lib.load()
    dev = mean.device
    n = mean.shape[0]
    sym = torch.zeros(n, dtype=torch.int16, device=dev)
    ws = _workspace(n, chunk_size, dev)
    _lib.check(lib.gpc_attr_decode_gaussian(_ptr(mean), _ptr(scale), _ptr(Q), _ptr(in_cache_all), _ptr(in_cnt_all.to(torch.int32)), n,
                                            int(min_value), int(max_value), chunk_size, _ptr(sym), _ptr(ws), ws.numel(), _stream(dev)),
               "gaussian_decode")
    return sym


def _check_mixture(mean, scale, prob, Q, n):
    if mean.dim() != 2 or mean.shape[1] != n or scale.shape != mean.shape or prob.shape != mean.shape or Q.shape != (n,):
        raise RuntimeError(f"mixture coder: mean / scale / prob must be [K, {n}] and Q [{n}]")
    if any(t.dtype != torch.float32 for t in (mean, scale, prob, Q)):
        raise RuntimeError("mixture coder: mean / scale / prob / Q must be float32")


def mixture_encode(sym, mean, scale, prob, Q, min_value, max_value, chunk_size):
    """The table of a K-component mixture (clamp(sum_k calculate_cdf(mean[k], scale[k]) * prob[k], 0, 1), as
    encodings_cuda.encoder_gaussian_mixed builds it) + arithmetic_encode, without the table.  mean / scale / prob: [K, n]
    float32, 1 <= K <= 4."""
    _check_cuda(sym, mean, scale, prob, Q)
    n = sym.shape[0]
    _check_mixture(mean, scale, prob, Q, n)
    lib = _lib.load()
    dev = sym.device
    chunks = (n + chunk_size - 1) // chunk_size
    cnt = torch.zeros(chunks, dtype=torch.int32, device=dev)
    offsets = torch.zeros(chunks + 1, dtype=torch.int32, device=dev)
    ws = _workspace(n, chunk_size, dev)
    _lib.check(lib.gpc_mixture_encode(_ptr(sym), _ptr(mean), _ptr(scale), _ptr(prob), _ptr(Q), n, mean.shape[0], int(min_value),
                                      int(max_value), chunk_size, _ptr(cnt), _ptr(offsets), _ptr(ws), ws.numel(), _stream(dev)),
               "mixture_encode")
    return _finish_encode(ws, n, chunk_size, cnt, offsets, dev)


def mixture_decode(mean, scale, prob, Q, in_cache_all, in_cnt_all, min_value, max_value, chunk_size):
    """The mixture's table + arithmetic_decode, without the table -> int16[n]."""
    _check_cuda(mean, scale, prob, Q, in_cache_all, in_cnt_all)
    n = mean.shape[-1]
    _check_mixture(mean, scale, prob, Q, n)
    lib = _lib.load()
    dev = mean.device
    sym = torch.zeros(n, dtype=torch.int16, device=dev)
    ws = _workspace(n, chunk_size, dev)
    _lib.check(lib.gpc_mixture_decode(_ptr(mean), _ptr(scale), _ptr(prob), _ptr(Q), _ptr(in_cache_all), _ptr(in_cnt_all.to(torch.int32)),
                                      n, mean.shape[0], int(min_value), int(max_value), chunk_size, _ptr(sym), _ptr(ws), ws.numel(),
                                      _stream(dev)), "mixture_decode")
    return sym


def _check_row(row):
    if row.dim() != 1 or row.dtype != torch.float32:
        raise RuntimeError("row coder: the row must be 1-D float32")


def row_encode(sym, row, chunk_size):
    """arithmetic_encode of a table whose rows are all `row` (float32[Lp]), without the table."""
    _check_cuda(sym, row)
    _check_row(row)
    lib = _lib.load()
    dev = sym.device
    n = sym.shape[0]
    chunks = (n + chunk_size - 1) // chunk_size
    cnt = torch.zeros(chunks, dtype=torch.int32, device=dev)
    offsets = torch.zeros(chunks + 1, dtype=torch.int32, device=dev)
    ws = _workspace(n, chunk_size, dev)
    _lib.check(lib.gpc_row_encode(_ptr(sym), _ptr(row), n, row.shape[0], chunk_size, _ptr(cnt), _ptr(offsets), _ptr(ws), ws.numel(),
                                  _stream(dev)), "row_encode")
    return _finish_encode(ws, n, chunk_size, cnt, offsets, dev)


def row_decode(row, in_cache_all, in_cnt_all, N, chunk_size):
    """arithmetic_decode of N symbols under one shared row -> int16[N]."""
    _check_cuda(row, in_cache_all, in_cnt_all)
    _check_row(row)
    lib = _lib.load()
    dev = row.device
    sym = torch.zeros(N, dtype=torch.int16, device=dev)
    ws = _workspace(N, chunk_size, dev)
    _lib.check(lib.gpc_row_decode(_ptr(row), _ptr(in_cache_all), _ptr(in_cnt_all.to(torch.int32)), N, row.shape[0], chunk_size, _ptr(sym),
                                  _ptr(ws), ws.numel(), _stream(dev)), "row_decode")
    return sym
