"""ASCII PLY / point-text I/O on the GPU (libgpcgc's textio.cu), with the same bytes and rows as the Python it replaces.

- `write_ply_ascii(points, path)`: the geometry PLY `decompress_point_cloud(..., output_path)` writes (kit/io.py:36-49): a header and
  one `f"{x} {y} {z}\\n"` row per point, x, y, z float32 printed as Python prints them.  The rows are formatted on the GPU and come
  back in one copy into pinned memory.
- `read_points_device(path, device)`: `torch.from_numpy(cli.read_points(path))` on the GPU.  Text files are parsed there; the few
  lines the GPU cannot decide alone (non-ASCII or control bytes, `nan` / `inf` / `1_000` tokens, mantissas too long to round from
  a 128-bit product) come back as byte spans and go through `xyz_of_line`, the rule `cli.read_points` applies to every line.
"""
from __future__ import annotations

import ctypes as C
import io
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

# the encoding open(path, "r") reads text with: host-decided lines are decoded as cli.read_points decodes the whole file
_TEXT_ENCODING = io.TextIOWrapper(io.BytesIO(), errors="ignore").encoding
MAX_TEXT_BYTES = (1 << 32) - 1            # u32 byte offsets in the parser
_MAX_ROW_BYTES = 75                      # three values of at most 24 characters, two spaces, "\n"
_PINNED: List[torch.Tensor] = []         # one pinned staging buffer, grown on demand


def xyz_of_line(line: str) -> Optional[List[float]]:
    """The per-line rule of cli.read_points: the first three whitespace-separated tokens as floats; None when the line has fewer
    than three tokens or one of them is not a float (extra columns are ignored)."""
    parts = line.split()
    if len(parts) < 3:
        return None
    try:
        return [float(parts[0]), float(parts[1]), float(parts[2])]
    except ValueError:
        return None


def ply_header(n: int) -> bytes:
    return (f"ply\nformat ascii 1.0\nelement vertex {n}\n"
            "property float x\nproperty float y\nproperty float z\nend_header\n").encode()


def _device(device) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.GpcError("gauspcc_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise ValueError(f"{dev}: the PLY text kernels run on a CUDA device")
    return torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())


def _staging(nbytes: int) -> torch.Tensor:
    if not _PINNED or _PINNED[0].numel() < nbytes:
        _PINNED[:] = [torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, pin_memory=True)]
    return _PINNED[0][:nbytes]


def format_rows(points: torch.Tensor) -> torch.Tensor:
    """The "x y z\\n" rows of float32 [N, 3] CUDA points as a CUDA uint8 tensor of text (no header)."""
    lib = _lib.load()
    if points.dim() != 2 or points.shape[1] != 3:
        raise ValueError(f"points must be [N, 3], got {tuple(points.shape)}")
    dev = points.device if points.is_cuda else _device(None)
    pts = points.detach().to(device=dev, dtype=torch.float32).contiguous()
    n = pts.shape[0]
    out = torch.empty(max(n * _MAX_ROW_BYTES, 1), dtype=torch.uint8, device=dev)
    ws_b = lib.gpc_ply_format_workspace_bytes(n)
    ws = torch.empty(max(ws_b, 1), dtype=torch.uint8, device=dev)
    length = C.c_uint64(0)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(lib.gpc_ply_format_f32(C.c_void_p(pts.data_ptr()), n, C.c_void_p(out.data_ptr()), out.numel(), C.byref(length),
                                      C.c_void_p(ws.data_ptr()), ws_b, stream), "gpc_ply_format_f32")
    return out[:length.value]


def write_ply_ascii(points: torch.Tensor, path: str) -> None:
    """Write float32 [N, 3] CUDA points as the ASCII geometry PLY, byte for byte what the row-by-row Python writer
    (`f.write(f'{p[0]} {p[1]} {p[2]}\\n')` over float32 rows) writes."""
    text = format_rows(points)
    host = _staging(text.numel())
    host.copy_(text)
    with open(path, "wb") as f:
        f.write(ply_header(int(points.shape[0])))
        f.write(memoryview(host.numpy()))


def host_rows(text: bytes, spans: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """The lines the GPU left to the host: spans[k] = (first byte, end of content, GPU rows before the line).  Returns the rows
    those lines give under xyz_of_line (float64 [k, 3]) and, for each, the number of GPU rows that precede it."""
    before, rows = [], []
    for b, e, r in np.asarray(spans, dtype=np.int64).reshape(-1, 3):
        xyz = xyz_of_line(text[b:e].decode(_TEXT_ENCODING, errors="ignore"))
        if xyz is not None:
            before.append(r)
            rows.append(xyz)
    return np.asarray(before, dtype=np.int64), np.asarray(rows, dtype=np.float64).reshape(-1, 3)


def splice_rows(rows: torch.Tensor, before: Sequence[int], extra: torch.Tensor) -> torch.Tensor:
    """rows [n, 3] with extra[j] inserted before rows[before[j]] (before non-decreasing): the rows in line order."""
    k = len(before)
    if k == 0:
        return rows
    n = rows.shape[0]
    pos = torch.as_tensor(np.asarray(before, dtype=np.int64) + np.arange(k), device=rows.device)
    keep = torch.ones(n + k, dtype=torch.bool, device=rows.device)
    keep[pos] = False
    out = torch.empty((n + k, 3), dtype=rows.dtype, device=rows.device)
    out[keep] = rows
    out[pos] = extra.to(device=rows.device, dtype=rows.dtype)
    return out


def parse_text(data: np.ndarray, device=None) -> torch.Tensor:
    """float64 [N, 3] CUDA rows of point text (uint8 array of the file's bytes), as cli.read_points reads a text file."""
    dev = _device(device)
    nbytes = int(data.size)
    if nbytes > MAX_TEXT_BYTES:
        raise ValueError(f"{nbytes} bytes of text: the GPU parser takes files of fewer than 2^32 bytes")
    if nbytes == 0:
        return torch.empty((0, 3), dtype=torch.float64, device=dev)
    lib = _lib.load()
    text = torch.from_numpy(data).to(dev)
    rows = torch.empty((max((nbytes + 1) // 6, 1), 3), dtype=torch.float64, device=dev)
    spans = torch.empty(max((nbytes + 1) // 2, 1) * 3, dtype=torch.int32, device=dev)
    ws_b = lib.gpc_text_parse_workspace_bytes(nbytes)
    ws = torch.empty(max(ws_b, 1), dtype=torch.uint8, device=dev)
    n_rows, n_host = C.c_uint32(0), C.c_uint32(0)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(lib.gpc_text_parse_xyz(C.c_void_p(text.data_ptr()), nbytes, C.c_void_p(rows.data_ptr()), C.byref(n_rows),
                                      C.c_void_p(spans.data_ptr()), C.byref(n_host), C.c_void_p(ws.data_ptr()), ws_b, stream),
               "gpc_text_parse_xyz")
    got = rows[:n_rows.value].clone()          # not a view of the worst-case allocation
    if n_host.value:
        sp = spans[:3 * n_host.value].cpu().numpy().view(np.uint32)
        before, extra = host_rows(data.tobytes(), sp)
        got = splice_rows(got, before, torch.from_numpy(extra))
    return got


def read_points_device(path: str, device=None) -> torch.Tensor:
    """float64 [N, 3] CUDA tensor equal to torch.from_numpy(cli.read_points(path)): `.bin` and `.npy` through cli.read_points'
    numpy readers, anything else as text, parsed on the GPU."""
    dev = _device(device)
    ext = os.path.splitext(path)[-1].lower()
    if ext in (".bin", ".npy"):
        from . import cli
        return torch.from_numpy(np.ascontiguousarray(cli.read_points(path))).to(dev)
    if os.path.getsize(path) > MAX_TEXT_BYTES:
        raise ValueError(f"{path}: {os.path.getsize(path)} bytes of text: the GPU parser takes files of fewer than 2^32 bytes")
    return parse_text(np.fromfile(path, dtype=np.uint8), dev)
