"""Drop-in replacement for the reference's `utils/pcc_utils.py` (the L3 boundary).

Same three entry points, argument meaning, return dicts and `xyz_pcc.bin` layout as
/root/reference/src/gs_compress/HAC/utils/pcc_utils.py:
    calculate_morton_order(x)                                             :12-22
    compress_point_cloud(xyz_quantized, ckpt_path, output_path, ...)      :24-217
    decompress_point_cloud(bin_file_path, ckpt_path, output_path=None...) :230-400
so HAC / HAC++ / CAT-3DGS / TC-GS `scene/gaussian_model.py` can switch with
`from gauspcc_b200.pcc_utils import ...` (see INTEGRATION.md).  Underneath: libgpcgc.so (hand-written
sm_100a kernels behind the C ABI of include/gpcgc.h).  No torchsparse, no torchac, no Triton, no CPU
fallback -- without CUDA or without the built library these functions raise.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from typing import Dict, List

import numpy as np
import torch

from . import _lib, bitstream, plyio
from .batch import BatchCodec
from .codec import GausPcgcCodec, load_weights

_CODECS: Dict[tuple, GausPcgcCodec] = {}
_BATCH: Dict[int, BatchCodec] = {}


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.GpcError("gauspcc_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _codec(ckpt_path: str, channels: int, kernel_size: int) -> GausPcgcCodec:
    dev = _require_cuda()
    w = load_weights(ckpt_path, dev, channels, kernel_size)
    key = (id(w), str(dev))
    if key not in _CODECS:
        _CODECS[key] = GausPcgcCodec(w, dev)
    return _CODECS[key]


def _batch(codec: GausPcgcCodec) -> BatchCodec:
    """the batch driver over a codec: it follows the codec's kernel-family attributes, so both paths take the same decisions"""
    if id(codec) not in _BATCH:
        _BATCH[id(codec)] = BatchCodec(codec)
    return _BATCH[id(codec)]


def _check_chunk(gpu_coder_chunk) -> None:
    if gpu_coder_chunk and not (32 <= int(gpu_coder_chunk) <= 16384):
        raise ValueError("gpu_coder_chunk must be in 32..16384 (chunk byte counts are stored as u16)")


def _to_device_xyz(xyz_quantized, dev):
    xyz = torch.tensor(xyz_quantized) if isinstance(xyz_quantized, np.ndarray) else xyz_quantized.detach()
    if xyz.is_floating_point():
        return xyz.to(device=dev, dtype=torch.float32)
    return xyz.to(device=dev, dtype=torch.int32)


def calculate_morton_order(x: torch.Tensor) -> torch.Tensor:
    """
    Calculate Morton order of the input points.

    Same contract as the reference (pcc_utils.py:12-22): returns the int64 permutation, on `x.device`,
    that sorts the rows by x + y*M + z*M^2 after subtracting the per-axis minimum, i.e. ascending
    (z, y, x).  Ties (duplicate voxels) keep their input order (the reference leaves them unspecified).
    The sort runs on the GPU (key pack + LSD radix sort in libgpcgc); a CPU tensor is moved to the
    current CUDA device and the result moved back.
    """
    assert len(x.shape) == 2 and x.shape[1] == 3, f'Input data must be a 3D point cloud, but got {x.shape}.'
    lib = _lib.load()
    dev = _require_cuda()
    src_device = x.device
    xd = x.detach()
    if xd.is_floating_point():
        xd = xd.to(device=dev, dtype=torch.float32)
        is_f32 = 1
    else:
        xd = xd.to(device=dev, dtype=torch.int32)
        is_f32 = 0
    xd = xd.contiguous()
    n = xd.shape[0]
    out = torch.empty(n, dtype=torch.int64, device=dev)
    if n:
        ws_b = lib.gpc_lexorder_workspace_bytes(n)
        ws = torch.empty(ws_b, dtype=torch.uint8, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.gpc_lexorder_zyx(C.c_void_p(xd.data_ptr()), is_f32, n, C.c_void_p(out.data_ptr()),
                                        C.c_void_p(ws.data_ptr()), ws_b, stream), "gpc_lexorder_zyx")
    return out.to(src_device)


def compress_point_cloud(
    xyz_quantized,            # Quantized point cloud coordinates, numpy array or torch tensor
    ckpt_path,                # Path to pre-trained weights file
    output_path,              # Output bin file path
    channels=32,              # Network channel count
    kernel_size=5,            # Convolution kernel size
    posQ=1,                   # Quantization scale
    gpu_coder_chunk=0         # extension (not in the reference): > 0 writes container version 2, see below
):
    """
    Compress point cloud into a bin file (reference: pcc_utils.py:24-217).

    Returns {'bpp', 'enc_time', 'file_size_bits', 'num_points', 'output_path'}; `enc_time` is wall-clock
    between device synchronisations, including the host range coder and excluding the checkpoint load
    and the file write, as in the reference (:78-79,188-189).  Extra key 'gpu_time': CUDA-event time
    of the device segments only.

    gpu_coder_chunk > 0 (e.g. 2048): the occupancy streams are coded on the GPU in chunks of that many symbols and the file is
    container version 2 (bitstream.py) -- smaller PCIe traffic and no host range coder on either side, but NOT readable by the
    reference's decompress_point_cloud.  The default (0) writes the reference's own bitstream.
    """
    _check_chunk(gpu_coder_chunk)
    os.makedirs(os.path.dirname(output_path), exist_ok=True)
    codec = _codec(ckpt_path, channels, kernel_size)
    dev = codec.dev
    if isinstance(xyz_quantized, np.ndarray):
        xyz = torch.tensor(xyz_quantized)
    else:
        xyz = xyz_quantized.detach()          # never mutated (the reference clones, :61)
    N = xyz.shape[0]
    if xyz.is_floating_point():
        xyz = xyz.to(device=dev, dtype=torch.float32)
    else:
        xyz = xyz.to(device=dev, dtype=torch.int32)    # the reference casts with .int() (:73)

    torch.cuda.synchronize(dev)
    enc_time_start = time.time()
    base_xyz, base_occ, streams, _ = codec.encode(xyz, gpu_chunk=int(gpu_coder_chunk))
    torch.cuda.synchronize(dev)
    enc_time_end = time.time()
    if gpu_coder_chunk:
        streams = streams + [bitstream.v2_trailer(int(gpu_coder_chunk), int(codec.last_stats.get("n_unique", N)))]

    blob = bitstream.write_file(posQ, base_xyz, base_occ, streams)
    with open(output_path, 'wb') as f:
        f.write(blob)

    enc_time = enc_time_end - enc_time_start
    file_size_bits = os.stat(output_path).st_size * 8
    bpp = file_size_bits / N
    return {
        'bpp': bpp,
        'enc_time': enc_time,
        'file_size_bits': file_size_bits,
        'num_points': N,
        'output_path': output_path,
        'gpu_time': codec.last_stats.get("gpu_ms", 0.0) / 1e3,
    }


def decompress_point_cloud(
    bin_file_path,           # Path to compressed bin file
    ckpt_path,               # Path to pre-trained weights file
    output_path=None,        # Path for output ply file (optional)
    channels=32,             # Network channel count
    kernel_size=5,           # Convolution kernel size
    is_data_pre_quantized=True,  # Whether original point cloud is pre-quantized
    sorted_output=False      # extension (not in the reference): rows in calculate_morton_order order
):
    """
    Decompress point cloud from bin file (reference: pcc_utils.py:230-400).

    Returns {'dec_time', 'num_points', 'point_cloud': float32 [N,3] on the GPU, 'output_path'}.  Row
    order is the reference's: children of the (z,y,x)-sorted last level, octant ascending (:375).
    With sorted_output=True the rows come back in ascending (z,y,x) instead, which is the order
    calculate_morton_order produces: the re-sort HAC does right after this call
    (HAC/scene/gaussian_model.py:1253-1255) is then the identity permutation and can be dropped.
    """
    if output_path:
        os.makedirs(os.path.dirname(output_path), exist_ok=True)
    codec = _codec(ckpt_path, channels, kernel_size)
    dev = codec.dev
    with open(bin_file_path, 'rb') as f:
        blob = f.read()
    posQ, base_xyz, base_occ, streams = bitstream.read_file(blob)
    streams, gpu_chunk, n_coded = bitstream.split_v2(streams)    # container version 2 names itself in a trailing stream

    torch.cuda.synchronize(dev)
    dec_time_start = time.time()
    scan = codec.decode(base_xyz, base_occ, streams, scale=float(posQ), sorted_rows=bool(sorted_output), gpu_chunk=gpu_chunk)
    if n_coded is not None and scan.shape[0] != n_coded:
        raise ValueError(f"version-2 file decodes to {scan.shape[0]} voxels, its trailer says {n_coded}: corrupt file, wrong checkpoint "
                         "or a library whose kernels sum in another order than the writer's")
    if not is_data_pre_quantized:
        scan = (scan - 131072) * 0.001                 # pcc_utils.py:381
    torch.cuda.synchronize(dev)
    dec_time_end = time.time()
    dec_time = dec_time_end - dec_time_start

    point_cloud = scan
    if output_path:
        # the reference calls io.save_ply_ascii_geo here but never imports `io` (pcc_utils.py:392 would raise
        # NameError); write the same ASCII geometry PLY (kit/io.py:36-49) instead of failing, rows formatted on the GPU.
        plyio.write_ply_ascii(point_cloud, output_path)
    return {
        'dec_time': dec_time,
        'num_points': point_cloud.shape[0],
        'point_cloud': point_cloud,
        'output_path': output_path,
        'gpu_time': codec.last_stats.get("gpu_ms", 0.0) / 1e3,
    }


def compress_point_clouds(xyz_list, ckpt_path, output_paths, channels=32, kernel_size=5, posQ=1, gpu_coder_chunk=0) -> List[dict]:
    """
    Compress many point clouds in one call (extension, not in the reference): file i is byte-identical to
    compress_point_cloud(xyz_list[i], ckpt_path, output_paths[i], channels, kernel_size, posQ, gpu_coder_chunk).

    The scenes are coded together as one union octree (gauspcc_b200/batch.py): one set of launches per level and the range coders
    of all scenes side by side on the codec's thread pool, instead of one level loop per scene.  With gpu_coder_chunk > 0 the files
    are container version 2, as compress_point_cloud writes them: every chunk of every scene's streams is coded on the GPU by one
    launch per union, and no host range coder runs.  Returns one dict per scene with the single call's keys; 'enc_time' and
    'gpu_time' are 0.0 there (the scenes are coded together, there is no per-scene time) and 'batch_enc_time' is the wall-clock time
    of the whole batch, the same value in every dict.
    """
    _check_chunk(gpu_coder_chunk)
    xyz_list, output_paths = list(xyz_list), list(output_paths)
    if len(xyz_list) != len(output_paths):
        raise ValueError(f"compress_point_clouds: {len(xyz_list)} point clouds but {len(output_paths)} output paths")
    if not xyz_list:
        return []
    codec = _codec(ckpt_path, channels, kernel_size)
    dev = codec.dev
    xyzs = [_to_device_xyz(x, dev) for x in xyz_list]
    for p in output_paths:
        os.makedirs(os.path.dirname(p), exist_ok=True)
    torch.cuda.synchronize(dev)
    t0 = time.time()
    coded = _batch(codec).encode(xyzs, gpu_chunk=int(gpu_coder_chunk))
    torch.cuda.synchronize(dev)
    batch_enc_time = time.time() - t0
    out = []
    for xyz, p, (base_xyz, base_occ, streams) in zip(xyzs, output_paths, coded):
        with open(p, 'wb') as f:
            f.write(bitstream.write_file(posQ, base_xyz, base_occ, streams))
        N = xyz.shape[0]
        bits = os.stat(p).st_size * 8
        out.append({'bpp': bits / N, 'enc_time': 0.0, 'file_size_bits': bits, 'num_points': N, 'output_path': p, 'gpu_time': 0.0,
                    'batch_enc_time': batch_enc_time})
    return out


def decompress_point_clouds(bin_paths, ckpt_path, channels=32, kernel_size=5, is_data_pre_quantized=True,
                            sorted_output=False, output_paths=None) -> List[dict]:
    """
    Decompress many files in one call (extension): result i's 'point_cloud' equals
    decompress_point_cloud(bin_paths[i], ckpt_path, ...)['point_cloud'] row for row, in both row orders.  The files of one call are
    all container version 1 or all version 2 (their chunk sizes may differ); a call that mixes the two raises ValueError naming the
    first file whose version differs from the first file's.  Version-2 files are decoded on the GPU chunk by chunk, every stage of a
    union level by one launch, and each decoded count is checked against the file's trailer (ValueError naming the file, as
    decompress_point_cloud raises).  'dec_time' and 'gpu_time' are 0.0; 'batch_dec_time' is the wall-clock time of the whole batch,
    the same value in every dict.  With output_paths (one per file), scene i is also written to output_paths[i] as the ASCII PLY
    decompress_point_cloud(bin_paths[i], ..., output_path=output_paths[i]) writes, byte for byte, after the timed batch; that path
    is then result i's 'output_path'.
    """
    bin_paths = list(bin_paths)
    if output_paths is not None:
        output_paths = list(output_paths)
        if len(output_paths) != len(bin_paths):
            raise ValueError(f"decompress_point_clouds: {len(bin_paths)} files but {len(output_paths)} output paths")
        for p in output_paths:
            if p:
                os.makedirs(os.path.dirname(p), exist_ok=True)
    if not bin_paths:
        return []
    codec = _codec(ckpt_path, channels, kernel_size)
    dev = codec.dev
    files, coded = [], []
    for p in bin_paths:
        with open(p, 'rb') as f:
            blob = f.read()
        try:
            posQ, base_xyz, base_occ, streams = bitstream.read_file(blob)
        except ValueError as e:
            raise ValueError(f"{p}: {e}") from e
        streams, chunk, n_coded = bitstream.split_v2(streams)
        if files and bool(chunk) != bool(files[0][4]):
            # one container version per call keeps every union level on one decode discipline
            raise ValueError(f"{p}: container version {2 if chunk else 1} file after version {2 if files[0][4] else 1} files; "
                             "version 1 and version 2 files cannot be decoded in one call")
        files.append((float(posQ), base_xyz, base_occ, streams, chunk))
        coded.append(n_coded)
    torch.cuda.synchronize(dev)
    t0 = time.time()
    scans = _batch(codec).decode(files, sorted_rows=bool(sorted_output), names=bin_paths)
    for p, s, n_coded in zip(bin_paths, scans, coded):
        if n_coded is not None and s.shape[0] != n_coded:
            raise ValueError(f"{p}: version-2 file decodes to {s.shape[0]} voxels, its trailer says {n_coded}: corrupt file, wrong "
                             "checkpoint or a library whose kernels sum in another order than the writer's")
    if not is_data_pre_quantized:
        scans = [(s - 131072) * 0.001 for s in scans]             # pcc_utils.py:381
    torch.cuda.synchronize(dev)
    batch_dec_time = time.time() - t0
    outs = output_paths if output_paths is not None else [None] * len(scans)
    for s, p in zip(scans, outs):
        if p:
            plyio.write_ply_ascii(s, p)
    return [{'dec_time': 0.0, 'num_points': s.shape[0], 'point_cloud': s, 'output_path': p, 'gpu_time': 0.0,
             'batch_dec_time': batch_dec_time} for s, p in zip(scans, outs)]
