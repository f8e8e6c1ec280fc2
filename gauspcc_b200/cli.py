"""Stand-alone file-level tools over the same codec (SURVEY.md 8f-2): the B200 counterparts of the reference's
`src/ai_pcc/GausPcgc/compress_ue_4stage_conv.py` and `decompress_ue_4stage_conv.py`.

    python -m gauspcc_b200.cli compress   --input_glob DIR --output_folder OUT --ckpt CKPT [--posQ 16] [--is_data_pre_quantized]
    python -m gauspcc_b200.cli decompress --input_glob OUT --output_folder DEC --ckpt CKPT [--is_data_pre_quantized]
    python -m gauspcc_b200.cli train      --input_glob DIR --ckpt_out CKPT [--init CKPT] [--steps N] [--lr 5e-4] [--seed S]
                                          [--kernel_size 3|5] [--posQ 16] [--is_data_pre_quantized] [--max_points 150000]
                                          [--batch_size 1] [--conv_families v6|codec] [--resultdir R]

Same argument names, file discovery (recursive, sorted, h5 / ply / bin / npy; compress_ue_4stage_conv.py:57-63), coordinate
mapping (`x / 0.001 + 131072` unless pre-quantised, then `round(x / posQ)`, :90-95; inverse `(c * posQ - 131072) * 0.001`,
decompress_ue_4stage_conv.py:176-179), `.bin` container (one `<name>.bin` per input) and CSV report (`<prefix>_data<N>.csv` with a
final `avg` row, :253-276) as the reference scripts.  `--kernel_size` defaults to 3 as in the reference scripts
(compress_ue_4stage_conv.py:44; the HAC call sites use 5, pcc_utils.py:29): both are built, channels = 32 only.  Differences: point files are read in this process (the reference forks 64 workers); `h5` is not
read (the reference lists the suffix but `kit/io.py:read_points` cannot parse it either).  No torchsparse / torchac.

Text inputs (ASCII ply and other text) are parsed on the GPU (plyio.read_points_device: the rows `read_points` gives) and mapped
to voxels there with the same float64 operations as `quantise`; decoded clouds are written as ASCII ply rows formatted on the GPU
(plyio.write_ply_ascii: the bytes of the reference's writer).

`train` (not in the reference scripts, whose trainer runs on torchsparse): reads and quantises files exactly as `compress` does, cuts
them into kd-tree patches of at most --max_points points and trains a checkpoint on the GPU (gauspcc_b200/train.py), written in the
reference layout to --ckpt_out; `compress` / `decompress` load it with the same --kernel_size.  `--batch_size B` (default 1) codes B
patches per step as one union octree and takes one Adam step on their bits per point.  `--conv_families codec` runs every level
on the conv family the codec codes it with (the sparse or tcgen05 conv on levels of 150 K rows and more) instead of the mma.sync
conv everywhere (`v6`, the default).  The CSV log (`<prefix>_train_data<N>.csv`:
step, points of the step's patches, bpp, elapsed seconds) goes to --resultdir beside the other reports.

`--batch N` (default 1): with N > 1, consecutive groups of N files are coded in one call each (pcc_utils.compress_point_clouds /
decompress_point_clouds: one union octree per group, the same `.bin` and `.ply` bytes as one file at a time).  A group has no
per-file time, so each of its CSV rows reports `enc_time` / `dec_time` = the group's wall-clock coding time (`batch_enc_time` /
`batch_dec_time`) divided by its number of files.  With N = 1 every file is coded by its own call and timed alone, as before.
"""
from __future__ import annotations

import argparse
import csv
import os
import sys
import time
from glob import glob
from typing import Dict, List, Optional

import numpy as np
import torch

from . import pcc_utils, plyio

SUFFIXES = (".h5", ".ply", ".bin", ".npy")


def read_points(path: str) -> np.ndarray:
    """[N,3] float64 coordinates of one file (reference: kit/io.py:14-31): KITTI `.bin` = float32 x,y,z,i records; `.npy` = array
    whose first three columns are x,y,z; anything else = text with one point per line (ASCII ply: header lines do not parse as
    floats and are skipped, extra columns are ignored)."""
    ext = os.path.splitext(path)[-1].lower()
    if ext == ".bin":
        return np.fromfile(path, dtype=np.float32).reshape(-1, 4)[:, :3].astype(np.float64)
    if ext == ".npy":
        a = np.asarray(np.load(path), dtype=np.float64)
        return a.reshape(-1, a.shape[-1])[:, :3]
    rows: List[List[float]] = []
    with open(path, "r", errors="ignore") as f:
        for line in f:
            xyz = plyio.xyz_of_line(line)
            if xyz is not None:
                rows.append(xyz)
    return np.asarray(rows, dtype=np.float64).reshape(-1, 3)


def list_inputs(input_glob: str, num_samples: int = -1, suffixes=SUFFIXES) -> List[str]:
    paths = sorted(glob(os.path.join(input_glob, "**", "*.*"), recursive=True))
    paths = [p for p in paths if p.lower().endswith(suffixes)]
    return paths[:num_samples] if num_samples and num_samples > 0 else paths


def quantise(xyz: np.ndarray, posQ: int, is_data_pre_quantized: bool) -> torch.Tensor:
    """compress_ue_4stage_conv.py:90-95: (pre-quantised ? x : x / 0.001 + 131072), then round-half-even(x / posQ) as int32."""
    t = torch.tensor(xyz if is_data_pre_quantized else xyz / 0.001 + 131072)
    return torch.round(t / posQ).int()


def quantise_device(xyz: torch.Tensor, posQ: int, is_data_pre_quantized: bool) -> torch.Tensor:
    """`quantise` on a float64 CUDA tensor, with the same float64 operations: the divisors are device tensors, so the division is
    an IEEE division (not a multiplication by the rounded reciprocal, which a host scalar divisor would give)."""
    xyz = xyz.to(torch.float64)
    t = xyz if is_data_pre_quantized else xyz / torch.tensor(0.001, dtype=torch.float64, device=xyz.device) + 131072
    return torch.round(t / torch.tensor(float(posQ), dtype=torch.float64, device=xyz.device)).int()


def _groups(items: List[str], batch: int) -> List[List[str]]:
    if batch < 1:
        raise ValueError(f"batch must be >= 1, got {batch}")
    return [items[i:i + batch] for i in range(0, len(items), batch)]


def _write_csv(path: str, rows: List[Dict[str, object]], numeric: List[str]) -> None:
    avg: Dict[str, object] = {k: float(np.mean([float(r[k]) for r in rows])) for k in numeric}
    avg["filedir"] = "avg"
    with open(path, "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=list(rows[0].keys()))
        w.writeheader()
        for r in rows + [avg]:
            w.writerow(r)


def compress_files(input_glob: str, output_folder: str, ckpt: str, posQ: int = 16, is_data_pre_quantized: bool = False,
                   channels: int = 32, kernel_size: int = 5, num_samples: int = -1, resultdir: Optional[str] = None,
                   prefix: str = "ue_4stage_conv", batch: int = 1) -> List[Dict[str, object]]:
    os.makedirs(output_folder, exist_ok=True)
    paths = list_inputs(input_glob, num_samples)
    if not paths:
        raise FileNotFoundError(f"no point-cloud files (h5 / ply / bin / npy) under {input_glob}")
    dev = pcc_utils._require_cuda()
    rows: List[Dict[str, object]] = []
    for group in _groups(paths, batch):
        names = [os.path.split(p)[-1] for p in group]
        xyzs = [quantise_device(plyio.read_points_device(p, dev), posQ, is_data_pre_quantized) for p in group]
        outs = [os.path.join(output_folder, name + ".bin") for name in names]
        if batch == 1:
            rs = [pcc_utils.compress_point_cloud(xyzs[0], ckpt, outs[0], channels=channels, kernel_size=kernel_size, posQ=posQ)]
        else:
            rs = pcc_utils.compress_point_clouds(xyzs, ckpt, outs, channels=channels, kernel_size=kernel_size, posQ=posQ)
            for r in rs:
                r["enc_time"] = r["batch_enc_time"] / len(group)
        # the codec stores the SET of voxels; N of the report is the number of input points, as in the reference (:96, :246)
        for name, xyz, r in zip(names, xyzs, rs):
            rows.append({"filedir": name, "bpp": r["file_size_bits"] / max(xyz.shape[0], 1), "enc_time": r["enc_time"],
                         "file_size_bits": r["file_size_bits"], "num_points": int(xyz.shape[0])})
    if resultdir:
        os.makedirs(resultdir, exist_ok=True)
        _write_csv(os.path.join(resultdir, f"{prefix}_data{len(paths)}.csv"), rows, ["bpp", "enc_time", "file_size_bits", "num_points"])
    return rows


def decompress_files(input_glob: str, output_folder: str, ckpt: str, is_data_pre_quantized: bool = False, channels: int = 32,
                     kernel_size: int = 5, resultdir: Optional[str] = None, prefix: str = "ue_4stage_conv",
                     batch: int = 1) -> List[Dict[str, object]]:
    os.makedirs(output_folder, exist_ok=True)
    paths = list_inputs(input_glob, suffixes=(".bin",))
    if not paths:
        raise FileNotFoundError(f"no .bin files under {input_glob}")
    rows: List[Dict[str, object]] = []
    for group in _groups(paths, batch):
        names = [os.path.split(p)[-1] for p in group]
        outs = [os.path.join(output_folder, name + ".ply") for name in names]
        if batch == 1:
            rs = [pcc_utils.decompress_point_cloud(group[0], ckpt, outs[0], channels=channels, kernel_size=kernel_size,
                                                   is_data_pre_quantized=is_data_pre_quantized)]
        else:
            rs = pcc_utils.decompress_point_clouds(group, ckpt, channels=channels, kernel_size=kernel_size,
                                                   is_data_pre_quantized=is_data_pre_quantized, output_paths=outs)
            for r in rs:
                r["dec_time"] = r["batch_dec_time"] / len(group)
        for name, r in zip(names, rs):
            rows.append({"filedir": name, "dec_time": r["dec_time"], "num_points": int(r["num_points"])})
    if resultdir:
        os.makedirs(resultdir, exist_ok=True)
        _write_csv(os.path.join(resultdir, f"{prefix}_dec_data{len(paths)}.csv"), rows, ["dec_time", "num_points"])
    return rows


def _positive(v: str) -> int:
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {n}")
    return n


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="python -m gauspcc_b200.cli", description=__doc__.split("\n\n")[0],
                                 formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    sub = ap.add_subparsers(dest="cmd", required=True)
    for cmd in ("compress", "decompress"):
        sp = sub.add_parser(cmd, formatter_class=argparse.ArgumentDefaultsHelpFormatter)
        sp.add_argument("--input_glob", required=True, help="folder searched recursively for input files")
        sp.add_argument("--output_folder", required=True)
        sp.add_argument("--ckpt", required=True, help="Network(32, 5).state_dict() checkpoint")
        sp.add_argument("--is_data_pre_quantized", action="store_true", help="inputs are integer voxel coordinates already")
        sp.add_argument("--channels", type=int, default=32)
        sp.add_argument("--kernel_size", type=int, default=3)      # the reference scripts' default; the checkpoint must match
        sp.add_argument("--resultdir", default=None, help="folder for the CSV report")
        sp.add_argument("--prefix", default="ue_4stage_conv")
        sp.add_argument("--batch", type=int, default=1,
                        help="files coded per call: N > 1 codes consecutive groups of N files together (same output bytes); each "
                             "file's CSV time is then its group's wall-clock coding time divided by the group's file count")
        if cmd == "compress":
            sp.add_argument("--posQ", type=int, default=16, help="quantisation scale")
            sp.add_argument("--num_samples", type=int, default=-1, help="first N files only (-1 = all)")
    tp = sub.add_parser("train", formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                        help="train a checkpoint on the GPU (gauspcc_b200/train.py) from point-cloud files")
    tp.add_argument("--input_glob", required=True, help="folder searched recursively for training files")
    tp.add_argument("--ckpt_out", required=True, help="checkpoint written in the reference layout (every --save_every steps and at the end)")
    tp.add_argument("--init", default=None, help="checkpoint to start from (default: make_synthetic_state_dict(--init_seed))")
    tp.add_argument("--init_seed", type=int, default=5)
    tp.add_argument("--steps", type=int, default=1000)
    tp.add_argument("--lr", type=float, default=5e-4)
    tp.add_argument("--seed", type=int, default=0, help="draws the patch order")
    tp.add_argument("--kernel_size", type=int, default=3, choices=(3, 5))
    tp.add_argument("--posQ", type=int, default=16, help="quantisation scale (as compress)")
    tp.add_argument("--is_data_pre_quantized", action="store_true", help="inputs are integer voxel coordinates already")
    tp.add_argument("--max_points", type=int, default=150_000, help="largest kd-tree patch")
    tp.add_argument("--save_every", type=int, default=0)
    tp.add_argument("--batch_size", type=_positive, default=1,
                    help="patches per step, run as one union octree (batch 1 is single-patch training)")
    tp.add_argument("--conv_families", default="v6", choices=("v6", "codec"),
                    help="conv kernels of the levels: v6 = the mma.sync conv everywhere, codec = the family the codec codes each "
                         "level with (the sparse or tcgen05 conv on big levels)")
    tp.add_argument("--resultdir", default=None, help="folder for the CSV training log")
    tp.add_argument("--prefix", default="ue_4stage_conv")
    return ap


def train_files(input_glob: str, ckpt_out: str, init: Optional[str] = None, steps: int = 1000, lr: float = 5e-4, seed: int = 0,
                kernel_size: int = 3, posQ: int = 16, is_data_pre_quantized: bool = False, max_points: int = 150_000,
                save_every: int = 0, resultdir: Optional[str] = None, prefix: str = "ue_4stage_conv",
                init_seed: int = 5, batch_size: int = 1, conv_families: str = "v6") -> List[Dict[str, object]]:
    """Train a checkpoint (gauspcc_b200/train.py) on the files under input_glob, read and quantised exactly as `compress` reads them,
    so that the checkpoint learns the voxels it will code.  Writes `<prefix>_train_data<N>.csv` (one row per step) to resultdir."""
    from . import train as T
    dev = pcc_utils._require_cuda()
    paths = list_inputs(input_glob)
    if not paths:
        raise FileNotFoundError(f"no point-cloud files (h5 / ply / bin / npy) under {input_glob}")
    clouds = [quantise_device(plyio.read_points_device(p, dev), posQ, is_data_pre_quantized) for p in paths]
    d = os.path.dirname(os.path.abspath(ckpt_out))
    os.makedirs(d, exist_ok=True)
    _, rows = T.train(clouds, ckpt_out, init=init, steps=steps, lr=lr, seed=seed, kernel_size=kernel_size, max_points=max_points,
                      save_every=save_every, synthetic_seed=init_seed, batch_size=batch_size, conv_families=conv_families)
    if resultdir:
        os.makedirs(resultdir, exist_ok=True)
        with open(os.path.join(resultdir, f"{prefix}_train_data{len(paths)}.csv"), "w", newline="") as f:
            w = csv.DictWriter(f, fieldnames=list(rows[0].keys()))
            w.writeheader()
            w.writerows(rows)
    return rows


def main(argv: Optional[List[str]] = None) -> int:
    a = build_parser().parse_args(argv)
    t0 = time.time()
    if a.cmd == "train":
        rows = train_files(a.input_glob, a.ckpt_out, a.init, a.steps, a.lr, a.seed, a.kernel_size, a.posQ, a.is_data_pre_quantized,
                           a.max_points, a.save_every, a.resultdir, a.prefix, a.init_seed, a.batch_size, a.conv_families)
        tail = rows[-min(20, len(rows)):]
        print("Steps: {:d} | bpp first {:.3f} last {:.3f} (mean of up to 20 steps) | Max GPU memory:{:.2f}MB".format(
            len(rows), float(np.mean([r["bpp"] for r in rows[:20]])), float(np.mean([r["bpp"] for r in tail])),
            torch.cuda.max_memory_allocated() / 1024 / 1024))
    elif a.cmd == "compress":
        rows = compress_files(a.input_glob, a.output_folder, a.ckpt, a.posQ, a.is_data_pre_quantized, a.channels, a.kernel_size,
                              a.num_samples, a.resultdir, a.prefix, a.batch)
        print("Total: {:d} | Average bitrate:{:.3f} | Encoding time:{:.3f}s | Max GPU memory:{:.2f}MB".format(
            len(rows), float(np.mean([r["bpp"] for r in rows])), float(np.mean([r["enc_time"] for r in rows])),
            torch.cuda.max_memory_allocated() / 1024 / 1024))
    else:
        rows = decompress_files(a.input_glob, a.output_folder, a.ckpt, a.is_data_pre_quantized, a.channels, a.kernel_size,
                                a.resultdir, a.prefix, a.batch)
        print("Total: {:d} | Decoding time:{:.3f}s | Max GPU memory:{:.2f}MB".format(
            len(rows), float(np.mean([r["dec_time"] for r in rows])), torch.cuda.max_memory_allocated() / 1024 / 1024))
    print(f"wall {time.time() - t0:.2f} s")
    return 0


if __name__ == "__main__":
    sys.exit(main())
