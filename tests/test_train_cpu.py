"""Host logic of the trainer (gauspcc_b200/train.py) and of `cli train`: kd-tree patches, the state_dict layout, argument parsing and
the refusal to run without CUDA."""
import ast
import os

import numpy as np
import pytest
import torch

from gauspcc_b200 import _lib, cli
from gauspcc_b200 import train as T
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import make_synthetic_state_dict, reference_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n,limit", [(0, 10), (1, 1), (17, 5), (1000, 1000), (50_000, 7_000), (40_000, 150_000)])
def test_partition_covers_every_point_once(n, limit):
    xyz = torch.tensor(hac_like_cloud(n, seed=n, extent_log2=12)) if n else torch.zeros((0, 3), dtype=torch.int32)
    parts = T.partition(xyz, limit)
    assert all(0 < p.numel() <= limit for p in parts)
    got = torch.cat(parts) if parts else torch.zeros(0, dtype=torch.int64)
    assert torch.equal(torch.sort(got).values, torch.arange(n))
    again = T.partition(xyz, limit)
    assert len(again) == len(parts) and all(torch.equal(a, b) for a, b in zip(parts, again))


def test_partition_splits_at_the_median_of_the_longest_axis():
    rng = np.random.default_rng(3)
    xyz = torch.tensor(np.stack([rng.integers(0, 1000, 64), rng.integers(0, 10, 64), rng.integers(0, 10, 64)], 1), dtype=torch.int32)
    left, right = T.partition(xyz, 32)
    assert left.numel() == right.numel() == 32
    assert int(xyz[left, 0].max()) <= int(xyz[right, 0].min())
    tied = torch.zeros((9, 3), dtype=torch.int32)                   # every coordinate equal: split in input order
    assert [p.tolist() for p in T.partition(tied, 4)] == [[0, 1, 2, 3], [4, 5], [6, 7, 8]]


@pytest.mark.parametrize("k", [3, 5])
def test_state_dict_is_the_reference_layout(k):
    net = T.GausPcgcNet(k, seed=5)
    sd = net.state_dict()
    assert [(n, tuple(t.shape)) for n, t in sd.items()] == list(reference_layout(32, k).items())
    ref = make_synthetic_state_dict(5, 32, k)
    assert all(torch.equal(sd[n], ref[n]) for n in ref)
    assert "fog.conv.kernel" not in dict(net.named_parameters())                # a constant, not trained
    assert len(list(net.parameters())) == len(ref) - 1
    ck = net.checkpoint()
    assert all(torch.equal(ck[n], ref[n]) and ck[n].device.type == "cpu" for n in ref)
    other = make_synthetic_state_dict(9, 32, k)
    assert all(torch.equal(T.GausPcgcNet(k, state_dict=other).state_dict()[n], other[n]) for n in other)
    with pytest.raises(RuntimeError):
        T.GausPcgcNet(k, state_dict=make_synthetic_state_dict(5, 32, 8 - k))


def test_k3_offsets_are_the_inner_cube():
    assert len(T.K5_OF_K3) == 27 and T.K5_OF_K3[13] == 62
    assert sorted(124 - k for k in T.K5_OF_K3) == sorted(T.K5_OF_K3)          # the mirror keeps a 3^3 kernel inside the 3^3 slots


def test_cli_train_arguments():
    a = cli.build_parser().parse_args(["train", "--input_glob", "d", "--ckpt_out", "c.pth"])
    assert (a.cmd, a.input_glob, a.ckpt_out, a.init, a.steps, a.lr, a.seed, a.kernel_size, a.posQ, a.is_data_pre_quantized,
            a.max_points, a.resultdir) == ("train", "d", "c.pth", None, 1000, 5e-4, 0, 3, 16, False, 150_000, None)
    a = cli.build_parser().parse_args(["train", "--input_glob", "d", "--ckpt_out", "c", "--init", "i.pth", "--steps", "7", "--lr", "1e-3",
                                       "--seed", "4", "--kernel_size", "5", "--posQ", "2", "--is_data_pre_quantized", "--max_points",
                                       "999", "--resultdir", "r"])
    assert (a.init, a.steps, a.lr, a.seed, a.kernel_size, a.posQ, a.is_data_pre_quantized, a.max_points, a.resultdir) == \
        ("i.pth", 7, 1e-3, 4, 5, 2, True, 999, "r")
    for bad in (["train", "--input_glob", "d"], ["train", "--input_glob", "d", "--ckpt_out", "c", "--kernel_size", "4"]):
        with pytest.raises(SystemExit):
            cli.build_parser().parse_args(bad)
    a = cli.build_parser().parse_args(["compress", "--input_glob", "d", "--output_folder", "o", "--ckpt", "c"])   # unchanged
    assert (a.cmd, a.kernel_size, a.posQ, a.batch) == ("compress", 3, 16, 1)


def test_train_without_cuda_raises(monkeypatch, tmp_path):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(_lib.GpcError):
        T.train([torch.zeros((100, 3), dtype=torch.int32)], steps=1)
    np.save(tmp_path / "a.npy", np.zeros((10, 3)))
    with pytest.raises(_lib.GpcError):
        cli.main(["train", "--input_glob", str(tmp_path), "--ckpt_out", str(tmp_path / "c.pth"), "--steps", "1"])
    assert not (tmp_path / "c.pth").exists()


def test_trainer_never_imports_oracle():
    tree = ast.parse(open(os.path.join(ROOT, "gauspcc_b200", "train.py")).read())
    names = [a.name for n in ast.walk(tree) if isinstance(n, ast.Import) for a in n.names]
    names += [n.module or "" for n in ast.walk(tree) if isinstance(n, ast.ImportFrom)]
    assert not any(m.split(".")[0] == "oracle" for m in names)
