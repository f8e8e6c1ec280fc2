"""Host logic of training on the codec's conv families: `cli train --conv_families`, the argument checks of train() and
GausPcgcNet, and the family a kernel map reports."""
import pytest
import torch

from gauspcc_b200 import _lib, cli
from gauspcc_b200 import train as T
from gauspcc_b200.codec import KMap


def test_cli_conv_families_argument():
    base = ["train", "--input_glob", "d", "--ckpt_out", "c.pth"]
    assert cli.build_parser().parse_args(base).conv_families == "v6"
    assert cli.build_parser().parse_args(base + ["--conv_families", "codec"]).conv_families == "codec"
    for bad in ("um", "sparse", "V6", ""):
        with pytest.raises(SystemExit):
            cli.build_parser().parse_args(base + ["--conv_families", bad])


def test_conv_families_are_checked():
    assert T.CONV_FAMILIES == ("v6", "codec")
    assert T.check_conv_families("codec") == "codec"
    for bad in ("um", "sparse", None, "CODEC"):
        with pytest.raises(ValueError):
            T.check_conv_families(bad)
        with pytest.raises(ValueError):
            T.GausPcgcNet(5, conv_families=bad)
        with pytest.raises(ValueError):                     # checked before anything else, with or without a GPU
            T.train([torch.zeros((10, 3), dtype=torch.int32)], steps=1, conv_families=bad)


def test_default_network_is_v6():
    assert T.GausPcgcNet(5).conv_families == "v6"
    assert T.GausPcgcNet(3, conv_families="codec").conv_families == "codec"


def test_kmap_rule_rejects_an_unknown_family_value():
    net = T.GausPcgcNet(5)
    net.conv_families = "tcgen05"
    with pytest.raises(ValueError):
        net.kmap(torch.zeros(4, dtype=torch.int64))


def test_kmap_family():
    seg = torch.zeros(1, dtype=torch.int32)
    pairs = torch.zeros(1, dtype=torch.int64)
    assert T.kmap_family(KMap(seg, pairs, 0, 64)) == "v6"
    assert T.kmap_family(KMap(seg, pairs, 0, 0, sparse=True)) == "sparse"
    assert T.kmap_family(KMap(seg, None, 0, 512, um_rows=512)) == "um"
    assert T._family_counts([KMap(seg, pairs, 0, 64), KMap(seg, None, 0, 512, um_rows=512), KMap(seg, pairs, 0, 64)]) == \
        {"v6": 2, "sparse": 0, "um": 1}


def test_sparse_conv_fn_needs_a_built_kernel_map():
    """a map with neither a pair stream nor a tcgen05 tiling is refused before any kernel runs"""
    with pytest.raises(_lib.GpcError):
        T.SparseConvFn.apply(torch.zeros((4, 32)), torch.zeros((125, 32, 32)), KMap(torch.zeros(1, dtype=torch.int32), None, 0, 0))
