"""Host logic of minibatch training: `cli train --batch_size`, the patch order of train.batches and the union-level helper
batch.union_levels (a pure function of the members' levels and translations)."""
import pytest
import torch

from gauspcc_b200 import cli
from gauspcc_b200 import train as T
from gauspcc_b200.batch import Z_SHIFT, plan_unions, union_levels
from gauspcc_b200.codec import Level


def test_cli_batch_size_argument():
    base = ["train", "--input_glob", "d", "--ckpt_out", "c.pth"]
    assert cli.build_parser().parse_args(base).batch_size == 1
    assert cli.build_parser().parse_args(base + ["--batch_size", "8"]).batch_size == 8
    for bad in ("0", "-3", "x"):
        with pytest.raises(SystemExit):
            cli.build_parser().parse_args(base + ["--batch_size", bad])


def test_batch_size_one_is_the_single_patch_order():
    """the order train() used before batches existed: one permutation per pass, popped one patch per step"""
    n, seed, steps = 7, 3, 30
    gen = torch.Generator().manual_seed(seed)
    order, want = [], []
    for _ in range(steps):
        if not order:
            order = torch.randperm(n, generator=gen).tolist()
        want.append([order.pop(0)])
    it = T.batches(n, 1, seed)
    assert [next(it) for _ in range(steps)] == want


@pytest.mark.parametrize("n,b", [(8, 4), (7, 3), (5, 5), (16, 16), (9, 2)])
def test_every_patch_once_per_pass(n, b):
    it = T.batches(n, b, 11)
    flat = [i for _ in range(3 * n) for i in next(it)]
    assert all(len(x) == b for x in [next(T.batches(n, b, 11))])
    for p in range(3 * b):                                  # the stream is whole permutations of range(n), one after another
        assert sorted(flat[p * n:(p + 1) * n]) == list(range(n))
    again = T.batches(n, b, 11)
    assert [i for _ in range(3 * n) for i in next(again)] == flat
    single = T.batches(n, 1, 11)
    assert [next(single)[0] for _ in range(len(flat))] == flat          # batch b = b consecutive entries of the B = 1 stream


def test_batch_size_out_of_range():
    with pytest.raises(ValueError):
        T.batches(3, 4, 0)
    with pytest.raises(ValueError):
        T.batches(3, 0, 0)


def _key(x, y, z):
    return ((z + (1 << 20)) << Z_SHIFT) | ((y + (1 << 20)) << 21) | (x + (1 << 20))


def _levels(depth, rows, z0=0):
    """a synthetic pyramid, coarsest first: level i has rows[i] voxels at (r, 0, z0)"""
    return [Level(torch.tensor([_key(r, 0, z0) for r in range(rows[i])], dtype=torch.int64),
                  torch.full((rows[i],), 1 + i, dtype=torch.uint8), rows[i]) for i in range(depth)]


def test_union_levels_is_the_encoders_layout():
    a = _levels(3, [2, 4, 8])                # depth 3: scales 3, 2, 1
    b = _levels(2, [3, 5])                   # depth 2: scales 2, 1
    c = _levels(3, [1, 2, 6])
    members = [a, c, b]                      # plan_unions order: deepest first
    tz = [0, 64, 192]
    U, K, M = union_levels(members, tz)
    assert sorted(U) == [1, 2, 3] and K == {1: 3, 2: 2} and M == {1: 8 + 6 + 5, 2: 4 + 2}
    assert U[3].members == [0, 1] and U[3].ranges == [(0, 2), (2, 3)]
    assert U[2].members == [0, 1, 2] and U[2].ranges == [(0, 4), (4, 6), (6, 9)]
    assert U[1].ranges == [(0, 8), (8, 14), (14, 19)]
    for sg in (1, 2, 3):
        for j, (r0, r1) in zip(U[sg].members, U[sg].ranges):
            lv = members[j][len(members[j]) - sg]
            assert torch.equal(U[sg].keys[r0:r1], lv.keys + ((tz[j] >> sg) << Z_SHIFT))
            assert torch.equal(U[sg].occ[r0:r1], lv.occ)
    again = union_levels(members, tz)
    assert all(torch.equal(again[0][sg].keys, U[sg].keys) for sg in U)


def test_union_levels_from_the_planner():
    depths, rows = [4, 2, 3], [100, 40, 70]
    unions, singles = plan_unions([0, 0, 0], [500, 100, 300], depths, rows, 10_000)
    assert len(unions) == 1 and not singles
    up = unions[0]
    lv = {s: _levels(depths[s], [5 * (i + 1) for i in range(depths[s])]) for s in range(3)}
    U, K, M = union_levels([lv[s] for s in up.scenes], up.tz)
    assert [depths[s] for s in up.scenes] == [4, 3, 2]
    assert K == {1: 3, 2: 2, 3: 1}
    for sg in K:
        assert M[sg] == U[sg].ranges[K[sg] - 1][1]
