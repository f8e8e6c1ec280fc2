"""The union planner of the batched codec (gauspcc_b200/batch.py) as a pure function of per-scene z extents, depths and rows."""
import numpy as np
import pytest

from gauspcc_b200.batch import plan_unions
from gauspcc_b200.codec import COORD_LIMIT


def _scenes(n, seed=0, depth_range=(2, 13), ext_range=(10, 20000)):
    rng = np.random.default_rng(seed)
    depths = rng.integers(depth_range[0], depth_range[1], n)
    lo = rng.integers(-COORD_LIMIT // 2, COORD_LIMIT // 4, n)
    hi = lo + rng.integers(ext_range[0], ext_range[1], n)
    rows = rng.integers(100, 600_000, n)
    return lo.tolist(), hi.tolist(), depths.tolist(), rows.tolist()


def _check(lo, hi, depths, rows, max_rows, unions, singles):
    D = max(depths)
    seen = sorted([s for u in unions for s in u.scenes] + list(singles))
    assert seen == list(range(len(depths))), "every scene is planned exactly once"
    for u in unions:
        assert u.rows == sum(rows[s] for s in u.scenes) <= max_rows
        assert [depths[s] for s in u.scenes] == sorted((depths[s] for s in u.scenes), reverse=True), "deepest scenes first"
        for s, t in zip(u.scenes, u.tz):
            assert t % (1 << (D + 1)) == 0, "translation is a multiple of 2^(D+1)"
            assert -COORD_LIMIT <= lo[s] + t and hi[s] + t <= COORD_LIMIT, "translated z fits the key fields"
        for (a, ta), (b, tb) in zip(zip(u.scenes, u.tz), zip(u.scenes[1:], u.tz[1:])):
            assert hi[a] + ta < lo[b] + tb, "scenes are stacked in z order"
            for sg in range(0, D + 1):         # at every coded scale the two scenes are >= 3 voxels apart
                assert ((lo[b] + tb) >> sg) - ((hi[a] + ta) >> sg) >= 3


@pytest.mark.parametrize("seed", range(5))
def test_random_batches(seed):
    lo, hi, depths, rows = _scenes(40, seed)
    unions, singles = plan_unions(lo, hi, depths, rows, max_rows=4_000_000)
    _check(lo, hi, depths, rows, 4_000_000, unions, singles)
    assert not singles


def test_row_cap_splits_the_batch():
    lo, hi, depths, rows = [0] * 6, [1000] * 6, [8] * 6, [100] * 6
    unions, singles = plan_unions(lo, hi, depths, rows, max_rows=250)
    assert [u.scenes for u in unions] == [[0, 1], [2, 3], [4, 5]] and not singles
    _check(lo, hi, depths, rows, 250, unions, singles)


def test_key_capacity_splits_the_batch():
    ext = COORD_LIMIT * 4 // 5               # three such scenes cannot share the 2^21 z range
    lo, hi, depths, rows = [0] * 3, [ext] * 3, [4] * 3, [10] * 3
    unions, singles = plan_unions(lo, hi, depths, rows, max_rows=10**9)
    assert len(unions) == 2 and sum(len(u.scenes) for u in unions) == 3 and not singles
    _check(lo, hi, depths, rows, 10**9, unions, singles)


def test_oversized_scene_goes_to_the_single_path():
    lo, hi, depths, rows = [0, 5 - COORD_LIMIT, 0], [50, COORD_LIMIT + 5, 50], [3, 3, 3], [10, 10, 10]
    unions, singles = plan_unions(lo, hi, depths, rows, max_rows=10**9)
    assert singles == [1] and [u.scenes for u in unions] == [[0, 2]]
    unions, singles = plan_unions([0, 0], [5, 5], [3, 3], [10, 500], max_rows=100)
    assert singles == [1] and [u.scenes for u in unions] == [[0]]


def test_input_order_is_kept_among_equal_depths():
    lo, hi, depths, rows = [0] * 5, [100] * 5, [5, 7, 5, 7, 5], [1] * 5
    unions, _ = plan_unions(lo, hi, depths, rows, max_rows=100)
    assert [u.scenes for u in unions] == [[1, 3, 0, 2, 4]]


def test_empty_and_mismatched_inputs():
    assert plan_unions([], [], [], [], 10) == ([], [])
    with pytest.raises(ValueError):
        plan_unions([0], [1, 2], [3], [4], 10)
