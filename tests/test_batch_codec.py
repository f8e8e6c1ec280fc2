"""Batched compress / decompress (pcc_utils.compress_point_clouds / decompress_point_clouds, gauspcc_b200/batch.py): every file is
byte-identical to the single-scene call's, and every decoded cloud equals the single decode row for row."""
import contextlib
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    from gauspcc_b200.weights import save_synthetic_checkpoint
    return save_synthetic_checkpoint(str(tmp_path_factory.mktemp("w") / "GausPcgc" / "best_model_ue_4stage_conv.pt"))


def _mixed_scenes():
    """base-only, a few hundred, 2 K, 20 K and 40 K anchors of different depths; duplicates; int32 / float32 / numpy; far away"""
    from gauspcc_b200.synth import hac_like_cloud
    dev = torch.device("cuda")
    tiny = np.array([[1, 2, 3], [4, 5, 6], [1, 2, 3], [9, 9, 9]], np.int32)
    a = hac_like_cloud(300, seed=1, extent_log2=9)
    b = hac_like_cloud(2000, seed=2, extent_log2=12)
    b = np.concatenate([b, b[:200]])                                       # duplicate points
    c = hac_like_cloud(20000, seed=3, extent_log2=14)
    d = hac_like_cloud(40000, seed=4, extent_log2=16)
    far = hac_like_cloud(3000, seed=5, extent_log2=11) + np.array([900_000, -700_000, 1_500_000], np.int32)
    return [tiny, torch.tensor(a, device=dev), torch.tensor(b.astype(np.float32)), c, torch.tensor(d, dtype=torch.float32, device=dev),
            far]


def _single(xyzs, ckpt, root, **kw):
    from gauspcc_b200 import pcc_utils
    paths = [os.path.join(root, "single", f"{i}.bin") for i in range(len(xyzs))]
    for x, p in zip(xyzs, paths):
        pcc_utils.compress_point_cloud(x, ckpt, p, **kw)
    return paths


def _batch(xyzs, ckpt, root, **kw):
    from gauspcc_b200 import pcc_utils
    paths = [os.path.join(root, "batch", f"{i}.bin") for i in range(len(xyzs))]
    res = pcc_utils.compress_point_clouds(xyzs, ckpt, paths, **kw)
    return paths, res


def _same_bytes(pa, pb):
    for a, b in zip(pa, pb):
        with open(a, "rb") as fa, open(b, "rb") as fb:
            assert fa.read() == fb.read(), f"{b} differs from {a}"


@contextlib.contextmanager
def _attrs(codec, **kw):
    old = {k: getattr(codec, k) for k in kw}
    for k, v in kw.items():
        setattr(codec, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(codec, k, v)


def test_bytes_and_decode_match_the_single_path(ckpt, tmp_path):
    from gauspcc_b200 import pcc_utils
    xyzs = _mixed_scenes()
    single = _single(xyzs, ckpt, str(tmp_path))
    paths, res = _batch(xyzs, ckpt, str(tmp_path))
    _same_bytes(single, paths)
    assert len({r["batch_enc_time"] for r in res}) == 1 and all(r["num_points"] == x.shape[0] for r, x in zip(res, xyzs))
    assert pcc_utils._batch(pcc_utils._codec(ckpt, 32, 5)).last_stats["unions"] == 1
    for sorted_output in (False, True):
        for pre_q in (True, False):
            dec = pcc_utils.decompress_point_clouds(paths, ckpt, is_data_pre_quantized=pre_q, sorted_output=sorted_output)
            for p, d in zip(paths, dec):
                ref = pcc_utils.decompress_point_cloud(p, ckpt, is_data_pre_quantized=pre_q, sorted_output=sorted_output)["point_cloud"]
                assert torch.equal(d["point_cloud"], ref), (p, sorted_output, pre_q)
    dec = pcc_utils.decompress_point_clouds(paths, ckpt)
    for x, d in zip(xyzs, dec):                                               # lossless
        x = x.cpu().numpy() if torch.is_tensor(x) else x
        assert np.array_equal(np.unique(d["point_cloud"].cpu().numpy().astype(np.int64), axis=0),
                              np.unique(np.asarray(x, dtype=np.int64), axis=0))


@pytest.mark.parametrize("family", ["sparse", "umma", "v6d", "mixed"])
def test_forced_conv_families(ckpt, tmp_path, family):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    attrs = {"sparse": dict(sparse_min_rows=1, sparse_max_density=1e9),
             "umma": dict(um_min_rows=1, sparse_max_density=0.0),
             "v6d": dict(adaptive_tiles=False, tile_rows=128, v6_variant=48, um_min_rows=1 << 40, sparse_min_rows=1 << 40),
             # scenes of one union level on different families: the 20 K / 40 K scenes' big levels on tcgen05, the rest on mma.sync
             "mixed": dict(um_min_rows=8_000, sparse_max_density=0.0)}[family]
    xyzs = [hac_like_cloud(n, seed=10 + i, extent_log2=e) for i, (n, e) in enumerate([(20000, 14), (900, 10), (40000, 15), (5000, 12)])]
    with _attrs(codec, **attrs):
        single = _single(xyzs, ckpt, str(tmp_path))
        paths, _ = _batch(xyzs, ckpt, str(tmp_path))
        _same_bytes(single, paths)
        dec = pcc_utils.decompress_point_clouds(paths, ckpt)
        for p, d in zip(paths, dec):
            assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"])
        if family == "mixed":
            bc = pcc_utils._batch(codec)
            assert bc.last_stats["unions"] == 1


def test_kernel_size_3(tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ck3 = save_synthetic_checkpoint(str(tmp_path / "k3" / "w.pt"), kernel_size=3)
    xyzs = [hac_like_cloud(n, seed=20 + n, extent_log2=12) for n in (3000, 800)]
    single = _single(xyzs, ck3, str(tmp_path), kernel_size=3)
    paths, _ = _batch(xyzs, ck3, str(tmp_path), kernel_size=3)
    _same_bytes(single, paths)
    for p, d in zip(paths, pcc_utils.decompress_point_clouds(paths, ck3, kernel_size=3)):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ck3, kernel_size=3)["point_cloud"])


def test_two_unions_and_a_batch_of_one(ckpt, tmp_path):
    from gauspcc_b200 import bitstream, pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    bc = pcc_utils._batch(pcc_utils._codec(ckpt, 32, 5))
    xyzs = [hac_like_cloud(n, seed=30 + i, extent_log2=12) for i, n in enumerate((4000, 3000, 5000))]
    single = _single(xyzs, ckpt, str(tmp_path))
    with _attrs(bc, max_rows=5000):
        paths, _ = _batch(xyzs, ckpt, str(tmp_path))
        assert bc.last_stats["unions"] >= 2
        _same_bytes(single, paths)
    est = []                                          # the decoder plans with one row per stream byte
    for p in paths:
        with open(p, "rb") as f:
            est.append(sum(len(x) for x in bitstream.read_file(f.read())[3]))
    with _attrs(bc, max_rows=max(est) + min(est) // 2):
        dec = pcc_utils.decompress_point_clouds(paths, ckpt)
        assert bc.last_stats["unions"] >= 2
    for p, d in zip(paths, dec):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"])
    one, _ = _batch(xyzs[:1], ckpt, str(tmp_path / "one"))
    _same_bytes(single[:1], one)
    assert torch.equal(pcc_utils.decompress_point_clouds(one, ckpt)[0]["point_cloud"],
                       pcc_utils.decompress_point_cloud(one[0], ckpt)["point_cloud"])


def test_rejected_inputs_and_truncated_file(ckpt, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    assert pcc_utils.compress_point_clouds([], ckpt, []) == []
    assert pcc_utils.decompress_point_clouds([], ckpt) == []
    xyzs = [hac_like_cloud(n, seed=40 + n, extent_log2=12) for n in (3000, 2000)]
    with pytest.raises(ValueError):
        pcc_utils.compress_point_clouds(xyzs, ckpt, [str(tmp_path / "a.bin")])
    paths, _ = _batch(xyzs, ckpt, str(tmp_path))
    v2 = str(tmp_path / "v2" / "xyz_pcc.bin")
    pcc_utils.compress_point_cloud(xyzs[0], ckpt, v2, gpu_coder_chunk=2048)
    with pytest.raises(ValueError, match="version 2"):
        pcc_utils.decompress_point_clouds([paths[0], v2], ckpt)
    with open(paths[1], "rb") as f:
        blob = f.read()
    bad = str(tmp_path / "bad.bin")
    with open(bad, "wb") as f:
        f.write(blob[:len(blob) // 2])
    with pytest.raises(Exception):
        pcc_utils.decompress_point_clouds([paths[0], bad], ckpt)
    # the codec is still usable afterwards
    assert torch.equal(pcc_utils.decompress_point_clouds(paths[:1], ckpt)[0]["point_cloud"],
                       pcc_utils.decompress_point_cloud(paths[0], ckpt)["point_cloud"])


def test_batch_decode_issues_fewer_launches(ckpt, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    xyzs = [hac_like_cloud(1500 + 100 * i, seed=50 + i, extent_log2=11) for i in range(8)]
    paths, _ = _batch(xyzs, ckpt, str(tmp_path))
    single = 0
    for p in paths:
        pcc_utils.decompress_point_cloud(p, ckpt)
        single += codec.last_stats["launches"]
    pcc_utils.decompress_point_clouds(paths, ckpt)
    batch = pcc_utils._batch(codec).last_stats["launches"]
    assert batch < single, (batch, single)


def test_production_size_default_families(ckpt, tmp_path):
    """scenes of 400 K, 250 K and 160 K anchors under the default family thresholds: one union level has members on the sparse and on
    the tcgen05 conv (recorded from BatchCodec._kmaps, so that the test keeps meaning it); files and decoded rows as the single path"""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    assert (codec.um_min_rows, codec.sparse_min_rows, codec.sparse_max_density) == (150_000, 150_000, 4.5)
    bc = pcc_utils._batch(codec)
    xyzs = [hac_like_cloud(n, seed=61 + i, extent_log2=16) for i, n in enumerate((400_000, 250_000, 160_000))]
    single = _single(xyzs, ckpt, str(tmp_path))
    levels = []
    kmaps = bc._kmaps

    def record(lv):
        kms = kmaps(lv)
        levels.append(["um" if k.um_rows else ("sparse" if k.sparse else "v6") for k in kms])
        return kms
    bc._kmaps = record
    try:
        paths, _ = _batch(xyzs, ckpt, str(tmp_path))
        assert bc.last_stats["unions"] == 1
        assert any("sparse" in f and "um" in f for f in levels), levels
        levels.clear()
        dec = pcc_utils.decompress_point_clouds(paths, ckpt)
        assert any("sparse" in f and "um" in f for f in levels), levels
    finally:
        del bc._kmaps
    _same_bytes(single, paths)
    for p, d in zip(single, dec):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"]), p
