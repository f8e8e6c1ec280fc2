"""Container version 2 through the batch API (compress_point_clouds / decompress_point_clouds with gpu_coder_chunk): every file is
byte-identical to compress_point_cloud(..., gpu_coder_chunk=c)'s, every decoded cloud equals decompress_point_cloud's row for row,
and the union decoder decodes its stages on the GPU (gpc_chunk_decode_u16_ranges) without a host round trip per stage."""
import contextlib
import ctypes as C
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


def _same_rows(paths, ckpt, **kw):
    from gauspcc_b200 import pcc_utils
    dec = pcc_utils.decompress_point_clouds(paths, ckpt, **kw)
    for p, d in zip(paths, dec):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt, **kw)["point_cloud"]), (p, kw)
    return dec


@contextlib.contextmanager
def _attrs(obj, **kw):
    old = {k: getattr(obj, k) for k in kw}
    for k, v in kw.items():
        setattr(obj, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(obj, k, v)


@contextlib.contextmanager
def _counting(obj, name):
    """count the calls of obj.name (an instance attribute shadows the method for the duration)"""
    calls = []
    fn = getattr(obj, name)

    def wrapped(*a, **kw):
        calls.append(1)
        return fn(*a, **kw)
    setattr(obj, name, wrapped)
    try:
        yield calls
    finally:
        delattr(obj, name)


def _rewrite(path, out, edit):
    """write `out`: the file at `path` with edit(streams) applied to its stream list (trailer included)"""
    from gauspcc_b200 import bitstream
    with open(path, "rb") as f:
        posQ, bx, bo, streams = bitstream.read_file(f.read())
    with open(out, "wb") as f:
        f.write(bitstream.write_file(posQ, bx, bo, edit(list(streams))))
    return out


# ---------------------------------------------------------------------------------------------------------------- the kernel
def _encode_segments(lib, cdf, sym, bounds, dev):
    """gpc_chunk_encode_lohi over explicit chunk boundaries, the words built in numpy from the CDF rows -> (bytes, offsets)"""
    n, Lp = cdf.shape
    A = Lp - 1
    rows = np.arange(n)
    lo = cdf[rows, sym].astype(np.uint32)
    hi = np.where(sym == A - 1, 0, cdf[rows, np.minimum(sym.astype(np.int64) + 1, A)]).astype(np.uint32)   # 0 == 0x10000
    lohi = torch.from_numpy((lo | (hi << 16)).view(np.int32)).to(dev)
    starts = torch.from_numpy(bounds.view(np.int32)).to(dev)
    chunks = bounds.shape[0] - 1
    max_chunk = int(np.diff(bounds.astype(np.int64)).max())
    cnt = torch.empty(chunks, dtype=torch.int32, device=dev)
    offs = torch.empty(chunks + 1, dtype=torch.int32, device=dev)
    wb = lib.gpc_chunk_workspace_bytes(chunks, max_chunk)
    ws = torch.empty(wb, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    assert lib.gpc_chunk_encode_lohi(lohi.data_ptr(), starts.data_ptr(), chunks, max_chunk, cnt.data_ptr(), offs.data_ptr(),
                                     ws.data_ptr(), wb, st) == 0
    total = int(offs[-1].item())
    out = torch.empty(total + 64, dtype=torch.uint8, device=dev)
    assert lib.gpc_chunk_merge(ws.data_ptr(), chunks, max_chunk, offs.data_ptr(), out.data_ptr(), st) == 0
    return out, offs


def _decode_ranges(lib, cdf_d, Lp, payload, offs, bounds, n, dev, guard=0):
    rows = torch.from_numpy(np.asarray(bounds, dtype=np.uint32).view(np.int32)).to(dev)
    sym = torch.full((n + guard,), 0xAB, dtype=torch.uint8, device=dev)
    assert lib.gpc_chunk_decode_u16_ranges(cdf_d.data_ptr(), Lp, payload.data_ptr(), offs.data_ptr(), rows.data_ptr(),
                                           rows.shape[0] - 1, n, sym.data_ptr(), torch.cuda.current_stream(dev).cuda_stream) == 0
    return sym.cpu().numpy()


@pytest.mark.parametrize("Lp", [3, 5, 17])
def test_ranges_decoder_kernel(Lp):
    """random CDF rows and symbols in segments of different chunk lengths: the symbols come back exactly, every chunk is the oracle
    coder's stream of its rows, and on one uniform segment the output is gpc_chunk_decode_u16's byte for byte"""
    from gauspcc_b200 import _lib
    from oracle import oracle as O
    lib = _lib.load()
    dev = torch.device("cuda")
    rng = np.random.default_rng(Lp)
    A = Lp - 1
    segs = [(1000, 64), (97, 32), (5000, 2048), (1, 7), (3333, 100), (4097, 512)]       # (rows, chunk length)
    n = sum(r for r, _ in segs)
    bounds, r0 = [0], 0
    for r, cl in segs:
        bounds += [r0 + min(o + cl, r) for o in range(0, r, cl)]
        r0 += r
    bounds = np.array(bounds, dtype=np.uint32)
    p = rng.dirichlet(np.full(A, 0.3), size=n).astype(np.float32)
    p[:50] = 0
    p[:50, A - 1] = 1.0
    cdf = O.cdf_u16(p)
    sym = rng.integers(0, A, n).astype(np.uint8)
    pick = rng.random(n) < 0.5                                                          # half the symbols drawn from their rows
    sym[pick] = [rng.choice(A, p=q / q.sum()) for q in p[pick].astype(np.float64)]
    sym[:50] = A - 1
    payload, offs = _encode_segments(lib, cdf, sym, bounds, dev)
    cdf_d = torch.from_numpy(cdf.view(np.int16)).to(dev)
    got = _decode_ranges(lib, cdf_d, Lp, payload, offs, bounds, n, dev)
    assert np.array_equal(got, sym)
    host, offs_h = payload.cpu().numpy().tobytes(), offs.cpu().numpy().astype(np.int64)
    for w in range(bounds.shape[0] - 1):
        a, b = int(bounds[w]), int(bounds[w + 1])
        assert host[offs_h[w]:offs_h[w + 1]] == O.ac_encode(cdf[a:b], sym[a:b].astype(np.int16)), (Lp, w)
    # one uniform segment: the same bytes through the one-stream entry point and through the ranges one
    cl = 256
    ub = np.array([min(o, n) for o in range(0, n + cl, cl)], dtype=np.uint32)
    ub = ub[np.concatenate([[True], np.diff(ub) > 0])]
    upay, uoffs = _encode_segments(lib, cdf, sym, ub, dev)
    one = torch.empty(n, dtype=torch.uint8, device=dev)
    assert lib.gpc_chunk_decode_u16(cdf_d.data_ptr(), upay.data_ptr(), uoffs.data_ptr(), n, Lp, cl, one.data_ptr(),
                                    torch.cuda.current_stream(dev).cuda_stream) == 0
    assert np.array_equal(one.cpu().numpy(), _decode_ranges(lib, cdf_d, Lp, upay, uoffs, ub, n, dev))
    assert np.array_equal(one.cpu().numpy(), sym)


def test_ranges_decoder_stays_within_its_rows():
    """a chunk table that runs past n (or backwards) is clamped to rows [0, n): nothing is written beyond them"""
    from gauspcc_b200 import _lib
    from oracle import oracle as O
    lib = _lib.load()
    dev = torch.device("cuda")
    rng = np.random.default_rng(9)
    n, A = 300, 4
    cdf = O.cdf_u16(rng.dirichlet(np.full(A, 0.5), size=n).astype(np.float32))
    sym = rng.integers(0, A, n).astype(np.uint8)
    bounds = np.array([0, 100, 200, 300], dtype=np.uint32)
    payload, offs = _encode_segments(lib, cdf, sym, bounds, dev)
    cdf_d = torch.from_numpy(cdf.view(np.int16)).to(dev)
    guard = 4096
    got = _decode_ranges(lib, cdf_d, A + 1, payload, offs, [0, 100, 200, 300 + 1000], n, dev, guard=guard)
    assert np.array_equal(got[:n], sym) and np.all(got[n:] == 0xAB)
    offs4 = torch.cat([offs, offs[-1:]])
    got = _decode_ranges(lib, cdf_d, A + 1, payload, offs4, [0, 100, 200, 300, 50], n, dev, guard=guard)   # backwards last chunk
    assert np.array_equal(got[:n], sym) and np.all(got[n:] == 0xAB)


# ---------------------------------------------------------------------------------------------------------------- the codec
@pytest.mark.parametrize("chunk", [32, 2048])
def test_bytes_and_decode_match_the_single_path(ckpt, tmp_path, chunk):
    from gauspcc_b200 import bitstream, pcc_utils
    xyzs = _mixed_scenes()
    single = _single(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=chunk)
    paths, res = _batch(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=chunk)
    _same_bytes(single, paths)
    for p in paths:
        with open(p, "rb") as f:
            assert bitstream.split_v2(bitstream.read_file(f.read())[3])[1] == chunk
    assert len({r["batch_enc_time"] for r in res}) == 1 and all(r["num_points"] == x.shape[0] for r, x in zip(res, xyzs))
    bc = pcc_utils._batch(pcc_utils._codec(ckpt, 32, 5))
    assert bc.last_stats["unions"] == 1
    for sorted_output in ((False, True) if chunk == 2048 else (False,)):
        for pre_q in ((True, False) if chunk == 2048 else (True,)):
            _same_rows(paths, ckpt, is_data_pre_quantized=pre_q, sorted_output=sorted_output)
            assert bc.last_stats["unions"] >= 1 and bc.last_stats["stage_round_trips"] == 0
    dec = pcc_utils.decompress_point_clouds(paths, ckpt)
    for x, d in zip(xyzs, dec):                                               # lossless
        x = x.cpu().numpy() if torch.is_tensor(x) else x
        assert np.array_equal(np.unique(d["point_cloud"].cpu().numpy().astype(np.int64), axis=0),
                              np.unique(np.asarray(x, dtype=np.int64), axis=0))


def test_stage_round_trips_and_launches(ckpt, tmp_path):
    """version 1: four host round trips per decoded union level; version 2: none, and fewer launches than the per-scene v2 loop"""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    bc = pcc_utils._batch(codec)
    xyzs = [hac_like_cloud(1500 + 100 * i, seed=50 + i, extent_log2=11) for i in range(8)]
    p1, _ = _batch(xyzs, ckpt, str(tmp_path / "v1"))
    p2, _ = _batch(xyzs, ckpt, str(tmp_path / "v2"), gpu_coder_chunk=2048)
    for paths, per_level in ((p1, 4), (p2, 0)):
        with _counting(bc, "_counts") as calls:                              # once per union level, once more for a union's leaves
            pcc_utils.decompress_point_clouds(paths, ckpt)
        union_levels = len(calls) - bc.last_stats["unions"]
        assert bc.last_stats["unions"] >= 1 and union_levels >= 1
        assert bc.last_stats["stage_round_trips"] == per_level * union_levels, (paths[0], bc.last_stats, union_levels)
    loop = 0
    for p in p2:
        pcc_utils.decompress_point_cloud(p, ckpt)
        loop += codec.last_stats["launches"]
    pcc_utils.decompress_point_clouds(p2, ckpt)
    assert bc.last_stats["launches"] < loop, (bc.last_stats["launches"], loop)


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
        single = _single(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
        paths, _ = _batch(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
        _same_bytes(single, paths)
        _same_rows(paths, ckpt)
        assert pcc_utils._batch(codec).last_stats["unions"] >= 1


def test_kernel_size_3(tmp_path):
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ck3 = save_synthetic_checkpoint(str(tmp_path / "k3" / "w.pt"), kernel_size=3)
    xyzs = [hac_like_cloud(n, seed=20 + n, extent_log2=12) for n in (3000, 800)]
    single = _single(xyzs, ck3, str(tmp_path), kernel_size=3, gpu_coder_chunk=64)
    paths, _ = _batch(xyzs, ck3, str(tmp_path), kernel_size=3, gpu_coder_chunk=64)
    _same_bytes(single, paths)
    _same_rows(paths, ck3, kernel_size=3)


def test_two_unions_singles_and_a_batch_of_one(ckpt, tmp_path):
    from gauspcc_b200 import bitstream, pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    bc = pcc_utils._batch(codec)
    xyzs = [hac_like_cloud(n, seed=30 + i, extent_log2=12) for i, n in enumerate((4000, 3000, 5000, 14000))]
    single = _single(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
    with _attrs(bc, max_rows=5000), _counting(codec, "encode") as alone:
        paths, _ = _batch(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
        assert bc.last_stats["unions"] >= 2 and len(alone) >= 1              # the 14 K scene's finest level exceeds max_rows
    _same_bytes(single, paths)
    est = []                                          # the decoder plans with one row per stream byte
    for p in paths:
        with open(p, "rb") as f:
            est.append(sum(len(x) for x in bitstream.split_v2(bitstream.read_file(f.read())[3])[0]))
    with _attrs(bc, max_rows=sorted(est)[-2] + min(est) // 2), _counting(bc, "_single_decode") as alone:
        dec = pcc_utils.decompress_point_clouds(paths, ckpt)
        assert bc.last_stats["unions"] >= 2 and len(alone) == 1
    for p, d in zip(paths, dec):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"])
    one, _ = _batch(xyzs[:1], ckpt, str(tmp_path / "one"), gpu_coder_chunk=2048)
    _same_bytes(single[:1], one)
    _same_rows(one, ckpt)


def test_files_of_two_chunk_sizes_in_one_call(ckpt, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    xyzs = [hac_like_cloud(n, seed=70 + i, extent_log2=13) for i, n in enumerate((6000, 2500, 9000, 4000))]
    a, _ = _batch(xyzs[:2], ckpt, str(tmp_path / "a"), gpu_coder_chunk=32)
    b, _ = _batch(xyzs[2:], ckpt, str(tmp_path / "b"), gpu_coder_chunk=4096)
    paths = [a[0], b[0], a[1], b[1]]
    _same_rows(paths, ckpt, sorted_output=True)
    bc = pcc_utils._batch(pcc_utils._codec(ckpt, 32, 5))
    assert bc.last_stats["unions"] == 1 and bc.last_stats["stage_round_trips"] == 0


def test_production_size_default_families(ckpt, tmp_path):
    """scenes of 400 K, 250 K and 160 K anchors under the default family thresholds: one union level has members on the sparse and on
    the tcgen05 conv (recorded from BatchCodec._kmaps); files and decoded rows as the single path"""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    codec = pcc_utils._codec(ckpt, 32, 5)
    assert (codec.um_min_rows, codec.sparse_min_rows, codec.sparse_max_density) == (150_000, 150_000, 4.5)
    bc = pcc_utils._batch(codec)
    xyzs = [hac_like_cloud(n, seed=61 + i, extent_log2=16) for i, n in enumerate((400_000, 250_000, 160_000))]
    single = _single(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
    levels = []
    kmaps = bc._kmaps

    def record(lv):
        kms = kmaps(lv)
        levels.append(["um" if k.um_rows else ("sparse" if k.sparse else "v6") for k in kms])
        return kms
    bc._kmaps = record
    try:
        paths, _ = _batch(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
        assert bc.last_stats["unions"] == 1
        assert any("sparse" in f and "um" in f for f in levels), levels
        levels.clear()
        dec = pcc_utils.decompress_point_clouds(paths, ckpt)
        assert bc.last_stats["stage_round_trips"] == 0
        assert any("sparse" in f and "um" in f for f in levels), levels
    finally:
        del bc._kmaps
    _same_bytes(single, paths)
    for p, d in zip(single, dec):
        assert torch.equal(d["point_cloud"], pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"]), p


# ---------------------------------------------------------------------------------------------------------------- rejections
def test_rejections_leave_the_codec_usable(ckpt, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    xyzs = [hac_like_cloud(n, seed=40 + n, extent_log2=12) for n in (3000, 2000, 2500)]
    paths, _ = _batch(xyzs, ckpt, str(tmp_path), gpu_coder_chunk=2048)
    v1, _ = _batch(xyzs[:1], ckpt, str(tmp_path / "v1"))

    def still_good():
        _same_rows(paths, ckpt)

    for bad in (16, 16385):
        with pytest.raises(ValueError, match="32..16384"):
            pcc_utils.compress_point_clouds(xyzs, ckpt, paths, gpu_coder_chunk=bad)
    still_good()
    for mix in ([v1[0], paths[1]], [paths[0], v1[0]]):
        with pytest.raises(ValueError, match="version 2") as e:
            pcc_utils.decompress_point_clouds(mix, ckpt)
        assert mix[1] in str(e.value)
    still_good()

    def count(streams):                                                       # the trailer's voxel count, edited by one
        t = bytearray(streams[-1])
        t[-4:] = (int.from_bytes(t[-4:], "little") + 1).to_bytes(4, "little")
        return streams[:-1] + [bytes(t)]
    bad = _rewrite(paths[1], str(tmp_path / "count.bin"), count)
    with pytest.raises(ValueError, match="trailer") as e:
        pcc_utils.decompress_point_clouds([paths[0], bad, paths[2]], ckpt)
    assert bad in str(e.value)
    still_good()
    # a truncated stream of the finest level: too short for its count header, or counts that do not sum to its length
    for name, cut, what in (("short.bin", lambda s: s[:1], "truncated"), ("half.bin", lambda s: s[:len(s) // 2], "corrupt")):
        bad = _rewrite(paths[1], str(tmp_path / name), lambda st: st[:-2] + [cut(st[-2]), st[-1]])
        with pytest.raises(ValueError, match=f"{what} version-2 stream") as e:
            pcc_utils.decompress_point_clouds([paths[0], bad, paths[2]], ckpt)
        assert bad in str(e.value)
        still_good()
