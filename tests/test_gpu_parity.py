"""GPU parity tests: every stage of the CUDA path (through the C ABI) against the CPU oracle on the
same seeded inputs, the committed golden fixtures, and size-independent properties at full size.

Bars (BASELINE.json north_star): bit-exact order / kernel maps / pyramid / decoded geometry;
probabilities within 1e-3 abs; total bitstream bytes within 0.5 %."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3          # north_star: occupancy probabilities within 1e-3 absolute
SIZE_TOL = 0.005         # north_star: total geometry bitstream size within 0.5 %


@pytest.fixture(scope="module")
def env(weights_np):
    from gauspcc_b200 import _lib
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = make_synthetic_state_dict()
    codec = GausPcgcCodec(DeviceWeights(sd, dev), dev)
    return {"lib": _lib.load(), "codec": codec, "dev": dev, "sd": sd, "w": weights_np}


def _keys_of(codec, xyz_np):
    t = torch.tensor(np.ascontiguousarray(xyz_np, dtype=np.int32), device=codec.dev)
    keys, meta = codec.pack_keys(t)
    return keys, meta.cpu().numpy()


def _unpack(codec, keys):
    from gauspcc_b200.codec import _ptr
    out = torch.empty((keys.shape[0], 3), dtype=torch.int32, device=codec.dev)
    codec._call("gpc_unpack_keys_i32", _ptr(keys), keys.shape[0], _ptr(out), codec._stream())
    return out.cpu().numpy()


# ----------------------------------------------------------------------------- a-2 calculate_morton_order
@pytest.mark.parametrize("n,lo,hi,dtype", [(1, -5, 5, torch.float32), (2, 0, 2, torch.float32), (1000, -300, 300, torch.float32),
                                           (50000, -20000, 20000, torch.float32), (50000, 0, 40, torch.int32),
                                           (4097, -1000000, 1000000, torch.int32), (300000, -30000, 30000, torch.float32)])
def test_calculate_morton_order(env, n, lo, hi, dtype):
    from gauspcc_b200.pcc_utils import calculate_morton_order
    from oracle import oracle as O
    rng = np.random.default_rng(n)
    xyz = rng.integers(lo, hi, size=(n, 3))
    x = torch.tensor(xyz, dtype=dtype, device=env["dev"])
    got = calculate_morton_order(x)
    assert got.dtype == torch.int64 and got.device == x.device and got.shape == (n,)
    assert np.array_equal(got.cpu().numpy(), O.lexorder(xyz))          # duplicates included: stable
    cpu = calculate_morton_order(torch.tensor(xyz, dtype=dtype))       # CPU tensor in -> CPU tensor out
    assert cpu.device.type == "cpu" and np.array_equal(cpu.numpy(), got.cpu().numpy())


def test_calculate_morton_order_golden(env, golden_dir):
    from gauspcc_b200.pcc_utils import calculate_morton_order
    g = np.load(os.path.join(golden_dir, "op_golden.npz"))
    for i in range(3):
        x = torch.tensor(g[f"mo_in{i}"], device=env["dev"])
        assert np.array_equal(calculate_morton_order(x).cpu().numpy(), g[f"mo_out{i}"])   # reference's own output
    with pytest.raises(AssertionError):
        calculate_morton_order(torch.zeros(5, 2, device=env["dev"]))
    assert calculate_morton_order(torch.zeros(0, 3, device=env["dev"])).shape == (0,)


def test_morton_order_full_size_properties(env):
    from gauspcc_b200.pcc_utils import calculate_morton_order
    from gauspcc_b200.synth import hac_like_cloud
    xyz = hac_like_cloud(1_000_000, 0)
    x = torch.tensor(xyz, dtype=torch.float32, device=env["dev"])
    idx = calculate_morton_order(x)
    s = x[idx].to(torch.int64)
    key = (s[:, 2] + (1 << 20)) * (1 << 42) + (s[:, 1] + (1 << 20)) * (1 << 21) + (s[:, 0] + (1 << 20))
    assert bool((key[1:] > key[:-1]).all())                                            # sorted, unique cloud
    assert torch.equal(torch.sort(idx)[0], torch.arange(x.shape[0], device=env["dev"]))  # a permutation
    assert torch.equal(calculate_morton_order(x[idx]), torch.arange(x.shape[0], device=env["dev"]))  # idempotent


# ----------------------------------------------------------------------------- keys / sort / unique
def test_pack_unpack_and_status(env):
    codec = env["codec"]
    rng = np.random.default_rng(1)
    xyz = rng.integers(-(1 << 20) + 16, (1 << 20) - 16, size=(10000, 3)).astype(np.int32)
    keys, meta = _keys_of(codec, xyz)
    assert meta[0] == 0
    assert np.array_equal(_unpack(codec, keys), xyz)
    b = 1 << 20
    assert list(meta[2:8]) == list(xyz.min(0) + b) + list(xyz.max(0) + b)
    k64 = keys.cpu().numpy().astype(np.uint64)
    ref = ((xyz[:, 2].astype(np.int64) + b) << 42) | ((xyz[:, 1].astype(np.int64) + b) << 21) | (xyz[:, 0].astype(np.int64) + b)
    assert np.array_equal(k64, ref.astype(np.uint64))
    _, meta = codec.pack_keys(torch.tensor([[0.5, 1, 2]], dtype=torch.float32, device=codec.dev))
    assert meta.cpu().numpy()[0] & 1
    _, meta = codec.pack_keys(torch.tensor([[1 << 20, 1, 2]], dtype=torch.int32, device=codec.dev))
    assert meta.cpu().numpy()[0] & 2


def test_sort_unique(env):
    codec = env["codec"]
    rng = np.random.default_rng(2)
    xyz = rng.integers(-50, 50, size=(200000, 3)).astype(np.int32)       # many duplicates
    keys, meta = _keys_of(codec, xyz)
    leaf = codec.sort_unique(keys, meta[2:8].astype(np.uint32))
    ref = np.unique(xyz, axis=0)
    ref = ref[np.lexsort((ref[:, 0], ref[:, 1], ref[:, 2]))]
    assert np.array_equal(_unpack(codec, leaf), ref)


# ----------------------------------------------------------------------------- a-4 / a-8 pyramid
@pytest.mark.parametrize("n,seed,ext", [(5000, 0, 16), (60000, 1, 16), (3000, 2, 8), (40, 3, 6), (1, 4, 6)])
def test_pyramid_down_and_expand(env, n, seed, ext):
    from gauspcc_b200.synth import hac_like_cloud
    from oracle import oracle as O
    codec = env["codec"]
    xyz = hac_like_cloud(n, seed, extent_log2=ext) if n > 1 else np.array([[-7, 3, 900]], dtype=np.int32)
    ref_levels = O.build_pyramid(xyz)
    keys, meta = _keys_of(codec, xyz)
    leaf = codec.sort_unique(keys, meta[2:8].astype(np.uint32))
    levels = codec.build_pyramid(leaf, meta[2:8].astype(np.int64))
    assert [l.n for l in levels] == [c.shape[0] for c, _ in ref_levels]
    for lv, (rc, ro) in zip(levels, ref_levels):
        assert np.array_equal(_unpack(codec, lv.keys), rc)
        assert np.array_equal(lv.occ.cpu().numpy(), ro)
    # expansion (FCG + sort_CF) without a sort: children keys and parent rows, bit-exact
    for d, lv in enumerate(levels):
        cc, par = O.fcg(*ref_levels[d])
        ck, cp = codec.expand(lv, cc.shape[0])
        assert np.array_equal(_unpack(codec, ck), cc)
        assert np.array_equal(cp.cpu().numpy().astype(np.int64), par)
        if d + 1 < len(levels):
            assert torch.equal(ck, levels[d + 1].keys)


# ----------------------------------------------------------------------------- kernel maps
@pytest.mark.parametrize("n,seed,ext", [(3000, 0, 7), (40000, 1, 16), (50, 2, 3), (1, 3, 3)])
def test_kernel_map(env, n, seed, ext):
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    codec = env["codec"]
    xyz = uniform_unique_cloud(n, seed, extent_log2=ext) if ext < 10 else hac_like_cloud(n, seed, extent_log2=ext)
    xyz = xyz[O.sort_zyx_perm(xyz)]
    keys, _ = _keys_of(codec, xyz)
    from gauspcc_b200.codec import _ptr
    dense = codec.dense_map(keys)
    ref = O.kmap(xyz, 5)
    assert np.array_equal(dense.cpu().numpy().T, ref)                   # dense map, canonical indexing
    # pair lists: segment (tile, k) lists exactly the rows with a neighbour at k, ascending
    tr = 64
    seg_t, n_pairs, n_real = codec._count_pairs(dense, n, tr, 1)
    nbr_t = torch.empty((max(n_pairs, 1),), dtype=torch.int32, device=codec.dev)
    row_t = torch.empty((max(n_pairs, 1),), dtype=torch.int16, device=codec.dev)
    codec._call("gpc_kmap_pairs_fill", _ptr(dense), n, tr, _ptr(seg_t), _ptr(nbr_t), _ptr(row_t), None, 0, codec._stream())
    seg = seg_t.cpu().numpy().astype(np.int64)
    nbr = nbr_t.cpu().numpy()
    row = row_t.cpu().numpy().astype(np.int64) & 0xFFFF
    assert n_pairs == n_real == int((ref >= 0).sum()) == seg[-1]
    # the conv's own map counts the same pairs
    assert codec.build_kmap(keys).n_real == n_real
    # counts taken from the probes (per (tile, offset) cell) == counts of the map, for tile heights that do / do not divide a block
    for ctile in (256, 384):
        dense2, cells = codec.dense_map(keys, ctile)
        assert torch.equal(dense2, dense)
        tiles = (n + ctile - 1) // ctile
        pad = np.full((tiles * ctile, 125), -1, dtype=ref.dtype)
        pad[:n] = ref
        want = (pad.reshape(tiles, ctile, 125) >= 0).sum(1)
        got = cells.cpu().numpy().reshape(tiles, 126)
        assert np.array_equal(got[:, :125], want) and not got[:, 125].any()
        a, b = codec._scan_um(cells, n, ctile), codec._count_um(dense, n, ctile)
        assert torch.equal(a[0], b[0]) and a[1:] == b[1:] and a[2] == n_real
    for t in range((n + tr - 1) // tr):
        sub = ref[t * tr:(t + 1) * tr]
        for k in (0, 31, 62, 63, 124):
            rr = np.nonzero(sub[:, k] >= 0)[0]
            a, b = seg[t * 126 + k], seg[t * 126 + k + 1]
            assert np.array_equal(row[a:b], rr) and np.array_equal(nbr[a:b], sub[rr, k])


def test_hash_lookup_misses(env):
    from gauspcc_b200.codec import _ptr
    codec = env["codec"]
    xyz = np.array([[0, 0, 0], [1, 0, 0], [-5, 7, 9]], dtype=np.int32)
    keys, _ = _keys_of(codec, xyz)
    cap = codec.lib.gpc_hash_capacity(3)
    table = codec._ws(cap * 16)
    codec._call("gpc_hash_build", _ptr(keys), 3, _ptr(table), cap, codec._stream())
    q, _ = _keys_of(codec, np.array([[1, 0, 0], [2, 0, 0], [-5, 7, 9], [0, 0, 1]], dtype=np.int32))
    rows = torch.empty(4, dtype=torch.int32, device=codec.dev)
    codec._call("gpc_hash_lookup", _ptr(table), cap, _ptr(q), 4, _ptr(rows), codec._stream())
    assert rows.cpu().tolist() == [1, -1, 2, -1]


# ----------------------------------------------------------------------------- sparse conv / head
@pytest.mark.parametrize("n,ext", [(2000, 6), (30000, 16), (700, 4)])
def test_sparse_conv(env, n, ext):
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    codec, w = env["codec"], env["w"]
    xyz = uniform_unique_cloud(n, 5, extent_log2=ext) if ext < 10 else hac_like_cloud(n, 5, extent_log2=ext)
    xyz = xyz[O.sort_zyx_perm(xyz)]
    keys, _ = _keys_of(codec, xyz)
    km = codec.build_kmap(keys)
    ref_km = O.kmap(xyz, 5)
    rng = np.random.default_rng(0)
    x = rng.normal(size=(n, 32)).astype(np.float32)
    res = rng.normal(size=(n, 32)).astype(np.float32)
    xd, rd = torch.tensor(x, device=codec.dev), torch.tensor(res, device=codec.dev)
    Wk = w["target_resnet.2.conv1.kernel"]
    y = codec.conv(xd, 7, km).cpu().numpy()
    ref = O.conv(x, Wk, ref_km)
    scale = np.abs(ref).max()
    assert np.abs(y - ref).max() <= 2e-5 * max(scale, 1.0)
    y2 = codec.conv(xd, 7, km, residual=rd, relu=True).cpu().numpy()
    assert np.abs(y2 - np.maximum(ref + res, 0)).max() <= 2e-5 * max(scale, 1.0)
    # deterministic: bit-identical on a second launch (encoder/decoder CDF identity depends on it)
    assert np.array_equal(codec.conv(xd, 7, km).cpu().numpy(), y)
    # linearity in x
    y3 = codec.conv(2 * xd, 7, km).cpu().numpy()
    assert np.allclose(y3, 2 * y, rtol=1e-6, atol=1e-6)


@pytest.fixture(scope="module")
def env_sparse(env):
    """A codec whose levels ALL run the centre + stragglers conv (spconv_sparse.cu), whatever their size and density."""
    from gauspcc_b200.codec import GausPcgcCodec
    codec = GausPcgcCodec(env["codec"].w, env["dev"])
    codec.sparse_min_rows, codec.sparse_max_density = 1, 1e9
    return dict(env, codec=codec)


@pytest.mark.parametrize("n,ext", [(30000, 16), (20000, 14), (9000, 6), (700, 4), (33, 3)])
def test_sparse_conv_centre_stragglers(env_sparse, n, ext):
    """dense centre product + offset-sorted stragglers against the fp32 oracle conv; several 8192-row blocks, ragged tails,
    rows without any neighbour and rows with many"""
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    codec, w = env_sparse["codec"], env_sparse["w"]
    xyz = uniform_unique_cloud(n, 5, extent_log2=ext) if ext < 10 else hac_like_cloud(n, 5, extent_log2=ext)
    xyz = xyz[O.sort_zyx_perm(xyz)]
    keys, _ = _keys_of(codec, xyz)
    km = codec.build_kmap(keys)
    assert km.sparse
    ref_km = O.kmap(xyz, 5)
    assert km.n_real == int((ref_km >= 0).sum())
    rng = np.random.default_rng(0)
    x = rng.normal(size=(n, 32)).astype(np.float32)
    res = rng.normal(size=(n, 32)).astype(np.float32)
    xd, rd = torch.tensor(x, device=codec.dev), torch.tensor(res, device=codec.dev)
    ref = O.conv(x, w["target_resnet.2.conv1.kernel"], ref_km)
    scale = max(np.abs(ref).max(), 1.0)
    y = codec.conv(xd, 7, km).cpu().numpy()
    assert np.abs(y - ref).max() <= 3e-5 * scale
    y2 = codec.conv(xd, 7, km, residual=rd, relu=True).cpu().numpy()
    assert np.abs(y2 - np.maximum(ref + res, 0)).max() <= 3e-5 * scale
    assert np.array_equal(codec.conv(xd, 7, km).cpu().numpy(), y)            # deterministic


@pytest.mark.parametrize("n,seed,ext", [(20000, 1, 16), (2500, 5, 12)])
def test_codec_sparse_conv_vs_oracle(env_sparse, n, seed, ext):
    """the whole codec with every level on the centre + stragglers conv: same bars as test_codec_vs_oracle"""
    test_codec_vs_oracle(env_sparse, n, seed, ext)


@pytest.fixture(scope="module")
def env_v6d(env):
    """A codec whose levels ALL run the v6d conv (rows straight into the MMA fragments) with 128-row tiles: what the levels
    with >= 150 K rows of a full-size scene take."""
    from gauspcc_b200.codec import GausPcgcCodec
    codec = GausPcgcCodec(env["codec"].w, env["dev"], tile_rows=128)
    codec.v6_variant = 48
    codec.um_min_rows = codec.sparse_min_rows = 1 << 40                     # every level on the mma.sync conv
    codec6 = GausPcgcCodec(env["codec"].w, env["dev"], tile_rows=64)       # v6, one warp per 64-row tile, on every level
    codec6.um_min_rows = codec6.sparse_min_rows = 1 << 40
    return dict(env, codec=codec, codec6=codec6)


@pytest.mark.parametrize("n,ext,tile", [(30000, 16, 128), (30000, 16, 64), (30000, 16, 32), (2000, 6, 128), (700, 4, 128),
                                        (129, 4, 128), (5, 2, 128)])
def test_sparse_conv_v6d(env_v6d, n, ext, tile):
    """v6d against the fp32 oracle conv and, bit for bit, against v6 (same products, same summation order per row); ragged last
    tile, fewer than four 8-pair tiles per warp, entry bulks that end inside the unrolled 8-tile body"""
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    codec, w = env_v6d["codec"], env_v6d["w"]
    codec.tile_rows = tile
    try:
        xyz = uniform_unique_cloud(n, 5, extent_log2=ext) if ext < 10 else hac_like_cloud(n, 5, extent_log2=ext)
        xyz = xyz[O.sort_zyx_perm(xyz)]
        keys, _ = _keys_of(codec, xyz)
        km = codec.build_kmap(keys)
        assert km.tile_rows == tile and not km.sparse
        ref_km = O.kmap(xyz, 5)
        assert km.n_real == int((ref_km >= 0).sum())
        rng = np.random.default_rng(0)
        x = rng.normal(size=(n, 32)).astype(np.float32)
        res = rng.normal(size=(n, 32)).astype(np.float32)
        xd, rd = torch.tensor(x, device=codec.dev), torch.tensor(res, device=codec.dev)
        ref = O.conv(x, w["target_resnet.2.conv1.kernel"], ref_km)
        scale = max(np.abs(ref).max(), 1.0)
        y = codec.conv(xd, 7, km).cpu().numpy()
        assert np.abs(y - ref).max() <= 2e-5 * scale
        y2 = codec.conv(xd, 7, km, residual=rd, relu=True).cpu().numpy()
        assert np.abs(y2 - np.maximum(ref + res, 0)).max() <= 2e-5 * scale
        assert np.array_equal(codec.conv(xd, 7, km).cpu().numpy(), y)            # deterministic
        base = env_v6d["codec6"]
        km6 = base.build_kmap(keys)
        assert km6.v6_variant == 42 and km6.tile_rows == 64
        assert np.array_equal(base.conv(xd, 7, km6).cpu().numpy(), y)            # v6: same sums bit for bit
    finally:
        codec.tile_rows = 128


@pytest.mark.parametrize("n,seed,ext", [(20000, 1, 16), (2500, 5, 12)])
def test_codec_v6d_vs_oracle(env_v6d, n, seed, ext):
    """the whole codec with every level on v6d<128>: same bars as test_codec_vs_oracle"""
    test_codec_vs_oracle(env_v6d, n, seed, ext)


@pytest.fixture(scope="module")
def env_umma(env):
    """A second codec whose levels ALL run the tcgen05 conv (spconv_um.cu, split rows), whatever their size and density."""
    from gauspcc_b200.codec import GausPcgcCodec
    codec = GausPcgcCodec(env["codec"].w, env["dev"])
    codec.um_min_rows, codec.sparse_max_density = 1, 0.0
    return dict(env, codec=codec)


@pytest.mark.parametrize("n,ext,tile", [(30000, 16, 512), (2000, 6, 512), (513, 5, 512), (77, 4, 512), (12000, 5, 512),
                                        (1025, 5, 512), (1024, 5, 512), (512, 5, 512)])
def test_sparse_conv_tcgen05(env_umma, n, ext, tile):
    """tcgen05 / TMEM conv over split rows against the fp32 oracle conv: fp32 and split outputs, residual in both formats, row-range
    launches (decoder wavefront) bit-identical to the whole launch, ragged last tile (down to one row), levels of exactly one and
    two tiles, and a dense level (~40 pairs per row) whose (tile, offset) cells take several 64-pair chunks."""
    from gauspcc_b200.codec import _ptr
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    codec, w = env_umma["codec"], env_umma["w"]
    xyz = uniform_unique_cloud(n, 5, extent_log2=ext) if ext < 10 else hac_like_cloud(n, 5, extent_log2=ext)
    xyz = xyz[O.sort_zyx_perm(xyz)]
    keys, _ = _keys_of(codec, xyz)
    km = codec.build_kmap(keys)
    assert km.um_rows == tile and km.tile_rows == tile
    ref_km = O.kmap(xyz, 5)
    assert km.n_real == int((ref_km >= 0).sum())
    rng = np.random.default_rng(0)
    x = rng.normal(size=(n, 32)).astype(np.float32)
    res = rng.normal(size=(n, 32)).astype(np.float32)
    xd, rd = torch.tensor(x, device=codec.dev), torch.tensor(res, device=codec.dev)
    ref = O.conv(x, w["target_resnet.2.conv1.kernel"], ref_km)
    scale = max(np.abs(ref).max(), 1.0)
    y = codec.conv(xd, 7, km).cpu().numpy()
    assert np.abs(y - ref).max() <= 3e-5 * scale
    # split-row input / output / residual: same numbers up to the 2^-17 relative rounding of a split row
    xs, rs = codec.split_rows(xd), codec.split_rows(rd)
    y2f, y2s = codec.conv(xs, 7, km, residual=rs, relu=True, fmt="both")
    y2 = y2f.cpu().numpy()
    assert np.abs(y2 - np.maximum(ref + res, 0)).max() <= 6e-5 * scale
    joined = torch.empty_like(y2f)
    codec._call("gpc_rows_join", _ptr(y2s), n, _ptr(joined), codec._stream())
    assert np.abs(joined.cpu().numpy() - y2).max() <= 2e-5 * scale
    y3 = codec.conv(xs, 7, km, residual=rd, relu=True).cpu().numpy()          # fp32 residual
    assert np.abs(y3 - y2).max() <= 3e-5 * scale
    # deterministic: bit-identical on a second launch (encoder / decoder CDF identity depends on it)
    assert np.array_equal(codec.conv(xd, 7, km).cpu().numpy(), y)
    # row ranges (whole tiles): the same sums bit for bit
    if n > tile:
        cut = (n // 2) // tile * tile or tile
        yr = torch.full((n, 32), float("nan"), device=codec.dev)
        codec.conv(xs, 7, km, out=yr, rows=(0, cut))
        codec.conv(xs, 7, km, out=yr, rows=(cut, n))
        assert np.array_equal(yr.cpu().numpy(), y)


@pytest.mark.parametrize("n,seed,ext", [(20000, 1, 16), (2500, 5, 12)])
def test_codec_tcgen05_vs_oracle(env_umma, n, seed, ext):
    """the whole codec with every level on the tcgen05 conv: same bars as test_codec_vs_oracle"""
    test_codec_vs_oracle(env_umma, n, seed, ext)


@pytest.mark.parametrize("i", [0, 1, 2, 3])
def test_head_cdf(env, i):
    from gauspcc_b200.codec import _ptr
    from oracle import oracle as O
    codec, w = env["codec"], env["w"]
    A = (2, 2, 4, 16)[i]
    rng = np.random.default_rng(i)
    n = 5003
    f = (rng.normal(size=(n, 32)) * 3).astype(np.float32)
    f[:4] = 0
    f[4:8] = 1e4                     # saturating logits
    fd = torch.tensor(f, device=codec.dev)
    cdf = torch.empty((n, A + 1), dtype=torch.int16, device=codec.dev)
    prob = torch.empty((n, A), dtype=torch.float32, device=codec.dev)
    w1, b1, w2, b2 = codec.w.head[i]
    codec._call("gpc_head_cdf", _ptr(fd), n, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), A, _ptr(cdf), _ptr(prob), codec._stream())
    ref_p = O.head(f, w[f"pred_head_s{i}.0.weight"], w[f"pred_head_s{i}.0.bias"], w[f"pred_head_s{i}.2.weight"],
                   w[f"pred_head_s{i}.2.bias"])
    got_p = prob.cpu().numpy()
    assert np.abs(got_p - ref_p).max() < 1e-5
    got_c = cdf.cpu().numpy().view(np.uint16).astype(np.int64)
    # exact quantisation rule on the kernel's own probabilities (kit/op.py:67-79) ...
    assert np.array_equal(got_c, O.cdf_u16(got_p).astype(np.int64))
    # ... and within one step of the oracle's end-to-end CDF
    ref_c = O.cdf_u16(ref_p).astype(np.int64)
    assert np.abs(got_c[:, :-1] - ref_c[:, :-1]).max() <= 1
    assert (got_c[:, 0] == 0).all() and (np.diff(got_c[:, :-1], axis=1) >= 1).all()      # strictly increasing rows


# ----------------------------------------------------------------------------- full codec
def _encode_file(codec, xyz_t):
    from gauspcc_b200 import bitstream
    bx, bo, streams, aux = codec.encode(xyz_t, collect=True)
    return bitstream.write_file(1, bx, bo, streams), (bx, bo, streams), aux


@pytest.mark.parametrize("n,seed,ext", [(3000, 0, 16), (20000, 1, 16), (2500, 5, 12), (900, 7, 5), (100_000, 0, 16)])
def test_codec_vs_oracle(env, n, seed, ext):
    """(100 000, seed 0) is BASELINE config[0]: the reference's own CPU-runnable case, full codec against the oracle."""
    _check_codec_vs_oracle(env["codec"], env["w"], n, seed, ext)


def _check_codec_vs_oracle(codec, w, n, seed, ext, K=5, oracle=None, prob_tol=PROB_TOL):
    """oracle: (file, collected levels, decoded rows) of the oracle on this cloud and these weights, when already computed (they do
    not depend on the codec's conv families).  Returns dict(aux=the encoder's collected aux, oracle=that triple, worst=the worst
    probability gap, bytes=(file bytes, oracle file bytes))."""
    from gauspcc_b200.synth import hac_like_cloud
    from oracle import oracle as O
    xyz = hac_like_cloud(n, seed, extent_log2=ext)
    x = torch.tensor(xyz, dtype=torch.float32, device=codec.dev)
    blob, (bx, bo, streams), aux = _encode_file(codec, x)
    ref_blob, ref, ref_dec = oracle if oracle is not None else (*O.encode(xyz, w, K=K, collect=True), None)
    # pyramid / base / stream structure bit-exact
    assert np.array_equal(bx, ref["levels"][0][0]) and np.array_equal(bo, ref["levels"][0][1])
    assert len(streams) == 4 * len(ref["aux"])
    for ck, lv in zip(aux["child_keys"], ref["aux"]):
        assert np.array_equal(_unpack(codec, ck), lv["coords"])
    # probabilities of every (level, stage)
    k = 0
    worst = 0.0
    for lv in ref["aux"]:
        for p in lv["probs"]:
            worst = max(worst, float(np.abs(aux["probs"][k].cpu().numpy() - p).max()))
            k += 1
    assert worst <= prob_tol, worst
    # bitstream size
    assert abs(len(blob) - len(ref_blob)) <= max(4, SIZE_TOL * len(ref_blob)), (len(blob), len(ref_blob))
    # lossless round trip, decoded rows in the reference's order (oracle decode of its own file)
    dec = codec.decode(bx, bo, streams).cpu().numpy()
    assert dec.dtype == np.float32
    assert np.array_equal(np.unique(dec.astype(np.int32), axis=0), np.unique(xyz, axis=0))
    if ref_dec is None:
        ref_dec = O.decode(ref_blob, w, K=K)
    assert np.array_equal(dec, ref_dec)
    return dict(aux=aux, oracle=(ref_blob, ref, ref_dec), worst=worst, bytes=(len(blob), len(ref_blob)))


@pytest.mark.parametrize("n,seed,ext", [(20000, 1, 16), (2500, 5, 12)])
def test_codec_kernel_size_3_vs_oracle(env, n, seed, ext):
    """kernel_size = 3 (the reference CLI default, compress_ue_4stage_conv.py:44): the 27 offsets run on the K = 5 kernels; same bars
    against the oracle's K = 3 codec."""
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict, state_dict_to_numpy
    sd3 = make_synthetic_state_dict(kernel_size=3)
    codec3 = GausPcgcCodec(DeviceWeights(sd3, env["dev"], kernel_size=3), env["dev"])
    _check_codec_vs_oracle(codec3, state_dict_to_numpy(sd3), n, seed, ext, K=3)
    um3 = GausPcgcCodec(codec3.w, env["dev"])                                # and with every level on the tcgen05 conv
    um3.um_min_rows, um3.sparse_max_density = 1, 0.0
    _check_codec_vs_oracle(um3, state_dict_to_numpy(sd3), n, seed, ext, K=3)


@pytest.mark.parametrize("name", ["hac600", "blob", "hac2500"])
def test_codec_vs_reference_golden(env, golden_dir, name):
    """Against the fixtures produced by the reference's own driver (tests/golden/make_golden.py)."""
    from gauspcc_b200 import bitstream
    codec = env["codec"]
    cg = np.load(os.path.join(golden_dir, "codec_golden.npz"))
    xyz = cg[f"{name}_xyz"]
    ref_blob = cg[f"{name}_bin"].tobytes()
    blob, (bx, bo, streams), aux = _encode_file(codec, torch.tensor(xyz, dtype=torch.int32, device=codec.dev))
    _, rbx, rbo, rstreams = bitstream.read_file(ref_blob)
    assert np.array_equal(bx, rbx) and np.array_equal(bo, rbo) and len(streams) == len(rstreams)
    assert abs(len(blob) - len(ref_blob)) <= max(4, SIZE_TOL * len(ref_blob))
    if f"{name}_probs" in cg:
        got = np.concatenate([p.cpu().numpy().reshape(-1) for p in aux["probs"]])
        assert np.abs(got - cg[f"{name}_probs"]).max() <= PROB_TOL
    dec = codec.decode(bx, bo, streams).cpu().numpy()
    assert np.array_equal(dec, cg[f"{name}_decoded"])                    # same rows, same order as the reference run


def test_codec_vs_reference_golden_60k(env, golden_dir):
    """The 60 K-anchor fixture of the reference's own driver (make_golden.py section 3) against the CUDA codec: base level, stream
    sizes within 0.5 %, every 128th row of every probability tensor within 1e-3, decoded rows identical in the reference's order."""
    import hashlib
    from gauspcc_b200.synth import hac_like_cloud
    codec = env["codec"]
    g = np.load(os.path.join(golden_dir, "codec_golden_60k.npz"))
    xyz = hac_like_cloud(int(g["n"][0]), int(g["seed"][0]))
    assert hashlib.sha256(np.ascontiguousarray(xyz.astype(np.int32)).tobytes()).digest() == g["xyz_sha256"].tobytes()
    blob, (bx, bo, streams), aux = _encode_file(codec, torch.tensor(xyz, dtype=torch.int32, device=codec.dev))
    assert np.array_equal(bx, g["base_xyz"]) and np.array_equal(bo, g["base_occ"]) and len(streams) == len(g["stream_lens"])
    assert abs(len(blob) - int(g["file_bytes"][0])) <= SIZE_TOL * int(g["file_bytes"][0])
    assert all(abs(len(a) - int(b)) <= max(4, SIZE_TOL * int(b)) for a, b in zip(streams, g["stream_lens"]))
    every = int(g["probs_every"][0])
    assert [p.shape[0] for p in aux["probs"]] == list(g["nprob"])
    got = np.concatenate([p[::every].cpu().numpy().reshape(-1) for p in aux["probs"]])
    assert np.abs(got - g["probs"]).max() <= PROB_TOL
    dec = codec.decode(bx, bo, streams).cpu().numpy()
    assert hashlib.sha256(np.ascontiguousarray(dec.astype(np.int32)).tobytes()).digest() == g["decoded_sha256"].tobytes()


def test_edge_cases(env):
    codec = env["codec"]
    dev = codec.dev
    rng = np.random.default_rng(9)
    cases = [np.array([[5, -7, 9]], dtype=np.int32),                                   # single voxel
             rng.integers(-40, 40, size=(40, 3)).astype(np.int32),                     # < 64: base level only
             np.repeat(rng.integers(-400, 400, size=(500, 3)).astype(np.int32), 3, 0),  # duplicates merge
             np.array([[-(1 << 20) + 16, 0, (1 << 20) - 16], [0, 0, 0]], dtype=np.int32)]  # extreme coordinates
    for xyz in cases:
        bx, bo, streams, _ = codec.encode(torch.tensor(xyz, device=dev))
        dec = codec.decode(bx, bo, streams).cpu().numpy().astype(np.int32)
        assert np.array_equal(np.unique(dec, axis=0), np.unique(xyz, axis=0))
    with pytest.raises(ValueError):
        codec.encode(torch.tensor([[0.25, 0, 0]], dtype=torch.float32, device=dev))
    with pytest.raises(ValueError):                                                    # extent beyond the key fields
        codec.encode(torch.tensor([[0, 0, 0], [1 << 21, 0, 0]], dtype=torch.int32, device=dev))
    with pytest.raises(ValueError):
        codec.decode(np.zeros((1, 3), np.int32), np.array([1], np.uint8), [b"", b"", b""])


def test_far_from_origin_vs_oracle(env, weights_np):
    """Coordinates outside the 21-bit key fields (|c| > 2^20 - 16): the scene is coded translated by a multiple of 2^levels and the
    base level written back in the caller's coordinates, so file and decoded rows are those of the oracle (reference arithmetic on
    int32 coordinates, no range limit) -- for float and int input, default and sorted row order, and a single far voxel."""
    from gauspcc_b200 import bitstream
    from gauspcc_b200.synth import hac_like_cloud
    from oracle import oracle as O
    codec = env["codec"]
    off = np.array([3_000_000, -5_000_000, 7_000_123], dtype=np.int32)
    for xyz in (hac_like_cloud(6000, 2, extent_log2=13) + off, np.array([[1 << 20, 0, -(1 << 22)]], dtype=np.int32)):
        ref = O.encode(xyz, weights_np)
        for dt in (torch.int32, torch.float32):
            blob, (bx, bo, streams), _ = _encode_file(codec, torch.tensor(xyz, dtype=dt, device=codec.dev))
            _, rbx, rbo, rst = bitstream.read_file(ref)
            assert np.array_equal(bx, rbx) and np.array_equal(bo, rbo) and len(streams) == len(rst)
            assert abs(len(blob) - len(ref)) <= max(4, SIZE_TOL * len(ref))
            dec = codec.decode(bx, bo, streams).cpu().numpy()
            assert np.array_equal(dec, O.decode(ref, weights_np))
            srt = codec.decode(bx, bo, streams, sorted_rows=True).cpu().numpy().astype(np.int64)
            assert np.array_equal(srt, xyz[np.lexsort((xyz[:, 0], xyz[:, 1], xyz[:, 2]))])
        scaled = codec.decode(bx, bo, streams, scale=0.5).cpu().numpy()
        assert np.array_equal(scaled, dec * np.float32(0.5))


def test_container_v2_gpu_chunk_coder(env, tmp_path):
    """SURVEY 8f-3, opt-in container version 2: the occupancy streams coded on the GPU in chunks (csrc/attr_ac.cu on the codec's own
    CDF rows).  Every chunk is the range coder's stream of its symbols under the encoder's CDF rows (bit-exact against the oracle
    coder), the file round-trips to the same rows as the drop-in file, costs < 1.5 % more bytes, and names its own format."""
    from gauspcc_b200 import bitstream, pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    from oracle import oracle as O
    codec = env["codec"]
    xyz = hac_like_cloud(40000, 6)
    x = torch.tensor(xyz, dtype=torch.int32, device=codec.dev)
    chunk = 512
    bx, bo, streams, aux = codec.encode(x, collect=True, gpu_chunk=chunk)
    bx1, bo1, streams1, _ = codec.encode(x)
    assert np.array_equal(bx, bx1) and np.array_equal(bo, bo1) and len(streams) == len(streams1)
    levels = aux["levels"]
    for k in (len(streams) - 1, len(streams) - 2, len(streams) - 6, 3):                 # a few (level, stage) streams, all chunks
        d, i = divmod(k, 4)
        occ = levels[d + 1].occ.cpu().numpy()
        sym = O.split_symbols(occ)[i].astype(np.int16)
        cdf = aux["cdfs"][k].cpu().numpy().view(np.uint16)
        n = sym.shape[0]
        cl = codec.chunk_len(n, chunk)                                                    # short streams take shorter chunks
        assert cl == max(1, min(chunk, max(64, (n + 63) // 64)))
        chunks = (n + cl - 1) // cl
        cnt = np.frombuffer(streams[k], dtype="<u2", count=chunks).astype(np.int64)
        body = streams[k][2 * chunks:]
        assert cnt.sum() == len(body)
        pos = 0
        for c in range(chunks):
            want = O.ac_encode(cdf[c * cl:(c + 1) * cl], sym[c * cl:(c + 1) * cl])
            assert body[pos:pos + cnt[c]] == want, (k, c)
            pos += cnt[c]
    dec = codec.decode(bx, bo, streams, gpu_chunk=chunk)
    assert torch.equal(dec, codec.decode(bx1, bo1, streams1))
    # through the public API: the file says what it is; the default stays the reference bitstream
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    xs = x[pcc_utils.calculate_morton_order(x)].float()
    r1 = pcc_utils.compress_point_cloud(xs, ckpt, str(tmp_path / "v1" / "xyz_pcc.bin"))
    r2 = pcc_utils.compress_point_cloud(xs, ckpt, str(tmp_path / "v2" / "xyz_pcc.bin"), gpu_coder_chunk=2048)
    assert r1["file_size_bits"] < r2["file_size_bits"] < 1.015 * r1["file_size_bits"]
    d1 = pcc_utils.decompress_point_cloud(r1["output_path"], ckpt)
    d2 = pcc_utils.decompress_point_cloud(r2["output_path"], ckpt)
    assert torch.equal(d1["point_cloud"], d2["point_cloud"])
    _, _, _, st2 = bitstream.read_file(open(r2["output_path"], "rb").read())
    assert bitstream.split_v2(st2)[1:] == (2048, 40000) and bitstream.split_v2(bitstream.read_file(open(r1["output_path"], "rb").read())[3])[1] == 0
    # the trailer's voxel count is an integrity check: a file whose streams decode to another count raises
    blob2 = bytearray(open(r2["output_path"], "rb").read())
    blob2[-4:] = (39999).to_bytes(4, "little")
    open(str(tmp_path / "v2" / "bad.bin"), "wb").write(bytes(blob2))
    with pytest.raises(ValueError):
        pcc_utils.decompress_point_cloud(str(tmp_path / "v2" / "bad.bin"), ckpt)
    with pytest.raises(ValueError):
        pcc_utils.compress_point_cloud(xs, ckpt, str(tmp_path / "bad" / "xyz_pcc.bin"), gpu_coder_chunk=100000)
    with pytest.raises(ValueError):                                                       # a truncated version-2 stream is an error, not a hang
        codec.decode(bx, bo, [s[:1] for s in streams], gpu_chunk=chunk)
    # sizes around the chunk boundaries and clouds without coded levels
    rng = np.random.default_rng(4)
    for pts in (np.array([[5, -7, 9]], dtype=np.int32), rng.integers(-40, 40, size=(40, 3)).astype(np.int32),
                hac_like_cloud(3000, 1, extent_log2=10), hac_like_cloud(chunk * 9 + 1, 2, extent_log2=12)):
        for ck in (32, chunk):
            b3, o3, s3, _ = codec.encode(torch.tensor(pts, device=codec.dev), gpu_chunk=ck)
            got = codec.decode(b3, o3, s3, gpu_chunk=ck).cpu().numpy().astype(np.int32)
            assert np.array_equal(np.unique(got, axis=0), np.unique(pts, axis=0))


def test_scene_as_morton_blocks(env, tmp_path):
    """One scene cut into Morton-ordered spatial blocks (shard.compress_point_cloud_blocks), coded as if by two ranks: every block is
    an ordinary xyz_pcc.bin, the blocks concatenated by index are the scene in calculate_morton_order order, few per cent more bits."""
    from gauspcc_b200 import pcc_utils, shard
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    x = torch.tensor(hac_like_cloud(60000, 8), dtype=torch.float32, device=env["dev"])
    x = x[pcc_utils.calculate_morton_order(x)]
    binp = str(tmp_path / "scene" / "xyz_pcc.bin")
    whole = pcc_utils.compress_point_cloud(x, ckpt, binp)
    enc = [shard.compress_point_cloud_blocks(x, ckpt, binp, 3, rank, 2) for rank in (0, 1)]
    assert sorted(b for e in enc for b, *_ in e["blocks"]) == [0, 1, 2] and sum(r for e in enc for _, r, *_ in e["blocks"]) == 60000
    dec = {}
    for rank in (0, 1):
        dec.update(shard.decompress_point_cloud_blocks(binp, ckpt, 3, rank, 2)["blocks"])
    assert torch.equal(torch.cat([dec[b] for b in range(3)]), x)
    bits = sum(e["file_size_bits"] for e in enc)
    assert bits == 8 * sum(os.path.getsize(shard.block_path(binp, b)) for b in range(3))
    assert whole["file_size_bits"] < bits < 1.05 * whole["file_size_bits"]
    # a block file is an ordinary file of the drop-in format
    d1 = pcc_utils.decompress_point_cloud(shard.block_path(binp, 1), ckpt)
    assert d1["num_points"] == 20000


def test_pcc_utils_api(env, tmp_path):
    """The drop-in boundary: same call pattern as HAC's conduct_encoding/conduct_decoding
    (scene/gaussian_model.py:1106-1121, 1248-1257)."""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    voxel = 0.001
    xyz = hac_like_cloud(30000, 4)
    anchor = torch.tensor(xyz, dtype=torch.float32, device=env["dev"]) * voxel
    anchor_int = torch.round(anchor / voxel)
    before = anchor_int.clone()
    order = pcc_utils.calculate_morton_order(anchor_int)
    anchor_int = anchor_int[order]
    out = pcc_utils.compress_point_cloud(anchor_int, ckpt, str(tmp_path / "bits" / "xyz_pcc.bin"))
    assert set(out) >= {"bpp", "enc_time", "file_size_bits", "num_points", "output_path"}
    assert out["num_points"] == 30000 and out["file_size_bits"] == 8 * os.path.getsize(out["output_path"])
    assert abs(out["bpp"] - out["file_size_bits"] / 30000) < 1e-9 and out["enc_time"] > 0
    assert torch.equal(before[order], anchor_int)                         # input not mutated
    dec = pcc_utils.decompress_point_cloud(out["output_path"], ckpt)
    assert set(dec) >= {"dec_time", "num_points", "point_cloud", "output_path"}
    pc = dec["point_cloud"]
    assert pc.dtype == torch.float32 and pc.is_cuda and dec["num_points"] == 30000
    order2 = pcc_utils.calculate_morton_order(pc)
    assert torch.equal(pc[order2], anchor_int)                            # HAC re-sorts and gets the encoder's order back
    # numpy input + posQ, is_data_pre_quantized=False mapping
    out2 = pcc_utils.compress_point_cloud(xyz[:5000], ckpt, str(tmp_path / "b2" / "x.bin"))
    d2 = pcc_utils.decompress_point_cloud(out2["output_path"], ckpt, is_data_pre_quantized=False)
    want = (torch.tensor(xyz[:5000], dtype=torch.float32) - 131072) * 0.001       # pcc_utils.py:381
    got = d2["point_cloud"].cpu()
    key = lambda t: t[np.lexsort((t[:, 0].numpy(), t[:, 1].numpy(), t[:, 2].numpy()))]
    assert torch.equal(key(got), key(want))
    with pytest.raises(FileNotFoundError):
        pcc_utils.compress_point_cloud(xyz[:100], str(tmp_path / "nope.pt"), str(tmp_path / "b3" / "x.bin"))
    bad = str(tmp_path / "bad.pt")
    torch.save({"prior_embedding.weight": torch.zeros(256, 32)}, bad)
    with pytest.raises(RuntimeError):
        pcc_utils.compress_point_cloud(xyz[:100], bad, str(tmp_path / "b4" / "x.bin"))


def test_sorted_output_is_morton_order(env, tmp_path):
    """SURVEY 8f-1: decompress_point_cloud(sorted_output=True) hands the rows back in calculate_morton_order order, so the re-sort
    at HAC/scene/gaussian_model.py:1253-1255 is the identity."""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    xyz = hac_like_cloud(30000, 3)
    x = torch.tensor(xyz, dtype=torch.float32, device=env["dev"])
    binp = str(tmp_path / "out" / "xyz_pcc.bin")
    pcc_utils.compress_point_cloud(x, ckpt, binp)
    ref_order = pcc_utils.decompress_point_cloud(binp, ckpt)["point_cloud"]
    srt = pcc_utils.decompress_point_cloud(binp, ckpt, sorted_output=True)["point_cloud"]
    perm = pcc_utils.calculate_morton_order(srt)
    assert torch.equal(perm, torch.arange(srt.shape[0], device=perm.device))
    assert torch.equal(srt, ref_order[pcc_utils.calculate_morton_order(ref_order)])
    assert np.array_equal(np.unique(srt.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz, axis=0))


def test_cli_file_roundtrip(env, tmp_path):
    """SURVEY 8f-2: the stand-alone compress / decompress tools over files, metric coordinates and posQ (lossless on the voxel set)."""
    from gauspcc_b200 import cli
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    rng = np.random.default_rng(4)
    src = tmp_path / "in"
    src.mkdir()
    pts = (rng.normal(size=(20000, 3)) * np.array([8.0, 8.0, 1.0])).astype(np.float32)         # metres, KITTI-like
    np.concatenate([pts, np.ones((20000, 1), np.float32)], axis=1).tofile(src / "000001.bin")
    np.save(src / "000002.npy", pts[:5000].astype(np.float64) * 0.5)
    rows = cli.compress_files(str(src), str(tmp_path / "cmp"), ckpt, posQ=16, resultdir=str(tmp_path / "res"))
    assert [r["filedir"] for r in rows] == ["000001.bin", "000002.npy"] and all(r["bpp"] > 0 for r in rows)
    assert os.path.exists(tmp_path / "res" / "ue_4stage_conv_data2.csv")
    drows = cli.decompress_files(str(tmp_path / "cmp"), str(tmp_path / "dec"), ckpt)
    assert [r["filedir"] for r in drows] == ["000001.bin.bin", "000002.npy.bin"]
    for name, p in (("000001.bin", pts.astype(np.float64)), ("000002.npy", pts[:5000].astype(np.float64) * 0.5)):
        q = np.unique(cli.quantise(p, 16, False).numpy(), axis=0)
        dec = cli.read_points(str(tmp_path / "dec" / (name + ".bin.ply")))
        back = np.unique(np.round((dec / 0.001 + 131072) / 16).astype(np.int32), axis=0)          # undo decompress_ue_4stage_conv.py:176-179
        assert drows[0]["num_points"] > 0 and np.array_equal(back, q)


@pytest.mark.parametrize("scenes", [((120_000, 3), (30_000, 4)), ((30_000, 4), (120_000, 3))], ids=["shrinking", "growing"])
@pytest.mark.parametrize("kind", ["um", "v6d", "sparse"])
def test_decoder_wavefront(env, env_v6d, env_sparse, env_umma, kind, scenes):
    """The decoder's stage wavefront (chunks of rows, four range-decoder threads) against the stage-by-stage decode of the same
    streams: identical geometry row for row; levels of every chunk count (ragged last chunk, levels too small for two chunks fall
    back).  All three conv families of the big levels.  Two scenes on one codec, in both orders: the buffers the codec keeps
    across calls (wavefront feature arrays, pinned staging) are reused by a smaller scene and grown for a bigger one."""
    from gauspcc_b200.codec import GausPcgcCodec
    from gauspcc_b200.synth import hac_like_cloud
    src = {"v6d": env_v6d, "sparse": env_sparse, "um": env_umma}[kind]["codec"]
    codec = GausPcgcCodec(src.w, env["dev"], tile_rows=128 if kind == "v6d" else None)
    codec.v6_variant, codec.um_min_rows = src.v6_variant, src.um_min_rows
    codec.sparse_min_rows, codec.sparse_max_density = src.sparse_min_rows, src.sparse_max_density
    codec.wave_min_rows, codec.wave_chunk_rows = 1, 8192
    if kind == "sparse":
        codec.wave_chunk_rows = 16384
    for n, seed in scenes:
        x = torch.tensor(hac_like_cloud(n, seed), dtype=torch.float32, device=codec.dev)
        bx, bo, streams, _ = codec.encode(x)
        codec.wave_decode = True
        seen = []
        orig = codec._decode_level_wavefront
        codec._decode_level_wavefront = lambda *a, **k: (seen.append(a[2]), orig(*a, **k))[1]
        try:
            d_wave = codec.decode(bx, bo, streams)
        finally:
            codec._decode_level_wavefront = orig
        codec.wave_decode = False
        d_ref = codec.decode(bx, bo, streams)
        assert torch.equal(d_wave, d_ref)
        if n >= 100_000:
            assert len(seen) >= 2 and max(seen) > 4 * 8192, seen          # the big levels did take the wavefront
    # a corrupt stream must surface as an error or as wrong geometry, never as a hang
    bad = list(streams)
    bad[-1] = bad[-1][: len(bad[-1]) // 2]
    codec.wave_decode = True
    codec.decode(bx, bo, bad)


def test_full_size_roundtrip_1m(env):
    """BASELINE config 2 size: lossless round trip, encoder == decoder CDFs (else the range decoder
    desynchronises and the geometry is garbage), teacher-forced decode == real decode."""
    from gauspcc_b200.synth import hac_like_cloud
    codec = env["codec"]
    xyz = hac_like_cloud(1_000_000, 0)
    x = torch.tensor(xyz, dtype=torch.float32, device=codec.dev)
    bx, bo, streams, aux = codec.encode(x, collect=False)
    dec = codec.decode(bx, bo, streams)
    a = dec.to(torch.int64)
    key = (a[:, 2] + (1 << 20)) * (1 << 42) + (a[:, 1] + (1 << 20)) * (1 << 21) + (a[:, 0] + (1 << 20))
    b = x.to(torch.int64)
    keyb = (b[:, 2] + (1 << 20)) * (1 << 42) + (b[:, 1] + (1 << 20)) * (1 << 21) + (b[:, 0] + (1 << 20))
    assert torch.equal(torch.sort(key)[0], torch.sort(keyb)[0])
    bits = 8 * sum(len(s) for s in streams)
    assert 0 < bits / 1e6 < 200


def test_full_size_1m_vs_oracle(env):
    """BASELINE config[1] at full size against the oracle's encode of the SAME cloud (one-off ~30 s of CPU): base level and stream
    structure identical, total bytes within 0.5 %, probabilities of the two largest levels within 1e-3, and the CDF rows the
    decoder computes on those levels bit-identical to the encoder's (a single differing uint16 desynchronises the range coder)."""
    from gauspcc_b200 import bitstream
    from gauspcc_b200.synth import hac_like_cloud
    from oracle import oracle as O
    codec, w = env["codec"], env["w"]
    xyz = hac_like_cloud(1_000_000, 0)
    x = torch.tensor(xyz, dtype=torch.float32, device=codec.dev)
    bx, bo, streams, aux = codec.encode(x, collect=True)
    blob = bitstream.write_file(1, bx, bo, streams)
    ref_blob, ref = O.encode(xyz, w, collect=True)
    assert np.array_equal(bx, ref["levels"][0][0]) and np.array_equal(bo, ref["levels"][0][1])
    assert len(streams) == 4 * len(ref["aux"])
    assert abs(len(blob) - len(ref_blob)) <= SIZE_TOL * len(ref_blob), (len(blob), len(ref_blob))
    L = len(ref["aux"])
    big = sorted(range(L), key=lambda d: -ref["aux"][d]["coords"].shape[0])[:2]
    for d in big:
        assert np.array_equal(_unpack(codec, aux["child_keys"][d]), ref["aux"][d]["coords"])
        for i in range(4):
            got = aux["probs"][4 * d + i].cpu().numpy()
            assert np.abs(got - ref["aux"][d]["probs"][i]).max() <= PROB_TOL
    # decoder CDFs == encoder CDFs, bit for bit (stage-by-stage decode exposes them; the wavefront runs the same kernels)
    codec.wave_decode = False
    codec.debug_dec_cdfs = {}
    try:
        dec = codec.decode(bx, bo, streams)
        for d in big:
            for i in range(4):
                assert torch.equal(codec.debug_dec_cdfs[(d, i)], aux["cdfs"][4 * d + i]), (d, i)
    finally:
        codec.wave_decode = True
        codec.debug_dec_cdfs = None
    assert np.array_equal(np.unique(dec.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz, axis=0))


def test_full_size_roundtrip_3m(env, tmp_path):
    """BASELINE config[3]: a 3M-anchor Mip-NeRF360-scale scene through the drop-in API (HAC's call sequence), lossless."""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import save_synthetic_checkpoint
    ckpt = save_synthetic_checkpoint(str(tmp_path / "GausPcgc" / "best_model_ue_4stage_conv.pt"))
    xyz = hac_like_cloud(3_000_000, 0, extent_log2=17)
    a = torch.tensor(xyz, dtype=torch.float32, device=env["dev"])
    a = a[pcc_utils.calculate_morton_order(a)]
    out = pcc_utils.compress_point_cloud(a, ckpt, str(tmp_path / "bits" / "xyz_pcc.bin"))
    dec = pcc_utils.decompress_point_cloud(out["output_path"], ckpt)["point_cloud"]
    assert dec.shape[0] == 3_000_000
    assert torch.equal(dec[pcc_utils.calculate_morton_order(dec)], a)          # HAC's re-sort gives the encoder's order back
    assert 0 < out["bpp"] < 200
