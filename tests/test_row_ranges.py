"""Row-range pair streams and convs (a batch of scenes coded as one union level, gauspcc_b200/batch.py) and the row-restricted convs
of the decoder wavefront, against numpy restatements of the stream layouts of include/gpcgc.h, the whole-level launches and an fp64
reference conv.

What the C ABI promises for a row range [row0, row1) of a level of n_level rows:
  * the pair streams are exactly those of the range's rows coded as a level of their own, with neighbour indices + row0;
  * a range conv writes the rows [row0, row1) and nothing else, and reads only the neighbours of those rows;
  * every row is summed in one fixed order (offsets ascending), so a range conv equals the whole-level launch of the same family and
    tiling bit for bit, and a scene of a union equals the scene coded alone.

The references and the stream layouts run on the CPU; the kernels are called through the C ABI (codec._call), so that every
(variant, tile_rows) is reachable whatever the codec's family thresholds."""
import numpy as np
import pytest

try:
    import torch
except ImportError:                                           # the CPU references below do not need it
    torch = None

GPC_EINVAL = -1
SP_TB = 8192                                                  # rows per block of the sparse map (spconv_sparse.cu)
CENTRE = 62
WIDX = 7                                                      # the conv whose weights the tests use (target_resnet.2.conv1)

# ------------------------------------------------------------------------------------------------------------ fp64 reference
# Error bound of the three-term bf16 split used by every conv family (mma.sync, sparse, tcgen05): x = xh + xl and W = Wh + Wl with
# bf16 round-to-nearest halves, and the kernels sum Wh.xh + Wh.xl + Wl.xh in fp32.
#   * xh is x to 8 mantissa bits (|x - xh| <= 2^-9 |x|), xl rounds the remainder to 8 bits again: |x - xh - xl| <= 2^-18 |x|,
#     the same for W: the two representation errors cost <= 2^-17 |W| |x| per product;
#   * the dropped Wl.xl term is <= 2^-9 * 2^-9 = 2^-18 |W| |x|;
#   * fp32 accumulation: the products of one pair are summed inside the MMA, the offsets of a row (<= 125) and the residual in fp32
#     registers / shared memory; with u = 2^-24 and a few hundred additions that is well below 2^-16 of the sum of magnitudes in
#     practice (a random-walk bound; the worst case of 160 additions in a row would be 2^-16.7).
# Together 0.75 * 2^-16 + accumulation, per element, relative to absref = sum |W| |x| (+ |residual|): c = 2.  Keeping only two of
# the three terms (Wh.xh + Wh.xl) leaves an error of ~2^-9 |W| |x| per product, which this bound catches by a wide margin
# (test_two_term_split_exceeds_the_bound).
BOUND_C = 2.0
BOUND_TINY = 1e-30


def conv64(x, W, km, residual=None, relu=False):
    """y = act(sum_k W[k]^T x[nbr_k(o)] + residual) in float64, and absref = sum_k |W[k]|^T |x[nbr_k(o)]| (+ |residual|).
    km: dense map [n, 125] (oracle.kmap layout, -1 = absent)."""
    n = km.shape[0]
    x64, W64 = np.asarray(x, np.float64), np.asarray(W, np.float64)
    y = np.zeros((n, W64.shape[2]))
    absref = np.zeros_like(y)
    for k in range(km.shape[1]):
        idx = km[:, k]
        m = idx >= 0
        if m.any():
            xi = x64[idx[m]]
            y[m] += xi @ W64[k]
            absref[m] += np.abs(xi) @ np.abs(W64[k])
    if residual is not None:
        y += residual
        absref += np.abs(np.asarray(residual, np.float64))
    if relu:
        y = np.maximum(y, 0.0)                                # 1-Lipschitz: the bound carries over
    return y, absref


def bound(absref):
    return BOUND_C * 2.0 ** -16 * absref + BOUND_TINY


def err_ratio(y, ref, absref):
    """worst |y - ref| / absref of the rows given"""
    return float((np.abs(np.asarray(y, np.float64) - ref) / np.maximum(absref, BOUND_TINY)).max(initial=0.0))


def bf16(a):
    """round to bf16 (nearest, ties to even), as float32"""
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def emulate_split_conv(x, W, km, terms):
    """the kernels' arithmetic in numpy: per offset the split products (3 terms: Wh.xh + Wh.xl + Wl.xh; 2 terms: without Wl.xh)
    rounded to fp32, offsets added in ascending order in fp32"""
    x = np.asarray(x, np.float32)
    xh, Wh = bf16(x), bf16(W)
    xl, Wl = bf16(x - xh), bf16(W - Wh)
    y = np.zeros((km.shape[0], W.shape[2]), np.float32)
    for k in range(km.shape[1]):
        idx = km[:, k]
        m = idx >= 0
        if m.any():
            p = xh[idx[m]].astype(np.float64) @ Wh[k] + xl[idx[m]].astype(np.float64) @ Wh[k]
            if terms == 3:
                p += xh[idx[m]].astype(np.float64) @ Wl[k]
            y[m] = y[m] + p.astype(np.float32)
    return y


# ------------------------------------------------------------------------------------------------------------ stream layouts
# Pure functions of the dense map km [n_level, 125] and (row0, row1), restated from include/gpcgc.h, kmap.cu and spconv_sparse.cu.
ALL64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _cells(sub, T, ncol):
    """rows of sub in tiles of T: (cube [tiles, ncol, T] of neighbour rows, -1 = absent / past the end)"""
    n = sub.shape[0]
    tiles = (n + T - 1) // T
    full = np.full((tiles * T, ncol), -1, np.int64)
    full[:n] = sub
    return full.reshape(tiles, T, ncol).transpose(0, 2, 1)


def _stream(cube, pad, pad_slot):
    """seg (exclusive scan of the per-(tile, offset) counts rounded up to `pad`, one zero pad slot per tile when pad_slot) and the
    (tile, offset, row) of every true pair with its stream position; rows ascending inside a cell"""
    valid = cube >= 0
    raw = valid.sum(2)
    padded = (raw + pad - 1) // pad * pad
    if pad_slot:
        padded = np.concatenate([padded, np.zeros((padded.shape[0], 1), np.int64)], axis=1)
    seg = np.concatenate([[0], np.cumsum(padded.ravel())]).astype(np.int64)
    t, k, r = np.nonzero(valid)                              # lexicographic: (tile, offset, row)
    raw_start = np.concatenate([[0], np.cumsum(raw.ravel())])[:-1]
    cell = t * raw.shape[1] + k
    q = seg[t * padded.shape[1] + k] + (np.arange(t.size) - raw_start[cell])
    return seg, t, k, r, q, int(valid.sum())


def ref_pairs_stream(km, row0, row1, tile_rows, pad=8):
    """mma.sync conv (gpc_kmap_pairs_count_range / _fill_range): seg u32[tiles * 126 + 1], pairs u64 = nbr | row_in_tile << 32 |
    k << 48 (padding all ones), totals {entries, true pairs}"""
    cube = _cells(km[row0:row1], tile_rows, 125)
    seg, t, k, r, q, n_real = _stream(cube, pad, True)
    pairs = np.full(int(seg[-1]), ALL64, np.uint64)
    pairs[q] = cube[t, k, r].astype(np.uint64) | (r.astype(np.uint64) << np.uint64(32)) | (k.astype(np.uint64) << np.uint64(48))
    return seg.astype(np.uint32), pairs, (int(seg[-1]), n_real)


def ref_um_stream(km, row0, row1, tile_rows=512):
    """tcgen05 conv (gpc_kmap_um_count_range / _fill_range): cells padded to 16, pair_nbr (padding 0xFFFFFFFF), pair_off = row * 128
    (padding: the dummy row tile_rows * 128), totals u64 {entries, true pairs}"""
    cube = _cells(km[row0:row1], tile_rows, 125)
    seg, t, k, r, q, n_real = _stream(cube, 16, True)
    nbr = np.full(int(seg[-1]), 0xFFFFFFFF, np.uint32)
    off = np.full(int(seg[-1]), tile_rows * 128, np.uint32)
    nbr[q] = cube[t, k, r]
    off[q] = r * 128
    return seg.astype(np.uint32), nbr, off, (int(seg[-1]), n_real)


SP_OFFSETS = np.array([k for k in range(125) if k != CENTRE])


def ref_sparse_stream(km, row0, row1):
    """sparse map (gpc_kmap_sparse_count_range / _fill_range): per (8192-row block, non-centre offset kk) a segment padded to 8 (slot
    124 of a block: empty), pairs u64 = nbr | dst << 32 with dst = rowptr[row] + rank of kk among the row's stragglers, rowptr
    u32[n + 1] range-local, totals {entries, stragglers}"""
    sub = km[row0:row1][:, SP_OFFSETS]
    has = sub >= 0
    rowptr = np.concatenate([[0], np.cumsum(has.sum(1))]).astype(np.int64)
    rank = np.cumsum(has, axis=1) - 1
    cube = _cells(sub, SP_TB, 124)
    seg, b, kk, r, q, _ = _stream(cube, 8, True)
    row = b * SP_TB + r
    pairs = np.full(int(seg[-1]), ALL64, np.uint64)
    pairs[q] = cube[b, kk, r].astype(np.uint64) | ((rowptr[row] + rank[row, kk]).astype(np.uint64) << np.uint64(32))
    return seg.astype(np.uint32), pairs, rowptr.astype(np.uint32), (int(seg[-1]), int(rowptr[-1]))


def _hand_map():
    """three rows on a line along x: row o has itself (offset 62) and its x-neighbours (61: dx = -1, 63: dx = +1)"""
    km = np.full((3, 125), -1, np.int32)
    km[:, CENTRE] = [0, 1, 2]
    km[0, 63], km[1, 63] = 1, 2
    km[1, 61], km[2, 61] = 0, 1
    return km


def _e(nbr, row, k):
    return np.uint64(nbr | (row << 32) | (k << 48))


def test_ref_pairs_stream_hand_built():
    km = _hand_map()
    seg, pairs, tot = ref_pairs_stream(km, 0, 3, 8)
    assert seg.shape == (127,) and tot == (24, 7)
    assert seg[61] == 0 and seg[62] == 8 and seg[63] == 16 and seg[64] == 24 and seg[125] == 24 and seg[126] == 24
    assert list(pairs[:2]) == [_e(0, 1, 61), _e(1, 2, 61)] and (pairs[2:8] == ALL64).all()
    assert list(pairs[8:11]) == [_e(0, 0, 62), _e(1, 1, 62), _e(2, 2, 62)]
    assert list(pairs[16:18]) == [_e(1, 0, 63), _e(2, 1, 63)]
    # rows [1, 3) as a level of their own: rows 0, 1 in the tile, neighbour indices stay the level's
    seg, pairs, tot = ref_pairs_stream(km, 1, 3, 8)
    assert tot == (24, 5)
    assert list(pairs[:2]) == [_e(0, 0, 61), _e(1, 1, 61)] and list(pairs[8:10]) == [_e(1, 0, 62), _e(2, 1, 62)]
    assert pairs[16] == _e(2, 0, 63) and (pairs[17:] == ALL64).all()
    # tiles of one row: each row is its own tile, pad 1 keeps the true pairs only
    seg, pairs, tot = ref_pairs_stream(km, 0, 3, 1, pad=1)
    assert tot == (7, 7) and seg[126] == 2 and seg[2 * 126] == 5 and list(seg[126 + 61:126 + 64]) == [2, 3, 4]
    # an empty range
    seg, pairs, tot = ref_pairs_stream(km, 2, 2, 8)
    assert tot == (0, 0) and pairs.size == 0


def test_ref_um_stream_hand_built():
    km = _hand_map()
    seg, nbr, off, tot = ref_um_stream(km, 0, 3)
    assert tot == (48, 7) and seg[62] == 16 and seg[63] == 32 and seg[126] == 48
    assert list(nbr[:3]) == [0, 1, 0xFFFFFFFF] and list(off[:3]) == [128, 256, 512 * 128]
    assert list(nbr[16:19]) == [0, 1, 2] and list(off[16:19]) == [0, 128, 256]
    seg, nbr, off, tot = ref_um_stream(km, 2, 3)
    assert tot == (32, 2) and list(nbr[[0, 16]]) == [1, 2] and list(off[[0, 16]]) == [0, 0] and (off[[1, 17]] == 512 * 128).all()


def test_ref_sparse_stream_hand_built():
    km = _hand_map()
    seg, pairs, rowptr, tot = ref_sparse_stream(km, 0, 3)
    assert list(rowptr) == [0, 1, 3, 4] and tot == (16, 4) and seg.shape == (126,)
    assert seg[61] == 0 and seg[62] == 8 and seg[63] == 16 and seg[124] == 16 and seg[125] == 16
    d = lambda nbr, dst: np.uint64(nbr | (dst << 32))
    assert list(pairs[:2]) == [d(0, 1), d(1, 3)] and (pairs[2:8] == ALL64).all()      # kk 61 (offset 61)
    assert list(pairs[8:10]) == [d(1, 0), d(2, 2)]                                   # kk 62 (offset 63), second straggler of row 1
    seg, pairs, rowptr, tot = ref_sparse_stream(km, 1, 2)
    assert list(rowptr) == [0, 2] and tot == (16, 2) and pairs[0] == d(0, 0) and pairs[8] == d(2, 1)
    # blocks start at row0: 8193 rows with one straggler each are two blocks
    big = np.full((8193, 125), -1, np.int32)
    big[:, CENTRE] = np.arange(8193)
    big[1:, 61] = np.arange(8192)
    seg, pairs, rowptr, tot = ref_sparse_stream(big, 1, 8193)                 # one block
    assert seg.shape == (126,) and tot == (8192, 8192) and (pairs >> np.uint64(32) == np.arange(8192)).all()
    seg, pairs, rowptr, tot = ref_sparse_stream(big, 0, 8193)                 # 8191 + 1 pad in block 0, 1 + 7 pads in block 1
    assert seg.shape == (251,) and seg[125 + 61] == 8192 and tot == (8200, 8192) and pairs[8192] == np.uint64(8191 | (8191 << 32))


# ------------------------------------------------------------------------------------------------------------ clouds
def _cloud(name):
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    xyz = {"hac30k": lambda: hac_like_cloud(30000, 5, extent_log2=16),
           "dense12k": lambda: uniform_unique_cloud(12000, 5, extent_log2=5),         # ~40 pairs per row
           "small700": lambda: uniform_unique_cloud(700, 5, extent_log2=4)}[name]()
    return np.ascontiguousarray(xyz[O.sort_zyx_perm(xyz)])


LEVELS = ["hac30k", "dense12k", "small700"]


def _union_scenes():
    """four scenes stacked along z, more than 4 voxels apart: each is one contiguous row range of the union level.  A ~12 K row
    sparse-ish scene (two 8192-row blocks, a ragged last tcgen05 tile), a dense one, a one-row scene and a dense one ending the level"""
    from gauspcc_b200.synth import hac_like_cloud, uniform_unique_cloud
    from oracle import oracle as O
    parts = [hac_like_cloud(12000, 3, extent_log2=12), uniform_unique_cloud(1500, 3, extent_log2=4),
             np.array([[3, -2, 0]], np.int32), uniform_unique_cloud(700, 4, extent_log2=4)]
    out, z = [], -30000
    for p in parts:
        p = p.astype(np.int64)
        p[:, 2] += z - p[:, 2].min()
        z = int(p[:, 2].max()) + 9
        p = p.astype(np.int32)
        out.append(np.ascontiguousarray(p[O.sort_zyx_perm(p)]))
    return out


def test_two_term_split_exceeds_the_bound(weights_np):
    """the bound is a test of the split: on the levels of the GPU tests a numpy kernel with all three terms stays within it, one that
    keeps only Wh.xh + Wh.xl exceeds it by at least 8x"""
    from gauspcc_b200.weights import CONV_KEYS
    from oracle import oracle as O
    W = weights_np[CONV_KEYS[WIDX]].astype(np.float32)
    rng = np.random.default_rng(0)
    for name in LEVELS:
        xyz = _cloud(name)
        km = O.kmap(xyz, 5)
        x = rng.normal(size=(km.shape[0], 32)).astype(np.float32)
        res = rng.normal(size=(km.shape[0], 32)).astype(np.float32)
        ref, absref = conv64(x, W, km)
        b = bound(absref)
        assert (np.abs(emulate_split_conv(x, W, km, 3) - ref) <= b).all(), name
        assert (np.abs(emulate_split_conv(x, W, km, 2) - ref) / b).max() >= 8.0, name
        # residual and ReLU: the bound is relative to absref, which carries |residual|
        ref2, absref2 = conv64(x, W, km, res, relu=True)
        y2 = np.maximum(emulate_split_conv(x, W, km, 3) + res, 0)
        assert (np.abs(y2 - ref2) <= bound(absref2)).all(), name


def test_conv64_matches_the_fp32_oracle(weights_np):
    from gauspcc_b200.weights import CONV_KEYS
    from oracle import oracle as O
    W = weights_np[CONV_KEYS[WIDX]].astype(np.float32)
    xyz = _cloud("small700")
    km = O.kmap(xyz, 5)
    x = np.random.default_rng(1).normal(size=(km.shape[0], 32)).astype(np.float32)
    ref, absref = conv64(x, W, km)
    assert np.abs(O.conv(x, W, km) - ref).max() <= 1e-5 * np.abs(ref).max()
    assert (absref >= np.abs(ref)).all()


def test_union_scenes_are_contiguous_and_apart():
    from oracle import oracle as O
    scenes = _union_scenes()
    xyz = np.concatenate(scenes)
    assert np.array_equal(O.sort_zyx_perm(xyz), np.arange(xyz.shape[0]))       # scene-major rows
    km = O.kmap(xyz, 5)
    r = 0
    for s in scenes:
        sub = km[r:r + s.shape[0]]
        assert ((sub < 0) | ((sub >= r) & (sub < r + s.shape[0]))).all()         # no neighbour in another scene
        r += s.shape[0]


# ------------------------------------------------------------------------------------------------------------ GPU
def _ranges(n):
    """row ranges with neighbours on both sides of their boundaries: ends, tile boundaries of every tile height, an unaligned whole
    tcgen05 tile, sparse blocks, empty ranges"""
    rs = [(0, n), (0, 1), (n - 1, n), (1, n - 1), (513, 1025), (5000, 21000), (8191, 8193), (0, 0), (n // 2, n // 2), (n, n)]
    rs += [(T - 1, T + 1) for T in (8, 16, 32, 64, 128, 512)]
    out = []
    for r in rs:
        if 0 <= r[0] <= r[1] <= n and r not in out:
            out.append(r)
    return out


V6_CONFIGS = [(47, 8), (46, 16), (46, 32), (48, 32), (48, 64), (48, 128), (42, 64)]
FAMILIES = [("v6", v, t) for v, t in V6_CONFIGS] + [("um", 0, 512), ("sparse", 0, 0)]
SENTINEL = np.uint32(0x7FC0DEAD)                           # a NaN with a payload: a row the kernel writes cannot keep it


@pytest.fixture(scope="module")
def gpu(weights_np):
    from gauspcc_b200 import _lib
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import CONV_KEYS, make_synthetic_state_dict
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    codec = GausPcgcCodec(DeviceWeights(make_synthetic_state_dict(), dev), dev)
    return {"codec": codec, "dev": dev, "W": weights_np[CONV_KEYS[WIDX]].astype(np.float32), "GpcError": _lib.GpcError}


_LEVEL_CACHE = {}


def _level(gpu, name):
    """keys, dense map (device), dense map [n, 125] (host), x, residual and conv64 of one level, computed once"""
    if name in _LEVEL_CACHE:
        return _LEVEL_CACHE[name]
    from oracle import oracle as O
    codec = gpu["codec"]
    xyz = np.concatenate(_union_scenes()) if name == "union" else _cloud(name)
    keys, _ = codec.pack_keys(torch.tensor(xyz, device=codec.dev))
    dense = codec.dense_map(keys)
    km = dense.cpu().numpy().T.copy()
    assert np.array_equal(km, O.kmap(xyz, 5))
    rng = np.random.default_rng(len(xyz))
    x = rng.normal(size=(km.shape[0], 32)).astype(np.float32)
    res = rng.normal(size=(km.shape[0], 32)).astype(np.float32)
    lv = dict(xyz=xyz, keys=keys, dense=dense, km=km, n=km.shape[0], x=x, res=res)
    if name != "union":
        lv["ref"] = conv64(x, gpu["W"], km)
        lv["ref_res"] = conv64(x, gpu["W"], km, res, relu=True)
    _LEVEL_CACHE[name] = lv
    return lv


def _dev(codec, a):
    return torch.tensor(np.ascontiguousarray(a), device=codec.dev)


def _sentinel(codec, shape, dtype=None):
    t = torch.full(shape, int(SENTINEL.view(np.int32)), dtype=torch.int32, device=codec.dev)
    return t.view(torch.float32) if dtype == torch.float32 else t


GUARD = 16                                                  # seg / rowptr entries past their end: never written


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def _untouched(t, start):
    """every 32-bit word of t from element `start` on still holds the sentinel (checked on the device)"""
    words = t.view(torch.int32)[start * (t.element_size() // 4):]
    return bool((words == int(SENTINEL.view(np.int32))).all())


def _capacity(cells, cell_rows, pad):
    """stream entries a fill can address from ANY seg its count writes (every cell at most cell_rows rows, padded): the stream
    arrays are this long, so that a count kernel that disagrees with its fill is caught as writes past the reported total instead
    of writes past the buffer"""
    return max(cells * ((cell_rows + pad - 1) // pad * pad), 1)


def build_range_stream(codec, dense, n_level, r0, r1, fam, T):
    """count + fill of one range entry point into sentinel-filled arrays longer than any stream of the range; returns the device
    arrays and the totals (the convs take them as they are)"""
    from gauspcc_b200.codec import _ptr
    n = r1 - r0
    st = codec._stream()
    if fam == "sparse":
        m = int(codec.lib.gpc_kmap_sparse_segments(n)) + 1
        seg = _sentinel(codec, (m + GUARD,))
        rowptr = _sentinel(codec, (n + 1 + GUARD,))
        tot = torch.full((2,), 12345, dtype=torch.int32, device=codec.dev)
        wb = codec.lib.gpc_kmap_sparse_workspace_bytes(n)
        ws = codec._ws(wb)
        codec._call("gpc_kmap_sparse_count_range", _ptr(dense), n_level, r0, r1, _ptr(seg), _ptr(rowptr), _ptr(tot), _ptr(ws), wb, st)
        e, s = (int(v) for v in tot.tolist())
        pairs = _sentinel(codec, (2 * _capacity(m - 1, SP_TB, 8),)).view(torch.int64)
        codec._call("gpc_kmap_sparse_fill_range", _ptr(dense), n_level, r0, r1, _ptr(seg), _ptr(rowptr), _ptr(ws), _ptr(pairs), e, st)
        contrib = torch.empty((max(s, 1), 32), dtype=torch.float32, device=codec.dev)
        return dict(fam=fam, seg=seg, rowptr=rowptr, pairs=pairs, tot=(e, s), m=m, n=n, contrib=contrib)
    tiles = (n + T - 1) // T
    m = tiles * 126 + 1 if n > 0 else 1
    seg = _sentinel(codec, (m + GUARD,))
    if fam == "um":
        tot = torch.full((2,), 12345, dtype=torch.int64, device=codec.dev)
        wb = codec.lib.gpc_kmap_um_workspace_bytes(n, T)
        ws = codec._ws(wb)
        codec._call("gpc_kmap_um_count_range", _ptr(dense), n_level, r0, r1, T, _ptr(seg), _ptr(tot), _ptr(ws), wb, st)
        e, s = (int(v) for v in tot.tolist())
        nbr = _sentinel(codec, (_capacity(m - 1, T, 16),))
        off = _sentinel(codec, (_capacity(m - 1, T, 16),))
        codec._call("gpc_kmap_um_fill_range", _ptr(dense), n_level, r0, r1, T, _ptr(seg), _ptr(nbr), _ptr(off), st)
        return dict(fam=fam, seg=seg, nbr=nbr, off=off, tot=(e, s), m=m, n=n)
    tot = torch.full((2,), 12345, dtype=torch.int32, device=codec.dev)
    wb = codec.lib.gpc_kmap_pairs_workspace_bytes(n, T)
    ws = codec._ws(wb)
    codec._call("gpc_kmap_pairs_count_range", _ptr(dense), n_level, r0, r1, T, 8, _ptr(seg), _ptr(tot), _ptr(ws), wb, st)
    e, s = (int(v) for v in tot.tolist())
    pairs = _sentinel(codec, (2 * _capacity(m - 1, T, 8),)).view(torch.int64)
    codec._call("gpc_kmap_pairs_fill_range", _ptr(dense), n_level, r0, r1, T, _ptr(seg), _ptr(pairs), e, st)
    return dict(fam=fam, seg=seg, pairs=pairs, tot=(e, s), m=m, n=n, T=T)


def _check_stream(got, km, r0, r1, T):
    """one range stream against its numpy restatement, bit for bit; nothing written past the stream's total, past seg / rowptr, or
    at all for an empty range"""
    fam, n, e = got["fam"], r1 - r0, got["tot"][0]
    assert _untouched(got["seg"], got["m"] if n > 0 else 0), "seg written past its end (or for an empty range)"
    if fam == "sparse":
        rseg, rpairs, rrowptr, rtot = ref_sparse_stream(km, r0, r1)
        assert _untouched(got["rowptr"], n + 1 if n > 0 else 0)
    elif fam == "um":
        rseg, rnbr, roff, rtot = ref_um_stream(km, r0, r1, T)
    else:
        rseg, rpairs, rtot = ref_pairs_stream(km, r0, r1, T)
    assert got["tot"] == rtot
    if n == 0:
        assert rtot == (0, 0)
    else:
        assert np.array_equal(_u32(got["seg"][:got["m"]]), rseg)
    if fam == "um":
        assert np.array_equal(_u32(got["nbr"][:e]), rnbr) and np.array_equal(_u32(got["off"][:e]), roff)
        assert _untouched(got["nbr"], e) and _untouched(got["off"], e), "stream written past its total"
        return
    assert np.array_equal(_u64(got["pairs"][:e]), rpairs)
    assert _untouched(got["pairs"], e), "stream written past its total"
    if fam == "sparse" and n > 0:
        assert np.array_equal(_u32(got["rowptr"][:n + 1]), rrowptr)


STREAMS = [("v6", T) for T in (8, 16, 32, 64, 128)] + [("um", 512), ("sparse", 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", LEVELS)
def test_range_streams_match_the_layout(gpu, name):
    codec = gpu["codec"]
    lv = _level(gpu, name)
    for r0, r1 in _ranges(lv["n"]):
        for fam, T in STREAMS:
            got = build_range_stream(codec, lv["dense"], lv["n"], r0, r1, fam, T)
            try:
                _check_stream(got, lv["km"], r0, r1, T)
            except AssertionError as ex:
                raise AssertionError(f"{name} [{r0}, {r1}) {fam} {T}: {ex}") from ex


@pytest.mark.gpu
def test_range_arguments_rejected(gpu):
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    lv = _level(gpu, "small700")
    n, d, st = lv["n"], _ptr(lv["dense"]), codec._stream()
    buf = codec._ws(1 << 20)
    p = _ptr(buf)
    x = _dev(codec, lv["x"])
    calls = {
        "gpc_kmap_pairs_count_range": lambda a, b: (d, n, a, b, 8, 8, p, p, p, 1 << 20, st),
        "gpc_kmap_pairs_fill_range": lambda a, b: (d, n, a, b, 8, p, p, 0, st),
        "gpc_kmap_um_count_range": lambda a, b: (d, n, a, b, 512, p, p, p, 1 << 20, st),
        "gpc_kmap_um_fill_range": lambda a, b: (d, n, a, b, 512, p, p, p, st),
        "gpc_kmap_sparse_count_range": lambda a, b: (d, n, a, b, p, p, p, p, 1 << 20, st),
        "gpc_kmap_sparse_fill_range": lambda a, b: (d, n, a, b, p, p, p, p, 0, st),
        "gpc_spconv_fwd_v6_range": lambda a, b: (_ptr(x), p, p, p, n, a, b, 8, None, 0, p, 47, st),
        "gpc_spconv_fwd_um_range": lambda a, b: (p, p, p, p, p, n, a, b, None, None, 0, _ptr(x), None, st),
        "gpc_spconv_sparse_fwd_range": lambda a, b: (_ptr(x), p, p, p, p, n, a, b, 0, p, None, 0, p, st),
    }
    for fn, args in calls.items():
        for a, b in ((5, 4), (0, n + 1), (-1, 3), (n, n + 1)):
            rc = getattr(codec.lib, fn)(*args(a, b))
            assert rc == GPC_EINVAL, (fn, a, b, rc)
            with pytest.raises(gpu["GpcError"], match="rc=-1"):
                codec._call(fn, *args(a, b))
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_union_range_streams_are_the_scenes_own(gpu):
    """gpcgc.h: the streams of a range are exactly those of the range's rows coded as a level of their own, with neighbour indices +
    row0 -- compared with the non-range entry points on each scene's own dense map"""
    codec = gpu["codec"]
    lv = _level(gpu, "union")
    r0 = 0
    for s in _union_scenes():
        n = s.shape[0]
        r1 = r0 + n
        keys, _ = codec.pack_keys(_dev(codec, s))
        own = codec.dense_map(keys)
        for fam, T in STREAMS:
            got = build_range_stream(codec, lv["dense"], lv["n"], r0, r1, fam, T)
            e = got["tot"][0]
            if fam == "v6":
                seg, e1, real = codec._count_pairs(own, n, T, 8)
                km = codec._v6_map(own, n, T, 48, counted=(seg, e1, real))
                assert got["tot"] == (e1, real)
                pairs = _u64(km.pairs)[:e]
                nb = pairs & np.uint64(0xFFFFFFFF)
                pairs = np.where(pairs == ALL64, pairs, (pairs & ~np.uint64(0xFFFFFFFF)) | (nb + np.uint64(r0)))
                assert np.array_equal(_u64(got["pairs"][:e]), pairs)
            elif fam == "um":
                seg, e1, real = codec._count_um(own, n, T)
                km = codec._um_map(own, n, T, counted=(seg, e1, real))
                assert got["tot"] == (e1, real)
                nbr = _u32(km.pair_nbr)[:e]
                nbr = np.where(nbr == 0xFFFFFFFF, nbr, nbr + np.uint32(r0))
                assert np.array_equal(_u32(got["nbr"][:e]), nbr)
                assert np.array_equal(_u32(got["off"][:e]), _u32(km.pair_off)[:e])
            else:
                km = codec._sparse_map(own, n)
                assert got["tot"] == (km.n_pairs, km.n_real - n)
                pairs = _u64(km.pairs)[:e]
                pairs = np.where(pairs == ALL64, pairs, pairs + np.uint64(r0))
                assert np.array_equal(_u64(got["pairs"][:e]), pairs)
                assert np.array_equal(_u32(got["rowptr"][:n + 1]), _u32(km.rowptr)[:n + 1])
            assert np.array_equal(_u32(got["seg"][:got["m"]]), _u32(km.seg)[:got["m"]]), (fam, T, r0)
            assert _untouched(got["nbr"] if fam == "um" else got["pairs"], e), (fam, T, r0)
        r0 = r1
    assert r0 == lv["n"]
    torch.cuda.synchronize()


# ---- range convs
def run_range_conv(gpu, fam, variant, st_, n_level, r0, r1, xf, xs, res, flags, y, ys=None, order=None):
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    w = codec.w
    st = codec._stream()
    if fam == "um":
        codec._call("gpc_spconv_fwd_um_range", _ptr(xs), _ptr(w.convs_um[WIDX]), _ptr(st_["seg"]), _ptr(st_["nbr"]), _ptr(st_["off"]),
                    n_level, r0, r1, _ptr(order), _ptr(res), flags, _ptr(y), _ptr(ys), st)
    elif fam == "sparse":
        codec._call("gpc_spconv_sparse_fwd_range", _ptr(xf), _ptr(w.convs_frag[WIDX]), _ptr(st_["seg"]), _ptr(st_["pairs"]),
                    _ptr(st_["rowptr"]), n_level, r0, r1, st_["tot"][0], _ptr(st_["contrib"]), _ptr(res), flags, _ptr(y), st)
    else:
        codec._call("gpc_spconv_fwd_v6_range", _ptr(xf), _ptr(w.convs_frag[WIDX]), _ptr(st_["seg"]), _ptr(st_["pairs"]), n_level, r0, r1,
                    st_["T"], _ptr(res), flags, _ptr(y), variant, st)


def whole_level_kmap(codec, dense, n, fam, variant, T):
    if fam == "um":
        return codec._um_map(dense, n, T)
    if fam == "sparse":
        return codec._sparse_map(dense, n)
    return codec._v6_map(dense, n, T, variant)


def run_whole_conv(codec, km, xf, xs, res, relu, fmt="f32"):
    """the level's own launch (non-range entry points) through codec.conv"""
    if km.um_rows:
        return codec.conv(xs, WIDX, km, residual=res, relu=relu, fmt=fmt)
    return codec.conv(xf, WIDX, km, residual=res, relu=relu)


def _bits(t):
    return t.cpu().numpy().view(np.uint32)


def _tile_orders(codec, st_, n):
    tiles = (n + 511) // 512
    starts = st_["seg"][:tiles * 126 + 1][::126].to(torch.int64)
    heavy = torch.argsort(starts[1:] - starts[:-1], descending=True, stable=True).to(torch.int32)
    rnd = torch.tensor(np.random.default_rng(n).permutation(tiles).astype(np.int32), device=codec.dev)
    return [None, heavy, rnd]


WORST = {}                                                   # family -> worst |err| / absref seen (printed with -s)


@pytest.mark.gpu
@pytest.mark.parametrize("fam,variant,T", FAMILIES)
def test_union_range_conv_is_the_scene_conv(gpu, fam, variant, T):
    """each scene of a union level: the range conv equals the scene's own conv bit for bit while every row outside the scene's 5^3
    closure of x (and of the residual) is NaN; rows outside the range keep their sentinel; the centre TMA box of a ragged last
    tcgen05 tile reads the next scene's NaN rows (first scene) or past the end of the level (last scene) into padding columns"""
    codec = gpu["codec"]
    lv = _level(gpu, "union")
    N = lv["n"]
    r0 = 0
    for s in _union_scenes():
        n = s.shape[0]
        r1 = r0 + n
        xf_h = np.full((N, 32), np.nan, np.float32)
        xf_h[r0:r1] = lv["x"][r0:r1]
        rs_h = np.full((N, 32), np.nan, np.float32)
        rs_h[r0:r1] = lv["res"][r0:r1]
        xf, rf = _dev(codec, xf_h), _dev(codec, rs_h)
        xs, rsplit = codec.split_rows(xf), codec.split_rows(rf)
        st_ = build_range_stream(codec, lv["dense"], N, r0, r1, fam, T)
        _check_stream(st_, lv["km"], r0, r1, T)            # a conv only ever runs on a stream of the documented layout
        keys, _ = codec.pack_keys(_dev(codec, s))
        km = whole_level_kmap(codec, codec.dense_map(keys), n, fam, variant, T)
        oxf, orf = _dev(codec, lv["x"][r0:r1]), _dev(codec, lv["res"][r0:r1])
        oxs, ors = codec.split_rows(oxf), codec.split_rows(orf)
        cases = [(None, 0), ("f32", 1)] if fam != "um" else [(None, 0), ("f32", 1), ("split", 1)]
        for res_kind, relu in cases:
            flags = relu | (2 if res_kind == "split" else 0)
            res = {None: None, "f32": rf, "split": rsplit}[res_kind]
            ores = {None: None, "f32": orf, "split": ors}[res_kind]
            want = run_whole_conv(codec, km, oxf, oxs, ores, bool(relu), fmt="both" if fam == "um" else "f32")
            if fam != "um":
                y = _sentinel(codec, (N, 32), torch.float32)
                run_range_conv(gpu, fam, variant, st_, N, r0, r1, xf, xs, res, flags, y)
                got = _bits(y)
                assert np.array_equal(got[r0:r1], _bits(want)), (fam, variant, T, r0, res_kind)
                assert np.isfinite(got[r0:r1].view(np.float32)).all()
                assert (got[:r0] == SENTINEL).all() and (got[r1:] == SENTINEL).all(), (fam, variant, T, r0, res_kind)
                continue
            wy, wys = (_bits(t) for t in want)
            for i, (oy, oys) in enumerate([(True, False), (False, True), (True, True)]):
                for order in _tile_orders(codec, st_, n) if i == 2 else [None]:
                    y = _sentinel(codec, (N, 32), torch.float32) if oy else None
                    ys = _sentinel(codec, (N, 32)) if oys else None
                    run_range_conv(gpu, fam, variant, st_, N, r0, r1, xf, xs, res, flags, y, ys, order)
                    for out, ref in ((y, wy), (ys, wys)):
                        if out is None:
                            continue
                        got = _bits(out)
                        assert np.array_equal(got[r0:r1], ref), (r0, res_kind, oy, oys, order is None)
                        assert (got[:r0] == SENTINEL).all() and (got[r1:] == SENTINEL).all(), (r0, res_kind, oy, oys)
                    if y is not None:
                        assert np.isfinite(_bits(y)[r0:r1].view(np.float32)).all()
        r0 = r1
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("name", LEVELS)
@pytest.mark.parametrize("fam,variant,T", FAMILIES)
def test_range_conv_fp64_and_whole_level(gpu, name, fam, variant, T):
    """arbitrary ranges of one level, neighbours on both sides of the boundary: rows in range within the fp64 bound and equal to the
    whole-level launch of the same family and tiling bit for bit (every row is summed in one fixed order: offsets ascending, and a
    pair's product does not depend on its column); rows outside keep their sentinel"""
    codec = gpu["codec"]
    lv = _level(gpu, name)
    N = lv["n"]
    xf, rf = _dev(codec, lv["x"]), _dev(codec, lv["res"])
    xs, rsplit = codec.split_rows(xf), codec.split_rows(rf)
    km = whole_level_kmap(codec, lv["dense"], N, fam, variant, T)
    whole = _bits(run_whole_conv(codec, km, xf, xs, None, False))
    whole_res = _bits(run_whole_conv(codec, km, xf, xs, rsplit if fam == "um" else rf, True))
    (ref, absref), (ref2, absref2) = lv["ref"], lv["ref_res"]
    worst = 0.0
    for r0, r1 in _ranges(N):
        st_ = build_range_stream(codec, lv["dense"], N, r0, r1, fam, T)
        _check_stream(st_, lv["km"], r0, r1, T)
        for res, flags, w_bits, rr, ra in ((None, 0, whole, ref, absref),
                                           (rsplit if fam == "um" else rf, 3 if fam == "um" else 1, whole_res, ref2, absref2)):
            y = _sentinel(codec, (N, 32), torch.float32)
            run_range_conv(gpu, fam, variant, st_, N, r0, r1, xf, xs, res, flags, y)
            got = _bits(y)
            tag = (name, fam, variant, T, r0, r1, flags)
            assert (got[:r0] == SENTINEL).all() and (got[r1:] == SENTINEL).all(), tag
            g = got[r0:r1].view(np.float32)
            assert (np.abs(g - rr[r0:r1]) <= bound(ra[r0:r1])).all(), (tag, err_ratio(g, rr[r0:r1], ra[r0:r1]) * 2 ** 16)
            worst = max(worst, err_ratio(g, rr[r0:r1], ra[r0:r1]))
            assert np.array_equal(got[r0:r1], w_bits[r0:r1]), tag
    key = fam if fam != "v6" else f"v6 {variant}@{T}"
    WORST[key] = max(WORST.get(key, 0.0), worst)
    print(f"\nworst |err| / absref {key} on {name}: {worst * 2 ** 16:.3f} * 2^-16 (bound {BOUND_C} * 2^-16)")
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_batch_call_path_mixed_families(gpu):
    """BatchCodec._kmaps / _stack on one union level whose members take three families into the same aliased activation buffers:
    every member's rows equal the single-scene _res_stack bit for bit"""
    from gauspcc_b200 import weights as Wm
    from gauspcc_b200.batch import Act, BatchCodec, ULevel
    from gauspcc_b200.codec import GausPcgcCodec
    base = gpu["codec"]
    codec = GausPcgcCodec(base.w, gpu["dev"])
    codec.um_min_rows, codec.sparse_min_rows, codec.sparse_max_density = 1000, 1000, 4.5
    lv_h = _level(gpu, "union")
    scenes = _union_scenes()
    ranges, r = [], 0
    for s in scenes:
        ranges.append((r, r + s.shape[0]))
        r += s.shape[0]
    lv = ULevel(lv_h["keys"], None, list(range(len(scenes))), ranges)
    bc = BatchCodec(codec)
    lv.kmaps = bc._kmaps(lv)
    fams = ["um" if k.um_rows else ("sparse" if k.sparse else "v6") for k in lv.kmaps]
    assert fams == ["sparse", "um", "v6", "v6"], fams
    xf = _dev(codec, lv_h["x"])
    out = bc._stack(Act(xf, codec.split_rows(xf)), Wm.PRIOR_CONVS, lv, lv.n, len(scenes), both=True)
    for s, (r0, r1), f in zip(scenes, ranges, fams):
        keys, _ = codec.pack_keys(_dev(codec, s))
        km = codec.build_kmap(keys)
        assert bool(km.um_rows) == (f == "um") and km.sparse == (f == "sparse")
        want = codec._res_stack(xf[r0:r1].contiguous(), Wm.PRIOR_CONVS, km, "both" if f == "um" else "f32")
        if f == "um":
            assert np.array_equal(_bits(out.f)[r0:r1], _bits(want[0])) and np.array_equal(_bits(out.s)[r0:r1], _bits(want[1]))
        else:
            assert np.array_equal(_bits(out.f)[r0:r1], _bits(want)), (r0, f)
    torch.cuda.synchronize()


# ---- row-restricted convs of the decoder wavefront
def _closure(km, r0, r1):
    nb = km[r0:r1]
    return np.unique(nb[nb >= 0])


@pytest.mark.gpu
@pytest.mark.parametrize("fam,T", [("v6", 32), ("v6", 64), ("v6", 128), ("sparse", 0), ("um", 512)])
def test_rows_conv_reads_only_its_closure(gpu, fam, T):
    """codec.conv(..., rows=) (gpc_spconv_fwd_v6_rows, gpc_spconv_sparse_fwd_rows, gpc_spconv_fwd_um with a row range): with NaN in
    every input row outside the 5^3 closure of [r0, r1), the rows equal the whole launch bit for bit and every other row keeps its
    sentinel; a range that is not made of whole tiles / blocks is rejected"""
    codec = gpu["codec"]
    lv = _level(gpu, "hac30k")
    N, kmh = lv["n"], lv["km"]
    km = whole_level_kmap(codec, lv["dense"], N, fam, 48, T)
    xf, rf = _dev(codec, lv["x"]), _dev(codec, lv["res"])
    unit = SP_TB if fam == "sparse" else T
    spans = [(unit, 2 * unit), (SP_TB, SP_TB + 3 * unit if fam != "sparse" else 3 * SP_TB), (N // unit * unit, N), (0, N)]
    for res_on in (False, True):
        whole = _bits(run_whole_conv(codec, km, xf, codec.split_rows(xf), rf if res_on else None, res_on))
        for r0, r1 in spans:
            keep = _closure(kmh, r0, r1)
            x_h = np.full((N, 32), np.nan, np.float32)
            x_h[keep] = lv["x"][keep]
            r_h = np.full((N, 32), np.nan, np.float32)
            r_h[r0:r1] = lv["res"][r0:r1]
            x, res = _dev(codec, x_h), (_dev(codec, r_h) if res_on else None)
            y = _sentinel(codec, (N, 32), torch.float32)
            codec.conv(codec.split_rows(x) if fam == "um" else x, WIDX, km, residual=res, relu=res_on, out=y, rows=(r0, r1))
            got = _bits(y)
            assert np.array_equal(got[r0:r1], whole[r0:r1]), (fam, T, r0, r1, res_on)
            assert (got[:r0] == SENTINEL).all() and (got[r1:] == SENTINEL).all(), (fam, T, r0, r1, res_on)
    for r0, r1 in ((unit // 2, unit), (0, unit + 1 if unit + 1 < N else N - 1), (1, N)):
        with pytest.raises(gpu["GpcError"], match="rc=-1"):
            codec.conv(xf if fam != "um" else codec.split_rows(xf), WIDX, km, out=torch.empty_like(xf), rows=(r0, r1))
    torch.cuda.synchronize()
