"""The network of one octree level, kernel by kernel and call by call, against numpy restatements and an fp64 reference.

A level's network (oracle/oracle.py: _level_features, _res_stack, _stage) runs as these calls: the prior embedding, a 5-conv prior
stack, the parent gather plus the octant embedding, a 5-conv target stack, then four stages of (context embedding,) two convs and
the fused head.  On tcgen05 levels the activations between the calls are split rows (include/gpcgc.h, spconv_fmt.cu): one row =
16 words of bf16x2 hi | 16 words of bf16x2 lo, channel 2j in the low half of word j.

  * split rows: one numpy restatement (split_ref) and every producer of the format compared with it bit for bit;
  * the three producers (gpc_embed_rows, gpc_gather_parent_add_octant, gpc_add_ctx_embed): fp32 rows bit for bit against numpy
    float32, split rows against split_ref;
  * the head: probabilities against fp64 within a bound derived below, and the encoder's (c_low, c_high) words against the CDF rows;
  * the production chain, teacher-forced: every conv of an encode and of a stage-by-stage decode, recorded call by call, against an
    fp64 conv of that call's own recorded inputs, and the wiring of the calls against the network of the oracle.

The error bars here are far below what the codec's end-to-end bar (probabilities within 1e-3 of the fp32 oracle) can see: an error
of bf16 size at one seam (a producer dropping the lo half, a split residual read as hi only) moves the probabilities by less than
1e-3 and the bytes by less than 0.5 %, and encoder and decoder make the same error, so the round trip stays lossless."""
import numpy as np
import pytest

from test_row_ranges import bound, conv64

try:
    import torch
except ImportError:                                           # the CPU references below do not need it
    torch = None

GPC_EINVAL = -1
GPC_COORD_BIAS = 1 << 20
GPC_COORD_MAX = (1 << 20) - 16
CTX_SHIFT = (None, 7, 6, 4)                                   # codec.CTX_SHIFT
STAGE_SHIFT = (7, 6, 4, 0)                                    # codec.STAGE_SHIFT
U32 = 2.0 ** -24                                              # unit roundoff of fp32

# ------------------------------------------------------------------------------------------------------------ split rows
# The contract split_ref pins (every producer of split rows must meet it bit for bit):
#   hi = bf16 RNE(x), lo = bf16 RNE(x - hi) (the difference in fp32, exact for finite x), packed as in the module docstring;
#   * finite |x| below 0x7F7F8000 (as bits) joins back (hi + lo in fp32, exact) to within 2^-17 |x| -- 16 mantissa bits -- or
#     within 2^-134 (half the smallest bf16 subnormal) where lo is subnormal;
#   * non-finite in gives non-finite out, so NaN on join: NaN -> (NaN, NaN); +-inf -> (+-inf, NaN); a finite |x| >= 0x7F7F8000
#     rounds to hi = +-inf, lo = -+inf.
# NaN halves are compared as NaN, whatever their payload; every other half bit for bit.
def bf16_bits(a):
    """float32 -> uint16 bf16 bits, round to nearest even; NaN -> 0x7FFF (sign and payload are not part of the contract)"""
    a = np.ascontiguousarray(a, np.float32)
    u = a.view(np.uint32).astype(np.uint64)
    r = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF).astype(np.uint16)
    r[np.isnan(a)] = 0x7FFF
    return r


def bits_f32(h):
    """uint16 bf16 bits -> float32"""
    return (np.asarray(h, np.uint32) << 16).view(np.float32)


def split_halves(x):
    """float32 [..] -> (hi, lo) uint16 bf16 bits"""
    x = np.ascontiguousarray(x, np.float32)
    hi = bf16_bits(x)
    with np.errstate(invalid="ignore", over="ignore"):
        r = x - bits_f32(hi)
    return hi, bf16_bits(r)


def split_ref(x):
    """fp32 rows [n, 32] -> split rows uint32 [n, 32]: word j = hi[2j] | hi[2j+1] << 16, word 16 + j the same of lo"""
    hi, lo = split_halves(np.asarray(x, np.float32).reshape(-1, 32))
    pack = lambda h: h[:, 0::2].astype(np.uint32) | (h[:, 1::2].astype(np.uint32) << 16)
    return np.concatenate([pack(hi), pack(lo)], axis=1)


def unpack_halves(xs):
    """split rows uint32 [n, 32] -> (hi, lo) uint16 [n, 32] in channel order"""
    xs = np.asarray(xs).view(np.uint32).reshape(-1, 32)
    out = []
    for w in (xs[:, :16], xs[:, 16:]):
        h = np.empty((xs.shape[0], 32), np.uint16)
        h[:, 0::2], h[:, 1::2] = w & 0xFFFF, w >> 16
        out.append(h)
    return out


def join_ref(xs):
    """split rows -> fp32 rows: hi + lo in fp32"""
    hi, lo = unpack_halves(xs)
    with np.errstate(invalid="ignore", over="ignore"):
        return bits_f32(hi) + bits_f32(lo)


def join64(xs):
    """split rows -> float64 rows (hi + lo exactly)"""
    hi, lo = unpack_halves(xs)
    with np.errstate(invalid="ignore"):
        return bits_f32(hi).astype(np.float64) + bits_f32(lo).astype(np.float64)


def _nan_aware_equal(a, b):
    """uint16 / uint32 bit patterns of bf16 / fp32 values: equal bits, or both NaN"""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.uint16:
        na, nb = (a & 0x7FFF) > 0x7F80, (b & 0x7FFF) > 0x7F80
    else:
        a, b = a.view(np.uint32), b.view(np.uint32)
        na, nb = (a & 0x7FFFFFFF) > 0x7F800000, (b & 0x7FFFFFFF) > 0x7F800000
    return (na == nb) & (na | (a == b))


def assert_split_equal(got, want, what=""):
    """split rows bit for bit against split rows (NaN halves as NaN)"""
    gh, gl = unpack_halves(got)
    wh, wl = unpack_halves(want)
    for g, w, half in ((gh, wh, "hi"), (gl, wl, "lo")):
        ok = _nan_aware_equal(g, w)
        if not ok.all():
            r, c = np.argwhere(~ok)[0]
            raise AssertionError(f"{what}: {half} half of row {r} channel {c}: 0x{int(g[r, c]):04x}, want 0x{int(w[r, c]):04x}")


def assert_f32_equal(got, want, what=""):
    ok = _nan_aware_equal(np.ascontiguousarray(got, np.float32).view(np.uint32), np.ascontiguousarray(want, np.float32).view(np.uint32))
    if not ok.all():
        i = np.argwhere(~ok)[0]
        raise AssertionError(f"{what}: at {tuple(i)}: {np.asarray(got)[tuple(i)]!r}, want {np.asarray(want)[tuple(i)]!r}")


EDGE_BITS = np.array([
    0x00000000, 0x80000000,                                   # +-0
    0x00000001, 0x807FFFFF, 0x00400000, 0x00012345, 0x80008001,  # subnormals
    0x03800800, 0x83801000,                                   # 2^-120 (1 + 2^-12): hi normal, lo = 2^-132 subnormal
    0x3F808000, 0x3F818000, 0xBF808000, 0xC0018000,           # RNE ties: the bf16 bit below is even (down) / odd (up)
    0x3F808001, 0x3F807FFF,                                   # just above / below a tie
    0x3F800000, 0xC2F60000, 0x7F7F0000, 0x00010000,           # exact in bf16: lo = 0
    0x7F7F7FFF, 0xFF7F7FFF,                                   # largest finite below the bf16 overflow
    0x7F7F8000, 0xFF7F8000, 0x7F7FFFFF,                       # the first above it (a tie, to even = inf), FLT_MAX
    0x7F800000, 0xFF800000,                                   # +-inf
    0x7FC00000, 0x7FFFFFFF, 0xFFFFFFFF, 0x7F800001,           # NaN: quiet, all ones (what GPU arithmetic makes), payload low
    0x3EAAAAAB, 0x4049FDB0, 0xBDCCCCCD, 0x47C35000,           # ordinary values
], np.uint32)


def edge_rows(n, seed=0):
    """n rows of 32 channels: the edge values, each in even and odd channels, then random values of spread magnitudes"""
    rng = np.random.default_rng(seed)
    m = n * 32
    pad = np.full(1 - EDGE_BITS.size % 2, 0x3F800000, np.uint32)           # the second copy lands on the other channel parity
    base = np.concatenate([EDGE_BITS, pad, EDGE_BITS]).view(np.float32)
    rnd = (rng.normal(size=m) * np.exp2(rng.integers(-20, 20, size=m))).astype(np.float32)
    v = np.concatenate([base, rnd])[:m] if m > base.size else base[:m]
    return np.ascontiguousarray(v.reshape(n, 32))


def test_split_ref_hand_values():
    f = lambda b: np.array([b], np.uint32).view(np.float32)
    assert [int(v[0]) for v in split_halves(f(0x3F808000))] == [0x3F80, 0x3B80]      # tie, even: down, lo = +2^-8
    assert [int(v[0]) for v in split_halves(f(0x3F818000))] == [0x3F82, 0xBB80]      # tie, odd: up, lo = -2^-8
    assert [int(v[0]) for v in split_halves(f(0x03800800))] == [0x0380, 0x0002]      # lo = 2^-132, a bf16 subnormal
    assert [int(v[0]) for v in split_halves(f(0x7F7F8000))] == [0x7F80, 0xFF80]      # overflow: inf, -inf
    hi, lo = split_halves(f(0x7F800000))
    assert hi[0] == 0x7F80 and (lo[0] & 0x7FFF) > 0x7F80                           # inf: lo = inf - inf = NaN
    for b in (0x7FC00000, 0x7FFFFFFF, 0xFFFFFFFF, 0x7F800001):
        hi, lo = split_halves(f(b))
        assert (hi[0] & 0x7FFF) > 0x7F80 and (lo[0] & 0x7FFF) > 0x7F80, hex(b)
    xs = split_ref(np.arange(32, dtype=np.float32)[None] + 0.5)
    assert xs[0, 0] == 0x3FC03F00 and xs[0, 16] == 0                               # 0.5 | 1.5 << 16, exact: lo words 0


def test_split_ref_contract():
    """finite |x| < 0x7F7F8000 joins to within max(2^-17 |x|, 2^-134); everything else joins to NaN; bf16_bits is the RNE of
    test_row_ranges.bf16 on finite values"""
    from test_row_ranges import bf16
    rng = np.random.default_rng(1)
    x = np.concatenate([EDGE_BITS, rng.integers(0, 1 << 32, size=200_000, dtype=np.uint64).astype(np.uint32)]).view(np.float32)
    fin = np.isfinite(x)
    assert np.array_equal(bits_f32(bf16_bits(x[fin])).view(np.uint32), bf16(x[fin]).view(np.uint32))
    xs = split_ref(np.resize(x, (x.size + 31) // 32 * 32).reshape(-1, 32))
    j = join_ref(xs).ravel()[:x.size]
    small = fin & ((x.view(np.uint32) & 0x7FFFFFFF) < 0x7F7F8000)
    err = np.abs(j[small].astype(np.float64) - x[small])
    assert (err <= np.maximum(2.0 ** -17 * np.abs(x[small].astype(np.float64)), 2.0 ** -134)).all()
    assert np.isnan(j[~small]).all()
    assert np.array_equal(join64(xs).ravel()[:x.size][small], j[small].astype(np.float64))   # hi + lo is exact in fp32


# ------------------------------------------------------------------------------------------------------------ producers
def pack_keys_ref(xyz):
    """voxel keys (common.cuh key_pack): (z + 2^20) << 42 | (y + 2^20) << 21 | (x + 2^20)"""
    c = np.asarray(xyz, np.int64) + GPC_COORD_BIAS
    return ((c[:, 2] << 42) | (c[:, 1] << 21) | c[:, 0]).astype(np.int64)


def keys_to_xyz(keys):
    k = np.asarray(keys).view(np.uint64).astype(np.int64)
    m = (1 << 21) - 1
    return np.stack([k & m, (k >> 21) & m, (k >> 42) & m], axis=1) - GPC_COORD_BIAS


def octant_ref(xyz):
    """kit/nn.py:114-116: (x & 1) + 2 (y & 1) + 4 (z & 1) of the child's (signed) coordinates"""
    c = np.asarray(xyz, np.int64)
    return (c[:, 0] & 1) + 2 * (c[:, 1] & 1) + 4 * (c[:, 2] & 1)


def embed_ref(table, idx):
    return np.asarray(table, np.float32)[np.asarray(idx, np.int64)]


def gather_ref(feat, parent, temb, child_xyz):
    return np.asarray(feat, np.float32)[np.asarray(parent, np.int64)] + np.asarray(temb, np.float32)[octant_ref(child_xyz)]


def ctx_ref(u, occ, shift, emb):
    return np.asarray(u, np.float32) + np.asarray(emb, np.float32)[np.asarray(occ, np.int64) >> shift]


def _child_coords(n, rng):
    """coordinates with every octant, negative values, and both ends of the key range"""
    c = rng.integers(-GPC_COORD_MAX, GPC_COORD_MAX + 1, size=(n, 3))
    ends = np.array([[GPC_COORD_MAX, -GPC_COORD_MAX, -1], [-GPC_COORD_MAX, GPC_COORD_MAX, GPC_COORD_MAX],
                     [-1, -2, -3], [0, -GPC_COORD_MAX, 1], [-GPC_COORD_MAX + 1, GPC_COORD_MAX - 1, -GPC_COORD_MAX]])
    octs = np.array([[i & 1, (i >> 1) & 1, (i >> 2) & 1] for i in range(8)]) - 2 * np.array([[3, 1, 2]])   # negative, all octants
    fixed = np.concatenate([octs, ends])
    k = min(n, fixed.shape[0])
    c[:k] = fixed[:k]
    return c.astype(np.int32)


def test_octant_of_keys_matches_coordinates():
    """the octant restatement on signed coordinates equals the low bits of the biased key fields (common.cuh key_octant), and the
    key restatement round-trips, for negative coordinates and both ends of the range"""
    c = _child_coords(5003, np.random.default_rng(2))
    k = pack_keys_ref(c).view(np.uint64)
    ko = (k & np.uint64(1)) | (((k >> np.uint64(21)) & np.uint64(1)) << np.uint64(1)) | (((k >> np.uint64(42)) & np.uint64(1)) << np.uint64(2))
    assert np.array_equal(ko.astype(np.int64), octant_ref(c))
    assert set(octant_ref(c[:13]).tolist()) == set(range(8))
    assert np.array_equal(keys_to_xyz(k), c)


# ------------------------------------------------------------------------------------------------------------ head vs fp64
# gpc_head_cdf (head.cu), one thread per row: h_j = max(b1_j + sum_i x_i W1_ji, 0) and lg_a = b2_a + sum_j h_j W2_aj as 32
# sequential fp32 FMAs each, d_a = lg_a - max lg, E_a = expf(d_a), S = E_0 + ... + E_{A-1} (A - 1 additions), p_a = E_a / S.
# Error bound against the same formulas in fp64 on the same fp32 input (g_n = n u / (1 - n u), u = 2^-24):
#   * first layer: |h_j - h64_j| <= e1_j = g_32 (|b1_j| + sum_i |x_i| |W1_ji|) (32 roundings of a sequential sum; ReLU is
#     1-Lipschitz);
#   * second layer: |lg_a - lg64_a| <= e2_a = sum_j |W2_aj| e1_j + g_32 (|b2_a| + sum_j (|h64_j| + e1_j) |W2_aj|);
#   * softmax is shift-invariant, so the max cancels; the rounding of lg - mx perturbs logit a by u |lg_a - mx| <= u (|lg64_a -
#     max lg64| + 2 max e2): each logit carries eta_a = e2_a + that, and the exact softmax of the perturbed logits is within a
#     factor exp(+-(|eta_a| + max eta)) of p64_a;
#   * expf: at most 2 ulp (CUDA C Programming Guide), relative 2^-22; the A - 1 additions of positive terms: g_{A-1}; the division:
#     u.  Together p_a = p64_a (1 + r_a), |r_a| <= (1 + expm1(eta_a + max eta)) (1 + 2^-22) (1 + u) / ((1 - 2^-22) (1 - g_{A-1})) - 1,
#     plus 2^-126 absolute for terms expf flushes to (sub)normals near zero (S >= 1: the largest term is expf(0) = 1).
# A kernel that rounds h to bf16 (or anything else of bf16 size) exceeds this by a wide margin (test_head_bound_catches_bf16).
HEAD_TINY = 2.0 ** -126


def _gamma(n):
    return n * U32 / (1 - n * U32)


def head64(f, W1, b1, W2, b2):
    """fp64 probabilities and their bound for fp32 rows f [n, 32]: (p64 [n, A], bound [n, A])"""
    x = np.asarray(f, np.float64)
    W1, b1, W2, b2 = (np.asarray(a, np.float64) for a in (W1, b1, W2, b2))
    s1 = b1 + x @ W1.T
    h = np.maximum(s1, 0.0)
    e1 = _gamma(32) * (np.abs(b1) + np.abs(x) @ np.abs(W1).T)
    lg = b2 + h @ W2.T
    e2 = e1 @ np.abs(W2).T + _gamma(32) * (np.abs(b2) + (np.abs(h) + e1) @ np.abs(W2).T)
    mx = lg.max(axis=1, keepdims=True)
    p = np.exp(lg - mx)
    p /= p.sum(axis=1, keepdims=True)
    eta = e2 + U32 * (np.abs(lg - mx) + 2 * e2.max(axis=1, keepdims=True))
    A = W2.shape[0]
    r = (1 + np.expm1(eta + eta.max(axis=1, keepdims=True))) * (1 + 2.0 ** -22) * (1 + U32) / ((1 - 2.0 ** -22) * (1 - _gamma(A - 1))) - 1
    return p, p * r + HEAD_TINY


def head_emulated(f, W1, b1, W2, b2, h_bf16=False):
    """the kernel's arithmetic in numpy float32 (sequential FMAs emulated in float64 and rounded per step); h_bf16: the first
    layer's output rounded to bf16 (a mutation the bound must catch)"""
    from test_row_ranges import bf16
    x = np.asarray(f, np.float32)
    n = x.shape[0]
    W1, b1, W2, b2 = (np.asarray(a, np.float32) for a in (W1, b1, W2, b2))
    h = np.empty((n, 32), np.float32)
    for j in range(32):
        s = np.full(n, b1[j], np.float32)
        for i in range(32):
            s = (x[:, i].astype(np.float64) * W1[j, i] + s).astype(np.float32)
        h[:, j] = np.maximum(s, 0)
    if h_bf16:
        h = bf16(h)
    A = W2.shape[0]
    lg = np.empty((n, A), np.float32)
    for a in range(A):
        s = np.full(n, b2[a], np.float32)
        for j in range(32):
            s = (h[:, j].astype(np.float64) * W2[a, j] + s).astype(np.float32)
        lg[:, a] = s
    e = np.exp((lg - lg.max(axis=1, keepdims=True)).astype(np.float32))
    sm = np.zeros(n, np.float32)
    for a in range(A):
        sm = (sm + e[:, a]).astype(np.float32)
    return (e / sm[:, None]).astype(np.float32)


def head_rows(n, seed):
    """features of spread scale with tied (constant), saturating (+-1e4) and all-zero rows among them"""
    rng = np.random.default_rng(seed)
    f = (rng.normal(size=(n, 32)) * rng.choice([0.3, 3.0, 10.0], size=(n, 1))).astype(np.float32)
    special = [np.zeros(32), np.full(32, 0.75), np.full(32, -2.0), np.full(32, 1e4), np.full(32, -1e4),
               np.where(np.arange(32) % 2 == 0, 1e4, -1e4), np.full(32, 1e4) * np.sign(rng.normal(size=32))]
    for k in range(0, n, 61):                                 # spread over the CTAs, the last one included
        f[k] = special[(k // 61) % len(special)]
    if n > 1:
        f[n - 1] = 0.0
    return f


def head_weights(w, i, tied=False):
    """pred_head_s{i} of the synthetic model; tied: logits 0 and 1 equal for every row (second output row = first)"""
    W1, b1, W2, b2 = (np.array(w[f"pred_head_s{i}.{k}"], np.float32) for k in ("0.weight", "0.bias", "2.weight", "2.bias"))
    if tied:
        W2[1], b2[1] = W2[0], b2[0]
    return W1, b1, W2, b2


STAGE_OF_A = {2: 0, 4: 2, 16: 3}


def test_head_bound_catches_bf16(weights_np):
    """the numpy model of the kernel stays within the bound; rounding h to bf16 exceeds it by at least 16x"""
    f = head_rows(2000, 3)
    for A, i in STAGE_OF_A.items():
        hw = head_weights(weights_np, i)
        p64, b = head64(f, *hw)
        assert (np.abs(head_emulated(f, *hw) - p64) <= b).all(), A
        assert (np.abs(head_emulated(f, *hw, h_bf16=True) - p64) / b).max() >= 16.0, A


def test_head64_matches_the_fp32_oracle(weights_np):
    from oracle import oracle as O
    f = head_rows(500, 4)
    for A, i in STAGE_OF_A.items():
        hw = head_weights(weights_np, i)
        p64, b = head64(f, *hw)
        assert np.abs(O.head(f, *hw) - p64).max() <= 1e-6
        assert np.allclose(p64.sum(1), 1.0)


# ------------------------------------------------------------------------------------------------------------ GPU fixtures
SENT = 0x7FC0DEAD                                             # a NaN with a payload: a word the kernel writes cannot keep it
SENT_I32 = int(np.array([SENT], np.uint32).view(np.int32)[0])


@pytest.fixture(scope="module")
def gpu(weights_np):
    from gauspcc_b200 import _lib
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    codec = GausPcgcCodec(DeviceWeights(make_synthetic_state_dict(), dev), dev)
    return {"codec": codec, "dev": dev, "w": weights_np, "GpcError": _lib.GpcError}


def _dev(codec, a):
    return torch.tensor(np.ascontiguousarray(a), device=codec.dev)


def _sent(codec, shape, dtype=torch.int32):
    t = torch.full(shape, SENT_I32, dtype=torch.int32, device=codec.dev)
    return t.view(dtype)


def _host_u32(t):
    return t.cpu().numpy().view(np.uint32)


def _untouched(t, row):
    return bool((_host_u32(t)[row:] == SENT).all())


# ------------------------------------------------------------------------------------------------------------ §1 split rows
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 37, 4099])
def test_rows_split_join_bit_for_bit(gpu, n):
    """gpc_rows_split / gpc_rows_join against split_ref / join_ref on the edge values (n * 16 threads: 16, 592 and 65584, none a
    multiple of the 256-thread blocks but 16); the guard rows after n keep their sentinel"""
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    x = edge_rows(n, seed=n)
    xs = _sent(codec, (n + 2, 32))
    codec._call("gpc_rows_split", _ptr(_dev(codec, x)), n, _ptr(xs), codec._stream())
    got = _host_u32(xs)
    assert_split_equal(got[:n], split_ref(x), f"gpc_rows_split n={n}")
    assert _untouched(xs, n), "split written past n rows"
    # join: of the restatement's words, and of arbitrary words (every bf16 pair, NaN and inf halves included)
    rng = np.random.default_rng(n)
    for words in (split_ref(x), rng.integers(0, 1 << 32, size=(n, 32), dtype=np.uint64).astype(np.uint32)):
        y = _sent(codec, (n + 2, 32), torch.float32)
        codec._call("gpc_rows_join", _ptr(_dev(codec, words.view(np.int32))), n, _ptr(y), codec._stream())
        assert_f32_equal(y.cpu().numpy()[:n], join_ref(words), f"gpc_rows_join n={n}")
        assert _untouched(y, n), "join written past n rows"
    torch.cuda.synchronize()


def _um_level(gpu):
    from gauspcc_b200.synth import uniform_unique_cloud
    from oracle import oracle as O
    codec = gpu["codec"]
    xyz = uniform_unique_cloud(1500, 11, extent_log2=4)
    xyz = np.ascontiguousarray(xyz[O.sort_zyx_perm(xyz)])
    keys, _ = codec.pack_keys(_dev(codec, xyz))
    n = keys.shape[0]
    km = codec._um_map(codec.dense_map(keys), n, 512)
    return km, n, xyz


@pytest.mark.gpu
def test_tcgen05_split_output_is_split_ref(gpu):
    """the tcgen05 conv's ys (its epilogue's own rounding, spconv_um.cu) against split_ref: with x = 0 rows the output is the fp32
    residual exactly (0 + r), so the residual carries the edge values into the epilogue.  ys alone and fmt "both", with and
    without ReLU; NaN and inf rows must join to NaN, as gpc_rows_split's do.  Then on random rows: ys == split_ref(y) whenever both
    are written."""
    codec = gpu["codec"]
    km, n, _ = _um_level(gpu)
    x0 = torch.zeros((n, 32), dtype=torch.int32, device=codec.dev)          # split rows of 0.0
    res = edge_rows(n, seed=5)
    res[res.view(np.uint32) == 0x80000000] = 0.0              # the sign of 0 + (-0) depends on the sign of the zero sum: not pinned
    rd = _dev(codec, res)
    for relu in (False, True):
        with np.errstate(invalid="ignore"):
            o = np.float32(0) + res
            if relu:
                o = np.where(np.isnan(o), np.float32(0), np.maximum(o, np.float32(0)))   # fmaxf(NaN, 0) = 0
        for widx in (7, 16):
            ys = codec.conv(x0, widx, km, residual=rd, relu=relu, fmt="split")
            assert_split_equal(_host_u32(ys), split_ref(o), f"ys alone relu={relu}")
            y, ys = codec.conv(x0, widx, km, residual=rd, relu=relu, fmt="both")
            assert_f32_equal(y.cpu().numpy(), o, f"y relu={relu}")
            assert_split_equal(_host_u32(ys), split_ref(o), f"ys of both relu={relu}")
            if not relu:
                bad = ~np.isfinite(res) | ((res.view(np.uint32) & 0x7FFFFFFF) >= 0x7F7F8000)
                assert np.isnan(join_ref(_host_u32(ys))[bad]).all(), "a non-finite output must join to NaN"
    rng = np.random.default_rng(6)
    xf = _dev(codec, rng.normal(size=(n, 32)).astype(np.float32))
    xs = codec.split_rows(xf)
    for res_t in (None, _dev(codec, rng.normal(size=(n, 32)).astype(np.float32)), xs):
        for relu in (False, True):
            y, ys = codec.conv(xs, 3, km, residual=res_t, relu=relu, fmt="both")
            assert np.array_equal(_host_u32(ys), split_ref(y.cpu().numpy()))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------ §2 producers
PRODUCER_NS = [0, 1, 7, 5003]
OUTS = [(True, False), (False, True), (True, True)]


def _run_producer(gpu, name, n, want_f, make_args):
    """one producer call into sentinel buffers of n + 3 rows; checks rows [0, n) bit for bit and the guard rows"""
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    want = None
    for of, os_ in OUTS:
        out = _sent(codec, (n + 3, 32), torch.float32) if of else None
        outs = _sent(codec, (n + 3, 32)) if os_ else None
        codec._call(name, *make_args(_ptr(out), _ptr(outs)), codec._stream())
        if want is None:
            want = want_f()
        if of:
            assert_f32_equal(out.cpu().numpy()[:n], want, f"{name} n={n} fp32 (split too: {os_})")
            assert np.array_equal(out.cpu().numpy()[:n].view(np.uint32), np.ascontiguousarray(want).view(np.uint32))
            assert _untouched(out, n), f"{name}: fp32 rows written past n"
        if os_:
            assert np.array_equal(_host_u32(outs)[:n], split_ref(want)), \
                f"{name} n={n} split (fp32 too: {of})"
            assert _untouched(outs, n), f"{name}: split rows written past n"
    torch.cuda.synchronize()


def _table(rng, rows):
    """random fp32 rows of spread magnitudes, some exact in bf16, some with RNE ties in their low bits"""
    t = (rng.normal(size=(rows, 32)) * np.exp2(rng.integers(-8, 8, size=(rows, 32)))).astype(np.float32)
    u = t.view(np.uint32)
    u[::3, ::2] &= 0xFFFF0000
    u[1::3, 1::2] = (u[1::3, 1::2] & 0xFFFF0000) | 0x8000
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("n", PRODUCER_NS)
def test_embed_rows(gpu, n):
    codec = gpu["codec"]
    rng = np.random.default_rng(n + 1)
    table = _table(rng, 256)
    idx = rng.permutation(np.resize(np.arange(256, dtype=np.uint8), n))      # every byte (n = 5003)
    tb, ib = _dev(codec, table), _dev(codec, idx)
    _run_producer(gpu, "gpc_embed_rows", n, lambda: embed_ref(table, idx),
                  lambda o, s: (ib.data_ptr(), n, tb.data_ptr(), o, s))


@pytest.mark.gpu
@pytest.mark.parametrize("n", PRODUCER_NS)
def test_gather_parent_add_octant(gpu, n):
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    rng = np.random.default_rng(n + 2)
    c = _child_coords(max(n, 1), rng)[:n]
    m = max(n // 3, 1)
    feat = _table(rng, m)
    temb = _table(rng, 8)
    parent = rng.integers(0, m, size=n).astype(np.uint32)
    keys, meta = codec.pack_keys(_dev(codec, c.reshape(-1, 3))) if n else (torch.zeros(0, dtype=torch.int64, device=codec.dev), None)
    if n:
        assert (meta.cpu().numpy()[0] & 2) == 0 and np.array_equal(keys.cpu().numpy(), pack_keys_ref(c))
        assert set(octant_ref(c[:13]).tolist()) >= set(range(min(8, n)))
    fb, pb, tb = _dev(codec, feat), _dev(codec, parent.view(np.int32)), _dev(codec, temb)
    _run_producer(gpu, "gpc_gather_parent_add_octant", n, lambda: gather_ref(feat, parent, temb, c),
                  lambda o, s: (_ptr(fb), _ptr(pb), _ptr(keys), n, _ptr(tb), o, s))


@pytest.mark.gpu
@pytest.mark.parametrize("n", PRODUCER_NS)
@pytest.mark.parametrize("shift", [7, 6, 4])
def test_add_ctx_embed(gpu, n, shift):
    """the encoder passes the FULL occupancy byte: the context is occ >> shift, whatever the bits below"""
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    rng = np.random.default_rng(n + shift)
    u = _table(rng, max(n, 1))[:n]
    emb = _table(rng, 256 >> shift)
    occ = rng.permutation(np.resize(np.arange(256, dtype=np.uint8), n)) if n else np.zeros(0, np.uint8)
    ub, ob, eb = _dev(codec, u.reshape(-1, 32)), _dev(codec, occ), _dev(codec, emb)
    _run_producer(gpu, "gpc_add_ctx_embed", n, lambda: ctx_ref(u.reshape(-1, 32), occ, shift, emb),
                  lambda o, s: (_ptr(ub), _ptr(ob), shift, _ptr(eb), n, o, s))


# ------------------------------------------------------------------------------------------------------------ §3 head
WORST_HEAD = {}


@pytest.mark.gpu
@pytest.mark.parametrize("A", [2, 4, 16])
@pytest.mark.parametrize("tied", [False, True])
def test_head_fp64_and_symbol_words(gpu, A, tied):
    """gpc_head_cdf probabilities within the fp64 bound; gpc_head_cdf_sym's words lohi = c_low | c_high << 16 equal (cdf[s],
    cdf[s + 1]) of gpc_head_cdf's rows (c_high == 0 for the top symbol), with cdf / prob NULL and given, and the same cdf / prob;
    occ bytes carry bits above the stage's field.  n ragged against the 128-row CTAs."""
    from gauspcc_b200.codec import _ptr
    codec = gpu["codec"]
    i = STAGE_OF_A[A]
    hw = head_weights(gpu["w"], i, tied)
    W1, b1, W2, b2 = (_dev(codec, a) for a in hw)
    st = codec._stream()
    worst = 0.0
    for n in (1, 127, 128, 129, 5003):
        f = head_rows(n, n + A)
        fd = _dev(codec, f)
        cdf = torch.full((n + 1, A + 1), 0x5A5A, dtype=torch.int16, device=codec.dev)
        prob = _sent(codec, (n + 1, A), torch.float32)
        codec._call("gpc_head_cdf", _ptr(fd), n, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), A, _ptr(cdf), _ptr(prob), st)
        p = prob.cpu().numpy()
        assert (p[n].view(np.uint32) == SENT).all() and (cdf.cpu().numpy()[n] == 0x5A5A).all(), "written past n rows"
        p64, bnd = head64(f, *hw)
        err = np.abs(p[:n] - p64)
        assert (err <= bnd).all(), (A, tied, n, float((err / bnd).max()))
        worst = max(worst, float((err / bnd).max()))
        if tied:
            assert np.array_equal(p[:n, 0], p[:n, 1])
        c = cdf.cpu().numpy()[:n].view(np.uint16).astype(np.int64)
        rng = np.random.default_rng(n)
        occ = rng.integers(0, 256, size=n).astype(np.uint8)
        occ[: min(n, 16)] = 0xFF                                   # bits above the field and the top symbol
        s = (occ.astype(np.int64) >> STAGE_SHIFT[i]) & (A - 1)
        ob = _dev(codec, occ)
        for with_bufs in (False, True):
            lohi = _sent(codec, (n + 1,))
            c2 = torch.full((n, A + 1), 0x5A5A, dtype=torch.int16, device=codec.dev) if with_bufs else None
            p2 = _sent(codec, (n, A), torch.float32) if with_bufs else None
            codec._call("gpc_head_cdf_sym", _ptr(fd), n, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), A, _ptr(ob), STAGE_SHIFT[i],
                        _ptr(lohi), _ptr(c2), _ptr(p2), st)
            w = _host_u32(lohi)
            assert w[n] == SENT
            lo, hi = (w[:n] & 0xFFFF).astype(np.int64), (w[:n] >> 16).astype(np.int64)
            r = np.arange(n)
            assert np.array_equal(lo, c[r, s]), (A, n, with_bufs)
            top = s == A - 1
            assert np.array_equal(hi[~top], c[r[~top], s[~top] + 1]) and (hi[top] == 0).all(), (A, n, with_bufs)
            if with_bufs:
                assert np.array_equal(c2.cpu().numpy(), cdf.cpu().numpy()[:n]) and np.array_equal(_host_u32(p2), p[:n].view(np.uint32))
    WORST_HEAD[(A, tied)] = worst
    print(f"\nhead A={A} tied={tied}: worst |p - p64| / bound {worst:.3g}")
    # arguments
    lib = codec.lib
    fd = _dev(codec, head_rows(8, 0))
    buf = torch.zeros(64, dtype=torch.int32, device=codec.dev)
    for bad_a in (0, 1, 3, 8, 32):
        assert lib.gpc_head_cdf(_ptr(fd), 8, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), bad_a, _ptr(buf), None, st) == GPC_EINVAL
        assert lib.gpc_head_cdf_sym(_ptr(fd), 8, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), bad_a, _ptr(buf), 0, _ptr(buf), None, None,
                                    st) == GPC_EINVAL
    assert lib.gpc_head_cdf_sym(_ptr(fd), 8, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), A, None, 0, _ptr(buf), None, None, st) == GPC_EINVAL
    assert lib.gpc_head_cdf_sym(_ptr(fd), 8, _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), A, _ptr(buf), 0, None, None, None, st) == GPC_EINVAL
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------ §4 the chain
# Position k of a conv call within one level (level_features, then the four stage_cdf calls), as oracle.py prescribes:
#   (conv index, level: parent "p" / child "c", relu, residual from position, input from position or producer, tcgen05 output)
def _prescription():
    out = []
    for base, lv, prod in ((0, "p", "embed"), (5, "c", "gather")):
        final = "f32" if lv == "p" else "both"
        out += [(base, lv, True, None, prod, "split"), (base + 1, lv, True, None, base, "split"),
                (base + 2, lv, True, base, base + 1, "split"), (base + 3, lv, True, None, base + 2, "split"),
                (base + 4, lv, True, base + 2, base + 3, final)]
    for i in range(4):
        out += [(10 + 2 * i, "c", True, None, 9 if i == 0 else "ctx", "split"), (11 + 2 * i, "c", False, None, 10 + 2 * i, "f32")]
    return out


PRESCRIBED = _prescription()
SPLIT_SLACK = 2.0 ** -17                                     # split output: hi + lo is y to within 2^-17 |y|


def _family(km):
    if km.um_rows:
        return "um"
    if km.sparse:
        return "sparse"
    return f"v6 {km.v6_variant}@{km.tile_rows}"


def _sample(n, seed):
    """every row of a small level; otherwise ~1.6 K rows: the first 64, the last 512 (the ragged last tile of every family) and
    1024 at random"""
    if n <= 4096:
        return np.arange(n)
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([np.arange(64), np.arange(n - 512, n), rng.choice(n, 1024, replace=False)]))


class ChainRecorder:
    """Wraps codec.build_kmap, level_features, conv and stage_cdf.  Every conv call is checked when it returns (after a device
    synchronise: encoder and decoder use side streams): the output on sampled rows against an fp64 conv of the call's own inputs,
    the call against its prescription, and its input / residual against the recorded outputs they must be (bit for bit, on the
    device), or against the producer restatement applied to the recorded predecessor."""

    def __init__(self, codec, w, K):
        from gauspcc_b200.weights import CONV_KEYS
        self.codec, self.w, self.K = codec, w, K
        self.W = [np.asarray(w[k], np.float64) for k in CONV_KEYS]
        self.levels = {}                                      # id(KMap) -> level record
        self.worst = {}                                       # (family, "f32" | "split" | "prob") -> worst error / bound
        self.families = set()
        self.convs = 0
        self.group = None
        self._orig = {k: getattr(codec, k) for k in ("build_kmap", "level_features", "conv", "stage_cdf")}
        codec.build_kmap, codec.level_features, codec.conv, codec.stage_cdf = (self.build_kmap, self.level_features, self.conv,
                                                                               self.stage_cdf)

    def close(self):
        for k in self._orig:
            delattr(self.codec, k)                            # back to the class's methods

    # ---- wrappers
    def build_kmap(self, keys, family=None):
        km = self._orig["build_kmap"](keys, family)
        torch.cuda.synchronize()
        from oracle import oracle as O
        k = keys.cpu().numpy()
        xyz = keys_to_xyz(k).astype(np.int32)
        n = xyz.shape[0]
        S = _sample(n, n)
        nb = O.kmap(xyz, self.K)[S]
        U, inv = np.unique(nb[nb >= 0], return_inverse=True)
        nbS = np.full(nb.shape, -1, np.int64)
        nbS[nb >= 0] = inv
        self.levels[id(km)] = dict(km=km, keys=k, xyz=xyz, n=n, S=S, S_t=torch.tensor(S, device=self.codec.dev),
                                   U_t=torch.tensor(U, device=self.codec.dev), nbS=nbS)
        return km

    def level_features(self, parent, n_child, child_kmap=None):
        torch.cuda.synchronize()
        self.group = dict(parent=parent, parent_occ=parent.occ.cpu().numpy(), outs=[], kms={})
        return self._orig["level_features"](parent, n_child, child_kmap)

    def stage_cdf(self, u, occ_partial, i, km, cdf_out, prob_out=None, lohi_out=None):
        torch.cuda.synchronize()
        g = self.group
        g["stage"], g["occ"] = i, occ_partial.cpu().numpy()
        r = self._orig["stage_cdf"](u, occ_partial, i, km, cdf_out, prob_out, lohi_out)
        torch.cuda.synchronize()
        lv = self.levels[id(km)]
        S, S_t = lv["S"], lv["S_t"]
        A = (2, 2, 4, 16)[i]
        if prob_out is not None:                              # the head on the last conv's recorded output, against fp64
            t = g["outs"][11 + 2 * i][torch.float32]
            p64, bnd = head64(t[S_t].cpu().numpy(), *head_weights(self.w, i))
            p = prob_out[S_t].cpu().numpy()
            err = np.abs(p - p64) / bnd
            assert (err <= 1).all(), ("head", i, _family(km), float(err.max()))
            self._worst(_family(km), "prob", float(err.max()))
        if lohi_out is not None and cdf_out is not None:     # the encoder's coder words are the CDF rows' entries of the symbol
            c = cdf_out[S_t].cpu().numpy().view(np.uint16).astype(np.int64)
            wv = lohi_out[S_t].cpu().numpy().view(np.uint32)
            s = (g["occ"][S].astype(np.int64) >> STAGE_SHIFT[i]) & (A - 1)
            r_ = np.arange(S.size)
            assert np.array_equal(wv & 0xFFFF, c[r_, s])
            assert np.array_equal((wv >> 16)[s < A - 1], c[r_[s < A - 1], s[s < A - 1] + 1]) and ((wv >> 16)[s == A - 1] == 0).all()
        return r

    def conv(self, x, widx, km, residual=None, relu=False, out=None, fmt="f32", rows=None):
        y = self._orig["conv"](x, widx, km, residual=residual, relu=relu, out=out, fmt=fmt, rows=rows)
        torch.cuda.synchronize()
        assert rows is None and out is None
        outs = {}
        if isinstance(y, tuple):
            outs[torch.float32], outs[torch.int32] = y
        else:
            outs[y.dtype] = y
        self._check_call(x, widx, km, residual, relu, fmt, outs)
        self.group["outs"].append({k: v.clone() for k, v in outs.items()})
        return y

    # ---- checks
    def _worst(self, fam, kind, v):
        self.worst[(fam, kind)] = max(self.worst.get((fam, kind), 0.0), v)

    def _rows64(self, t, idx_t):
        a = t[idx_t].cpu().numpy()
        return join64(a) if t.dtype == torch.int32 else a.astype(np.float64)

    def _check_call(self, x, widx, km, residual, relu, fmt, outs):
        g = self.group
        k = len(g["outs"])
        assert k < len(PRESCRIBED), "more conv calls in a level than the network has"
        pw, plv, prelu, pres, pin, pfmt = PRESCRIBED[k]
        lv = self.levels[id(km)]
        fam = _family(km)
        self.families.add(fam)
        self.convs += 1
        tag = (k, widx, fam, lv["n"])
        # prescription: conv index, level, relu, output format
        assert widx == pw and relu == prelu, tag
        if plv == "p":
            assert km is g["parent"].kmap, tag
        else:
            g["kms"].setdefault("c", km)
            assert km is g["kms"]["c"] and km is not g["parent"].kmap, tag
        assert fmt == (pfmt if km.um_rows else "f32"), (tag, fmt)
        assert x.dtype == (torch.int32 if km.um_rows else torch.float32), tag
        # wiring: residual and input are the prescribed earlier outputs, bit for bit
        if pres is None:
            assert residual is None, tag
        else:
            src = g["outs"][pres]
            assert residual.dtype in src and torch.equal(residual, src[residual.dtype]), (tag, "residual")
        S, S_t = lv["S"], lv["S_t"]
        if isinstance(pin, int):
            src = g["outs"][pin]
            assert x.dtype in src and torch.equal(x, src[x.dtype]), (tag, "input")
        else:
            self._check_producer(pin, x, lv, tag)
        # fp64 conv of this call's own inputs on the sampled rows
        x64 = self._rows64(x, lv["U_t"])
        r64 = self._rows64(residual, S_t) if residual is not None else None
        ref, absref = conv64(x64, self.W[widx], lv["nbS"], r64, relu)
        b = bound(absref)
        if torch.float32 in outs:
            yv = outs[torch.float32][S_t].cpu().numpy()
            e = np.abs(yv - ref) / b
            assert (e <= 1).all(), (tag, "f32", float(e.max()))
            self._worst(fam, "f32", float(e.max()))
        if torch.int32 in outs:
            ys = outs[torch.int32][S_t].cpu().numpy().view(np.uint32)
            bs = b + SPLIT_SLACK * (np.abs(ref) + b)
            e = np.abs(join64(ys) - ref) / bs
            assert (e <= 1).all(), (tag, "split", float(e.max()))
            self._worst(fam, "split", float(e.max()))
            if torch.float32 in outs:                          # fmt "both": ys is split_ref of y, bit for bit
                assert np.array_equal(ys, split_ref(yv)), (tag, "ys != split(y)")

    def _check_producer(self, kind, x, lv, tag):
        """x on the sampled rows against the producer restatement applied to the recorded predecessor"""
        g, w = self.group, self.w
        S, S_t = lv["S"], lv["S_t"]
        if kind == "embed":
            want = embed_ref(w["prior_embedding.weight"], g["parent_occ"][S])
        elif kind == "gather":
            plv = self.levels[id(g["parent"].kmap)]
            pk = pack_keys_ref(lv["xyz"][S] >> 1)
            parent = np.searchsorted(plv["keys"], pk)
            assert (parent < plv["n"]).all() and np.array_equal(plv["keys"][parent], pk), (tag, "a child without its parent")
            feat = g["outs"][4][torch.float32][torch.tensor(parent, device=self.codec.dev)].cpu().numpy()
            want = gather_ref(feat, np.arange(S.size), w["target_embedding.target_res_embedding.weight"], lv["xyz"][S])
        else:
            i = g["stage"]
            u = g["outs"][9][torch.float32][S_t].cpu().numpy()
            want = ctx_ref(u, g["occ"][S], CTX_SHIFT[i], w[f"pred_head_s{i}_emb.weight"])
        got = x[S_t].cpu().numpy()
        if x.dtype == torch.int32:
            assert np.array_equal(got.view(np.uint32), split_ref(want)), (tag, kind, "split")
        else:
            assert np.array_equal(got.view(np.uint32), np.ascontiguousarray(want, np.float32).view(np.uint32)), (tag, kind)


WORST_CHAIN = {}


def run_chain(codec, xyz, w, K=5):
    """teacher-forced: encode(collect=True) and a stage-by-stage decode, every conv checked as it returns; the decoder's CDF rows of
    every (level, stage) equal the encoder's; the round trip is lossless.  Returns the recorder."""
    x = torch.tensor(xyz, dtype=torch.float32, device=codec.dev)
    rec = ChainRecorder(codec, w, K)
    try:
        bx, bo, streams, aux = codec.encode(x, collect=True)
        L = len(streams) // 4
        assert rec.convs == 18 * L
        codec.wave_decode, codec.debug_dec_cdfs = False, {}
        dec = codec.decode(bx, bo, streams)
        assert rec.convs == 36 * L
        assert sorted(codec.debug_dec_cdfs) == [(d, i) for d in range(L) for i in range(4)]
        for (d, i), c in codec.debug_dec_cdfs.items():
            assert torch.equal(c, aux["cdfs"][4 * d + i]), (d, i)
        assert np.array_equal(np.unique(dec.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz, axis=0))
    finally:
        rec.close()
        codec.wave_decode, codec.debug_dec_cdfs = True, None
    for key, v in rec.worst.items():
        WORST_CHAIN[key] = max(WORST_CHAIN.get(key, 0.0), v)
    print("\n" + ", ".join(f"{f} {k} {v:.3g}" for (f, k), v in sorted(rec.worst.items())))
    torch.cuda.synchronize()
    return rec


def _codec(gpu, kind):
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict, state_dict_to_numpy
    base = gpu["codec"]
    w, K = gpu["w"], 5
    if kind == "k3":
        sd = make_synthetic_state_dict(kernel_size=3)
        codec = GausPcgcCodec(DeviceWeights(sd, gpu["dev"], kernel_size=3), gpu["dev"])
        w, K = state_dict_to_numpy(sd), 3
    elif kind == "v6d":
        codec = GausPcgcCodec(base.w, gpu["dev"], tile_rows=128)
        codec.v6_variant = 48
        codec.um_min_rows = codec.sparse_min_rows = 1 << 40
    else:
        codec = GausPcgcCodec(base.w, gpu["dev"])
    if kind == "sparse":
        codec.um_min_rows, codec.sparse_min_rows, codec.sparse_max_density = 1, 1, 1e9
    if kind in ("um", "k3"):
        codec.um_min_rows, codec.sparse_max_density = 1, 0.0
    return codec, w, K


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,seed,ext", [("default", 60_000, 2, 14), ("v6d", 20_000, 1, 16), ("sparse", 20_000, 3, 16),
                                              ("um", 20_000, 4, 16), ("k3", 12_000, 5, 12)])
def test_chain_teacher_forced(gpu, kind, n, seed, ext):
    from gauspcc_b200.synth import hac_like_cloud
    codec, w, K = _codec(gpu, kind)
    rec = run_chain(codec, hac_like_cloud(n, seed, extent_log2=ext), w, K)
    fams = rec.families
    if kind == "default":
        ran = {"v6 47@8", "v6 46@16", "v6 46@32", "v6 48@64"} & fams
        assert len(ran) >= 3, fams
    elif kind == "v6d":
        assert fams == {"v6 48@128"}, fams
    elif kind == "sparse":
        assert fams == {"sparse"}, fams
    else:
        assert fams == {"um"}, fams


@pytest.mark.gpu
def test_chain_production_scene(gpu):
    """a 400 K-anchor scene under the default thresholds: its big levels take both the tcgen05 conv (dense) and the sparse conv"""
    from gauspcc_b200.synth import hac_like_cloud
    codec, w, K = _codec(gpu, "default")
    rec = run_chain(codec, hac_like_cloud(400_000, 0), w, K)
    assert {"um", "sparse"} <= rec.families and any(f.startswith("v6 48@") for f in rec.families), rec.families
