"""The codec, its coders and the training loss on checkpoints the trainer makes, and on checkpoints pushed to the extremes.

Every other parity test runs make_synthetic_state_dict(), whose weights keep every level and stage at mid-range entropy.  A trained
checkpoint moves the network towards the low-entropy regime: probabilities near 0 and 1, u16 CDF rows with bins of width 1 next to
one of ~65 500, symbols of ~0 or ~16 bits, tiny coarse-level streams and long chunks of costly symbols.  The checkpoints here:

  trained5, trained3   train(...) on four 20 K-point HAC-like patches, 300 steps (K = 5) and 200 steps (K = 3)
  trained_codec        K = 5 with conv_families="codec" and batch_size=4 (every level on the family the codec codes it with)
  saturated8/64        trained5 with every pred_head_s{i}.2 (weight and bias: the logits) multiplied by 8 / 64
  inverted             trained5 with those logits multiplied by -8: confidently wrong.  Negating alone is not enough: after 300
                       steps the logit gaps are a few units, so the negated network would only be mildly wrong.

Each is run on a 20 K-point cloud of the training distribution; the regime it puts that cloud in is printed and guarded, so that
the checks below cannot silently fall back to mid-entropy streams.

The range coder (ac_host.cu, attr_ac.cu; torchac's): 32-bit low / high, 16-bit CDF counts.  A symbol whose bin is [c_lo, c_hi) of
65536 narrows a span S > 2^30 to floor(S c_hi / 2^16) - floor(S c_lo / 2^16), i.e. to S w / 2^16 within one, so its cost differs
from the exact -log2(w / 65536) by at most ETA = -log2(1 - 2^-14) bits (w >= 1).  Every renormalising shift doubles the span, and
the last span is in (2^30, 2^32]; the flush writes two bits more than were shifted (the last bit and one pending) and pads to a
byte.  So a stream of n symbols of exact code length E is 8 * bytes in (E - n ETA, E + 9 + n ETA]."""
import ctypes as C
import hashlib
import math
import time

import numpy as np
import pytest

from test_gpu_parity import PROB_TOL, _check_codec_vs_oracle
from test_level_network import family_codec, run_chain
from test_train import check_network_gradients

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                                 # unit roundoff of fp32
ETA = -math.log2(1.0 - 2.0 ** -14)             # bits a symbol may cost beyond its exact code length (module docstring)
FLUSH_BITS = 9                                 # 2 flush bits + up to 7 of padding
P_HIGH = 1.0 - 2.0 ** -10                      # "near-certain": coder probability w / 65536 at or above this
PATCH, TRAIN_EXT = 20_000, 13                  # 20 K-point patches of extent 2^13: the training distribution
CLOUD = (20_000, 901, TRAIN_EXT)               # (n, seed, extent_log2) of the 20 K test cloud, not a training patch
BIG = (100_000, 902, 14)                       # the 100 K oracle case (about the same density)
NAMES5 = ["trained5", "saturated8", "saturated64", "inverted", "trained_codec"]
NAMES = NAMES5 + ["trained3"]
FAMILIES = ["default", "v6d", "sparse", "um"]
CHUNK = 16384                                  # the largest chunk container version 2 allows
SCALED = {"saturated8": 8.0, "saturated64": 64.0, "inverted": -8.0}      # trained5 with its logits times these


def _scale_logits(sd, s):
    out = dict(sd)
    for i in range(4):
        for k in ("weight", "bias"):
            out[f"pred_head_s{i}.2.{k}"] = sd[f"pred_head_s{i}.2.{k}"] * s
    return out


def _sha(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()[:16]


@pytest.fixture(scope="module")
def dev():
    d = torch.device("cuda:0")
    torch.cuda.set_device(d)
    return d


@pytest.fixture(scope="module")
def ckpts(dev):
    """name -> dict(sd, K, s (the factor on trained5's logits, 1 for a trained one), w (numpy), dw, codec (default thresholds)), trained deterministically once per module"""
    from gauspcc_b200 import train as T
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import state_dict_to_numpy
    clouds = [torch.tensor(hac_like_cloud(PATCH, seed=700 + j, extent_log2=TRAIN_EXT)) for j in range(4)]
    runs = {"trained5": dict(steps=300, seed=1, kernel_size=5), "trained3": dict(steps=200, seed=2, kernel_size=3),
            "trained_codec": dict(steps=60, seed=3, kernel_size=5, batch_size=4, conv_families="codec")}
    sds = {}
    print()
    for name, kw in runs.items():
        t0 = time.time()
        sd, rows = T.train(clouds, max_points=PATCH, **kw)
        sds[name] = (sd, kw["kernel_size"])
        print(f"{name}: {kw['steps']} steps in {time.time() - t0:.1f} s, bpp {rows[0]['bpp']:.3f} -> {rows[-1]['bpp']:.3f}, "
              f"sha256 {_sha(sd)}")
    sd5 = sds["trained5"][0]
    for name, s in SCALED.items():
        sds[name] = (_scale_logits(sd5, s), 5)
    out = {}
    for name, (sd, K) in sds.items():
        dw = DeviceWeights(sd, dev, kernel_size=K)
        out[name] = dict(sd=sd, K=K, s=SCALED.get(name, 1.0), w=state_dict_to_numpy(sd), dw=dw, codec=GausPcgcCodec(dw, dev))
    return out


# ------------------------------------------------------------------------------------------------------------ helpers
def _widths(cdf, sym):
    """the coder's bin width of every symbol under u16 CDF rows [n, A + 1] (the top symbol's bin ends at 65536)"""
    c = np.asarray(cdf).view(np.uint16).astype(np.int64)
    A = c.shape[1] - 1
    r = np.arange(sym.shape[0])
    hi = np.where(sym == A - 1, 65536, c[r, np.minimum(sym + 1, A - 1)])
    return hi - c[r, sym]


def _bits(w):
    """exact code length of bins of widths w: sum of -log2(w / 65536), fp64"""
    return float(-np.log2(np.asarray(w, np.float64) / 65536.0).sum())


def _symbols(levels):
    """true symbols of every (level, stage) in stream order"""
    from oracle import oracle as O
    return [s.astype(np.int64) for lv in levels[1:] for s in O.split_symbols(lv.occ.cpu().numpy())]


def _capture_ws(codec):
    """record the workspaces codec._ws hands out; returns (list, restore)"""
    got, orig = [], codec._ws
    codec._ws = lambda nbytes: (got.append(orig(nbytes)), got[-1])[1]
    return got, lambda: delattr(codec, "_ws")


_ENC = {}


def encoded(ck, name, dev):
    """the 20 K test cloud through the checkpoint's default codec: version 1 and version 2 (chunk 16384), both collected, plus the
    status word of the chunk coder's workspace"""
    if name not in _ENC:
        from gauspcc_b200.synth import hac_like_cloud
        codec = ck["codec"]
        x = torch.tensor(hac_like_cloud(CLOUD[0], CLOUD[1], extent_log2=CLOUD[2]), dtype=torch.float32, device=dev)
        v1 = codec.encode(x, collect=True)
        ws, restore = _capture_ws(codec)
        try:
            v2 = codec.encode(x, collect=True, gpu_chunk=CHUNK)
        finally:
            restore()
        status = int(ws[-1][:4].view(torch.int32).item())
        _ENC[name] = dict(x=x, v1=v1, v2=v2, status=status, sym=_symbols(v1[3]["levels"]),
                          cdfs=[c.cpu().numpy().view(np.uint16) for c in v1[3]["cdfs"]])
    return _ENC[name]


def _chunks(codec, stream, n, chunk):
    """a version-2 stream of n symbols -> (chunk length, u16 byte counts, chunk bodies)"""
    cl = codec.chunk_len(n, chunk)
    k = (n + cl - 1) // cl
    cnt = np.frombuffer(stream, dtype="<u2", count=k).astype(np.int64)
    body = stream[2 * k:]
    assert int(cnt.sum()) == len(body)
    offs = np.concatenate([[0], np.cumsum(cnt)])
    return cl, cnt, [body[offs[c]:offs[c + 1]] for c in range(k)]


def _coder_window(E, n):
    """(lo, hi] of 8 * bytes for a stream of n symbols of exact code length E (module docstring)"""
    return E - n * ETA, E + FLUSH_BITS + n * ETA


# ------------------------------------------------------------------------------------------------------------ 1. regime
@pytest.mark.parametrize("name", NAMES)
def test_regime(ckpts, dev, name):
    """what the checkpoint does to a 20 K cloud: share of symbols with coder probability >= 1 - 2^-10, share of width-1 bins over
    all bins of all CDF rows, bits per symbol and the extreme version-2 chunk sizes.  Saturated and inverted checkpoints must be in
    the low-entropy regime; a trained one must code below the synthetic init."""
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict
    ck = ckpts[name]
    e = encoded(ck, name, dev)
    w = np.concatenate([_widths(c, s) for c, s in zip(e["cdfs"], e["sym"])])
    bins = np.concatenate([np.diff(np.concatenate([c[:, :-1].astype(np.int64), np.full((c.shape[0], 1), 65536)], 1), axis=1).ravel()
                           for c in e["cdfs"]])
    streams = e["v2"][2]
    cnts = np.concatenate([_chunks(ck["codec"], st, s.shape[0], CHUNK)[1] for st, s in zip(streams, e["sym"])])
    r = dict(p_high=float((w >= P_HIGH * 65536).mean()), w1=float((bins == 1).mean()), sym_w1=float((w == 1).mean()),
             bits_per_sym=_bits(w) / w.size, chunk_min=int(cnts.min()), chunk_max=int(cnts.max()), symbols=int(w.size))
    print(f"\n{name}: {r['symbols']} symbols, {100 * r['p_high']:.1f} % at p >= 1 - 2^-10, {100 * r['w1']:.1f} % of bins of width 1 "
          f"({100 * r['sym_w1']:.1f} % of the coded symbols in one), {r['bits_per_sym']:.3f} bits / symbol; version-2 chunks of "
          f"{r['chunk_min']} .. {r['chunk_max']} bytes")
    assert e["status"] == 0
    if name.startswith("saturated"):
        assert r["p_high"] >= 0.5 and r["w1"] >= 0.5, r
    elif name == "inverted":
        assert r["w1"] >= 0.5 and r["sym_w1"] >= 0.25 and r["bits_per_sym"] >= 4.0, r
    else:
        sd0 = make_synthetic_state_dict(5, 32, ck["K"])
        base = GausPcgcCodec(DeviceWeights(sd0, dev, kernel_size=ck["K"]), dev)
        _, _, st0, _ = base.encode(e["x"])
        assert sum(map(len, e["v1"][2])) < sum(map(len, st0)), "training did not lower the rate"


# ------------------------------------------------------------------------------------------------------------ 2. oracle parity
# The probability bar, in logs.  The 1e-3 bar is sharpest on a balanced binary row, p = (1/2, 1/2): there dp = d(L_0 - L_1) / 4, so
# it says that the two sides' logits agree to within TAU / 2 = 2e-3 each (TAU = 4 * PROB_TOL).  A checkpoint whose logits are the
# trained network's times s (saturated: 8, 64; inverted: -8) runs the same features into the same first head layer, so its logits
# carry the same differences times |s|: each within |s| TAU / 2.  ln p_k = s L_k - lse(s L), and lse moves by at most the largest
# change of its arguments, so
#     |ln p_gpu,k - ln p_ora,k| <= |s| TAU + 2^-20                                          (LOG_SLACK: fp32 rounding of p)
# for every entry both sides hold as a normal number above 2^-100; below it the entries are within 2^-99 of each other.  The bar
# does not depend on how far the two sides measure apart; for s = 1 it holds besides the 1e-3 bar, for s = 64 it replaces it: there
# a balanced row's probabilities move by |s| / 4 times the logit gap, and the absolute 1e-3 bar would demand logits 16 times closer
# than it does of the trained network itself.
#
# The code-length bar.  The oracle's CDF rows are O.cdf_u16 of the oracle's probabilities; the codec's are its head kernel's, by
# the same rule c_j = rn(clamp(C_{j-1}) (65536 - A)) + j on the fp32 cumsum C.  Given the same probabilities the two rows are
# within one step (test_gpu_parity.py::test_head_cdf).  End to end the probabilities differ as well, by at most
# d_k = (exp(|s| TAU + LOG_SLACK) - 1) p_ora,k + 2^-99 under the bar above, so entry j may differ by
#     D_j = (65536 - A) sum_{k<j} d_k + 1 + 2 (65536 - A) g_A + 2^-7
# (the probability bound, one rounding step, both cumsums' rounding, both products' rounding); entry 0 is 0 on both sides and the
# top of the last bin 65536.  Every entry is checked against D_j, and the bin of a symbol s is then within D = D_s + D_{s+1} counts
# of the oracle's: its exact code length -log2(w / 65536) differs by at most t = log2 max(w_ora / max(1, w_ora - D), (w_ora + D) /
# w_ora), so per (level, stage) |L_gpu - L_ora| <= sum over the symbols of t.  Both tolerances come from the oracle's own rows
# and the fixed logit bound.  This stays meaningful at low entropy, where the 1e-3 probability bar does not: 1e-3 is 65 counts,
# which lets a width-1 bin cost 6 bits less, while at s = 1 t is ~2e-4 bits for a near-certain symbol (w ~ 65 500).
TAU = 4 * PROB_TOL
LOG_SLACK = 2.0 ** -20
TINY = 2.0 ** -100
ORACLE = {}


def _oracle_of(name, cloud):
    return ORACLE.get((name, cloud))


def _check_stage_rows(pg, po, cg, co, sym, s, tag):
    """the log-probability bar, the per-entry CDF bound and the code-length bar of one (level, stage); returns (worst log gap /
    its bar, worst |L_gpu - L_ora| / its tolerance, entries that differ, their largest difference in counts)"""
    n, A = po.shape
    scale = 65536 - A
    bar = abs(s) * TAU + LOG_SLACK
    both = (pg >= TINY) & (po >= TINY)
    lg = np.abs(np.log(np.where(both, pg, 1.0)) - np.log(np.where(both, po, 1.0)))
    assert (lg <= bar).all(), (tag, float(lg.max()), bar)
    assert (np.abs(pg - po)[~both] <= 2 * TINY).all(), tag
    d = np.expm1(bar) * po + 2 * TINY
    D = np.zeros((n, A + 1))
    D[:, 1:A] = scale * np.cumsum(d, axis=1)[:, :A - 1] + 1 + 2 * scale * A * U / (1 - A * U) + 2.0 ** -7
    step = np.abs(cg[:, :A].astype(np.int64) - co[:, :A].astype(np.int64))
    assert (step <= D[:, :A]).all(), (tag, int(step.max()))
    wg, wo = _widths(cg, sym), _widths(co, sym)
    r = np.arange(n)
    Db = np.floor(D[r, sym] + D[r, sym + 1])
    tol = float(np.log2(np.maximum(wo / np.maximum(1, wo - Db), (wo + Db) / wo)).sum())
    gap = abs(_bits(wg) - _bits(wo))
    assert gap <= tol, (tag, gap, tol)
    return float(lg.max(initial=0)) / bar, gap / tol if tol > 0 else 0.0, int((step > 0).sum()), int(step.max(initial=0))


def _parity(ckpts, dev, name, family, cloud):
    from oracle import oracle as O
    ck = ckpts[name]
    codec = ck["codec"] if family == "default" else family_codec(ck["dw"], dev, family)
    t0 = time.time()
    # saturated64: the absolute 1e-3 bar is replaced by the log-probability bar derived from it (comment above)
    prob_tol = float("inf") if name == "saturated64" else PROB_TOL
    r = _check_codec_vs_oracle(codec, ck["w"], *cloud, K=ck["K"], oracle=_oracle_of(name, cloud), prob_tol=prob_tol)
    ORACLE[(name, cloud)] = r["oracle"]
    aux, ref = r["aux"], r["oracle"][1]
    worst_log = worst_len = 0.0
    diff = total = most = 0
    k = 0
    for lv in ref["aux"]:
        syms = O.split_symbols(lv["occ"])
        for i in range(4):
            cg = aux["cdfs"][k].cpu().numpy().view(np.uint16)
            pg = aux["probs"][k].cpu().numpy().astype(np.float64)
            wl, wc, nd, mx = _check_stage_rows(pg, lv["probs"][i].astype(np.float64), cg, lv["cdfs"][i], syms[i].astype(np.int64),
                                               ck["s"], (name, family, k))
            worst_log, worst_len = max(worst_log, wl), max(worst_len, wc)
            diff, total, most = diff + nd, total + cg[:, :-1].size, max(most, mx)
            k += 1
    print(f"\n{name} {family} {cloud[0]}: worst |p - p_oracle| {r['worst']:.2e}; log-probability gap <= {worst_log:.3f} of its bar; "
          f"code length gap <= {worst_len:.3f} of its tolerance; {diff} of {total} CDF entries differ, by at most {most}; "
          f"{r['bytes'][0]} bytes against the oracle's {r['bytes'][1]} ({time.time() - t0:.1f} s)")


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("name", NAMES)
def test_codec_vs_oracle(ckpts, dev, name, family):
    """test_gpu_parity's bars (structure bit-exact, probabilities within 1e-3, bytes within 0.5 %, decode equal to the oracle's)
    plus the code-length bar, every checkpoint, every conv family"""
    _parity(ckpts, dev, name, family, CLOUD)


def test_codec_vs_oracle_100k(ckpts, dev):
    _parity(ckpts, dev, "trained5", "default", BIG)


# ------------------------------------------------------------------------------------------------------------ 3. fp64 chain
CHAIN = [(n, kind) for n in ("trained5", "saturated64") for kind in FAMILIES] + [("trained3", "k3"), ("saturated3", "k3")]


@pytest.mark.parametrize("name,kind", CHAIN)
def test_chain_teacher_forced(ckpts, dev, name, kind):
    """test_level_network's teacher-forced chain (every conv and head of an encode and a stage-by-stage decode against fp64 within
    its bounds, decoder CDF rows == encoder CDF rows, lossless) on trained and saturated weights"""
    from gauspcc_b200.codec import DeviceWeights
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import state_dict_to_numpy
    if name == "saturated3":
        sd = _scale_logits(ckpts["trained3"]["sd"], 64.0)
        dw, w, K = DeviceWeights(sd, dev, kernel_size=3), state_dict_to_numpy(sd), 3
    else:
        dw, w, K = ckpts[name]["dw"], ckpts[name]["w"], ckpts[name]["K"]
    codec = family_codec(dw, dev, "um" if kind == "k3" else kind)
    t0 = time.time()
    # default: the 60 K cloud of test_level_network's default chain, whose levels take several mma.sync tilings
    xyz = hac_like_cloud(60_000, 2, extent_log2=14) if kind == "default" else hac_like_cloud(*CLOUD[:2], extent_log2=CLOUD[2])
    rec = run_chain(codec, xyz, w, K)
    fams = rec.families
    if kind == "default":
        assert len({"v6 47@8", "v6 46@16", "v6 46@32", "v6 48@64"} & fams) >= 3 and all(f.startswith("v6") for f in fams), fams
    elif kind == "v6d":
        assert fams == {"v6 48@128"}, fams
    elif kind in ("sparse", "um"):
        assert fams == {kind}, fams
    elif kind == "k3":
        assert fams == {"um"}, fams
    worst = {}
    for (_, what), v in rec.worst.items():
        worst[what] = max(worst.get(what, 0.0), v)
    print(f"{name} {kind}: families {sorted(fams)}; worst error / fp64 bound " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(worst.items()))
          + f" ({time.time() - t0:.1f} s)")


# ------------------------------------------------------------------------------------------------------------ 4. coders
def _decode_in_pieces(lib, cdf, stream, n):
    """the host range decoder fed a stream's CDF rows in pieces of 1, 7, 64, 1000 rows, then the rest"""
    from gauspcc_b200 import _lib
    state = (C.c_char * int(lib.gpc_ac_decode_state_bytes()))()
    buf = (C.c_char * max(len(stream), 1)).from_buffer_copy(stream if stream else b"\0")
    _lib.check(lib.gpc_ac_decode_begin_h(C.cast(state, C.c_void_p), C.cast(buf, C.c_void_p), len(stream)), "gpc_ac_decode_begin_h")
    out = np.full(n, 0xFF, np.uint8)
    cdf = np.ascontiguousarray(cdf)
    a = 0
    for size in (1, 7, 64, 1000, n):
        b = min(n, a + size)
        if b > a:
            _lib.check(lib.gpc_ac_decode_more_h(C.cast(state, C.c_void_p), cdf[a:].ctypes.data_as(C.c_void_p), b - a, cdf.shape[1],
                                                out[a:].ctypes.data_as(C.c_void_p)), "gpc_ac_decode_more_h")
        a = b
    return out


@pytest.mark.parametrize("name", NAMES)
def test_v1_streams(ckpts, dev, name):
    """every stream of the drop-in file bit-exact against the oracle's range coder on the encoder's own CDF rows, its bytes within
    the coder's window around the exact code length, and the host decoder, fed in pieces, gives the symbols back"""
    from oracle import oracle as O
    e = encoded(ckpts[name], name, dev)
    lib = ckpts[name]["codec"].lib
    streams = e["v1"][2]
    E_all, bytes_all = 0.0, 0
    for k, (st, cdf, sym) in enumerate(zip(streams, e["cdfs"], e["sym"])):
        assert st == O.ac_encode(cdf, sym.astype(np.int16)), (name, k)
        E = _bits(_widths(cdf, sym))
        lo, hi = _coder_window(E, sym.shape[0])
        assert lo < 8 * len(st) <= hi, (name, k, 8 * len(st), E)
        assert np.array_equal(_decode_in_pieces(lib, cdf, st, sym.shape[0]), sym), (name, k)
        E_all += E
        bytes_all += len(st)
    print(f"\n{name}: {len(streams)} streams, exact {E_all:.0f} bits, streams {8 * bytes_all} bits ({8 * bytes_all - E_all:+.0f}: "
          f"{(8 * bytes_all - E_all) / len(streams):.2f} bits per stream)")


@pytest.mark.parametrize("name", NAMES)
def test_v2_every_chunk(ckpts, dev, name):
    """every chunk of every stream of the version-2 encode (chunk 16384, so chunk_len's short chunks on every level) bit-exact
    against the oracle's range coder, inside the coder's window, and the version-2 decode equal to the drop-in decode"""
    from oracle import oracle as O
    ck = ckpts[name]
    codec = ck["codec"]
    e = encoded(ck, name, dev)
    bx, bo, streams, aux = e["v2"]
    assert np.array_equal(bx, e["v1"][0]) and np.array_equal(bo, e["v1"][1])
    sizes = []
    for k, (st, sym) in enumerate(zip(streams, e["sym"])):
        cdf = aux["cdfs"][k].cpu().numpy().view(np.uint16)
        assert np.array_equal(cdf, e["cdfs"][k])
        cl, cnt, bodies = _chunks(codec, st, sym.shape[0], CHUNK)
        for c, body in enumerate(bodies):
            rows = slice(c * cl, (c + 1) * cl)
            assert body == O.ac_encode(cdf[rows], sym[rows].astype(np.int16)), (name, k, c)
            lo, hi = _coder_window(_bits(_widths(cdf[rows], sym[rows])), sym[rows].shape[0])
            assert lo < 8 * len(body) <= hi, (name, k, c)
        sizes += cnt.tolist()
    dec = codec.decode(bx, bo, streams, gpu_chunk=CHUNK)
    assert torch.equal(dec, codec.decode(*e["v1"][:3]))
    print(f"\n{name}: {len(sizes)} chunks of {min(sizes)} .. {max(sizes)} bytes, {sum(s <= 2 for s in sizes)} of at most 2 bytes")
    if name.startswith("trained"):
        assert min(sizes) <= 2                  # chunks of near-free symbols (saturated ones pay 16 bits for each miss)


def test_largest_chunk_constructed(ckpts, dev):
    """a 16 384-symbol chunk (the most container version 2 allows) of width-1 bins only, bottom, top (c_high = 0x10000, written as
    0) and anywhere between: 16 bits a symbol, so 32 768 bytes and a few.  Bit-exact against the oracle coder, byte count within
    the u16 field, the workspace's overflow flag clear, and gpc_chunk_decode_u16 gives the symbols back."""
    from gauspcc_b200.codec import _ptr
    from oracle import oracle as O
    codec = ckpts["trained5"]["codec"]
    n, A = CHUNK, 16
    rng = np.random.default_rng(16384)
    s = rng.integers(0, A, n)
    s[:64], s[64:128] = A - 1, 0
    c_lo = rng.integers(s, 65536 - (A - 1 - s))
    c_lo[s == A - 1] = 65535
    k = np.arange(A)[None, :]
    rows = np.zeros((n, A + 1), np.int64)
    rows[:, :A] = np.where(k < s[:, None], k, c_lo[:, None] + (k - s[:, None]))
    assert (np.diff(rows[:, :A], axis=1) >= 1).all() and rows[:, :A].max() <= 65535
    cdf = rows.astype(np.uint16)
    assert (_widths(cdf, s) == 1).all()
    c_hi = np.where(s == A - 1, 0, c_lo + 1)
    lohi = (c_lo | (c_hi << 16)).astype(np.uint32)
    want = O.ac_encode(cdf, s.astype(np.int16))
    lohi_d = torch.tensor(lohi.view(np.int32), device=dev)
    starts = torch.tensor([0, n], dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    offs = torch.zeros(2, dtype=torch.int32, device=dev)
    ws_b = codec.lib.gpc_chunk_workspace_bytes(1, n)
    ws = torch.full((ws_b,), 0x55, dtype=torch.uint8, device=dev)
    codec._call("gpc_chunk_encode_lohi", _ptr(lohi_d), _ptr(starts), 1, n, _ptr(cnt), _ptr(offs), _ptr(ws), ws_b, codec._stream())
    nb = int(cnt.item())
    assert int(ws[:4].view(torch.int32).item()) == 0, "chunk coder overflow flag set"
    assert nb == len(want) <= 0xFFFF and int(offs[1].item()) == nb
    lo, hi = _coder_window(16.0 * n, n)
    assert lo < 8 * nb <= hi
    out = torch.zeros(nb + 64, dtype=torch.uint8, device=dev)
    codec._call("gpc_chunk_merge", _ptr(ws), 1, n, _ptr(offs), _ptr(out), codec._stream())
    assert out[:nb].cpu().numpy().tobytes() == want
    cdf_d = torch.tensor(cdf.view(np.int16), device=dev)
    sym_d = torch.full((n,), 0xFF, dtype=torch.uint8, device=dev)
    codec._call("gpc_chunk_decode_u16", _ptr(cdf_d), _ptr(out), _ptr(offs), n, A + 1, n, _ptr(sym_d), codec._stream())
    assert np.array_equal(sym_d.cpu().numpy(), s)
    print(f"\nconstructed 16384-symbol chunk of width-1 bins: {nb} bytes")


def test_longest_real_chunk(ckpts, dev, tmp_path):
    """the inverted checkpoint on a 100 K cloud at gpu_coder_chunk=16384: its longest chunk is within the u16 field with the
    overflow flag clear and bit-exact against the oracle coder, and the version-2 file round-trips to the drop-in decode"""
    from gauspcc_b200 import bitstream, pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    from oracle import oracle as O
    ck = ckpts["inverted"]
    codec = ck["codec"]
    xyz = hac_like_cloud(BIG[0], BIG[1], extent_log2=BIG[2])
    x = torch.tensor(xyz, dtype=torch.float32, device=dev)
    ws, restore = _capture_ws(codec)
    try:
        bx, bo, streams, aux = codec.encode(x, collect=True, gpu_chunk=CHUNK)
    finally:
        restore()
    assert int(ws[-1][:4].view(torch.int32).item()) == 0, "chunk coder overflow flag set"
    sym = _symbols(aux["levels"])
    best = (0, None)
    for k, (st, s) in enumerate(zip(streams, sym)):
        cl, cnt, bodies = _chunks(codec, st, s.shape[0], CHUNK)
        c = int(np.argmax(cnt))
        if cnt[c] > best[0]:
            best = (int(cnt[c]), (k, c, cl, bodies[c]))
    nb, (k, c, cl, body) = best
    cdf = aux["cdfs"][k].cpu().numpy().view(np.uint16)
    rows = slice(c * cl, (c + 1) * cl)
    assert nb <= 0xFFFF and body == O.ac_encode(cdf[rows], sym[k][rows].astype(np.int16))
    ckpt = str(tmp_path / "inverted.pth")
    torch.save(ck["sd"], ckpt)
    r2 = pcc_utils.compress_point_cloud(x, ckpt, str(tmp_path / "v2" / "xyz_pcc.bin"), gpu_coder_chunk=CHUNK)
    r1 = pcc_utils.compress_point_cloud(x, ckpt, str(tmp_path / "v1" / "xyz_pcc.bin"))
    _, _, _, st2 = bitstream.read_file(open(r2["output_path"], "rb").read())
    assert bitstream.split_v2(st2)[0] == streams
    d2 = pcc_utils.decompress_point_cloud(r2["output_path"], ckpt)["point_cloud"]
    d1 = pcc_utils.decompress_point_cloud(r1["output_path"], ckpt)["point_cloud"]
    assert torch.equal(d1, d2)
    assert np.array_equal(np.unique(d2.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz, axis=0))
    print(f"\ninverted, 100 K: longest chunk {nb} bytes ({cl} symbols, {8 * nb / cl:.2f} bits each), stream {k}; "
          f"version 2 {r2['file_size_bits']} bits against version 1 {r1['file_size_bits']}")


@pytest.mark.parametrize("name,chunk", [("trained5", 0), ("trained5", 2048), ("saturated64", 2048), ("inverted", 0),
                                        ("trained3", 2048)])
def test_batch_codecs(ckpts, dev, tmp_path, name, chunk):
    """compress_point_clouds / decompress_point_clouds: the same bytes as one call per file, and the same rows back, losslessly"""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.synth import hac_like_cloud
    ck = ckpts[name]
    ckpt = str(tmp_path / f"{name}.pth")
    torch.save(ck["sd"], ckpt)
    clouds = [hac_like_cloud(n, seed, extent_log2=TRAIN_EXT) for n, seed in ((20_000, 911), (6_000, 912), (40_000, 913))]
    xs = [torch.tensor(c, dtype=torch.float32, device=dev) for c in clouds]
    one = [pcc_utils.compress_point_cloud(x, ckpt, str(tmp_path / "one" / f"{j}.bin"), kernel_size=ck["K"], gpu_coder_chunk=chunk)
           for j, x in enumerate(xs)]
    many = pcc_utils.compress_point_clouds(xs, ckpt, [str(tmp_path / "many" / f"{j}.bin") for j in range(len(xs))],
                                           kernel_size=ck["K"], gpu_coder_chunk=chunk)
    for a, b in zip(one, many):
        assert open(a["output_path"], "rb").read() == open(b["output_path"], "rb").read()
    decs = pcc_utils.decompress_point_clouds([b["output_path"] for b in many], ckpt, kernel_size=ck["K"])
    for c, a, d in zip(clouds, one, decs):
        single = pcc_utils.decompress_point_cloud(a["output_path"], ckpt, kernel_size=ck["K"])["point_cloud"]
        assert torch.equal(d["point_cloud"], single)
        assert np.array_equal(np.unique(single.cpu().numpy().astype(np.int32), axis=0), np.unique(c, axis=0))


# ------------------------------------------------------------------------------------------------------------ 5. the loss
# Surrogate against exact.  The network's loss charges a symbol -log2(q / 65536) with q = p_net (65536 - A) + 1; the file charges
# -log2(w / 65536) with w the bin width of the codec's CDF row.  The head kernel makes entry j (1 <= j < A) of a row from its own
# fp32 probabilities p (collect=True's) as c_j = rn(fl(clamp(C_{j-1}) (65536 - A))) + j, with C the sequential fp32 cumsum.  With
# G_{j-1} = sum_{k<j} p_k exactly, |C_{j-1} - G_{j-1}| <= g_A G_{j-1} (g_n = n u / (1 - n u)), clamping adds at most
# max(0, G_{j-1} - 1), the product rounds by < 2^-8 and the rounding to an integer by <= 1/2:
#     |c_j - (G_{j-1} (65536 - A) + j)| <= e_j = 1/2 + 2^-8 + (65536 - A) (g_A G_{j-1} + max(0, G_{j-1} - 1)),   e_0 = 0.
# So a symbol s < A - 1 has |w - (p_s (65536 - A) + 1)| <= e_s + e_{s+1}: the numerator off by at most one count plus the cumsum
# error; the top symbol's bin ends at 65536 exactly, so |w - (p_s (65536 - A) + 1)| <= e_s + (65536 - A) |1 - G_{A-1}|.  The
# network's own p adds (65536 - A) |p_net - p|.  With D_s the sum, |log2 w - log2 q| <= log2(1 + D_s / min(w, q)), summed over the
# symbols.  The network sums its fp32 terms (each within 3u + 4u |t| of the fp64 one: two roundings into q, log2 within 2 ulp)
# per stage (within g_n of the sum of |t|) and then over the stages (g_stages).
def _surrogate_bound(p, p_net, cdf, sym):
    """(exact bits E, fp64 surrogate S of p_net, rigorous bound on |E - S|)"""
    n, A = p.shape
    scale = 65536 - A
    p64 = p.astype(np.float64)
    G = np.cumsum(p64, axis=1)
    gam = A * U / (1 - A * U)
    Gj = G[:, :A - 1]
    e = np.concatenate([np.zeros((n, 1)), 0.5 + 2.0 ** -8 + scale * (gam * Gj + np.maximum(Gj - 1.0, 0.0))], axis=1)
    r = np.arange(n)
    top = sym == A - 1
    D = e[r, sym] + np.where(top, scale * np.abs(1.0 - G[:, A - 1]), e[r, np.minimum(sym + 1, A - 1)])
    D = D + scale * np.abs(p_net[r, sym].astype(np.float64) - p64[r, sym])
    w = _widths(cdf, sym).astype(np.float64)
    q = p_net[r, sym].astype(np.float64) * scale + 1.0
    S = float(-np.log2(q / 65536.0).sum())
    return _bits(w), S, float(np.log2(1.0 + D / np.minimum(w, q)).sum())


@pytest.mark.parametrize("name", ["trained5", "trained3"])
def test_loss_against_the_coder(ckpts, dev, name):
    """GausPcgcNet's probabilities equal the encoder's within 2e-6; its loss is the exact code length of the codec's CDF rows
    within the derived rounding bound; the stream bytes are the exact code length within the coder's window"""
    from gauspcc_b200 import bitstream
    from gauspcc_b200 import train as T
    ck = ckpts[name]
    e = encoded(ck, name, dev)
    net = T.GausPcgcNet(ck["K"], state_dict=ck["sd"]).to(dev)
    with torch.no_grad():
        out = net(e["x"].to(torch.int32), collect=True)
    aux = e["v1"][3]
    assert len(out["probs"]) == len(aux["probs"]) == len(e["sym"])
    worst = max(float((a - b).abs().max()) for a, b in zip(out["probs"], aux["probs"]))
    assert worst <= 2e-6, worst
    E = S = bound = fp32_bound = 0.0
    for pn, pc, cdf, sym in zip(out["probs"], aux["probs"], e["cdfs"], e["sym"]):
        Ek, Sk, bk = _surrogate_bound(pc.cpu().numpy(), pn.cpu().numpy(), cdf, sym)
        assert abs(Ek - Sk) <= bk, (Ek, Sk, bk)
        n = sym.shape[0]
        fp32_bound += 3 * U * n + (4 * U + n * U / (1 - n * U)) * Sk
        E, S, bound = E + Ek, S + Sk, bound + bk
    m = len(e["sym"])
    fp32_bound = fp32_bound * (1 + 2 * m * U) + m * U / (1 - m * U) * S
    bits = float(out["bits"])
    assert abs(bits - S) <= fp32_bound, (bits, S, fp32_bound)
    assert abs(E - S) <= bound
    streams = e["v1"][2]
    sb = 8 * sum(len(s) for s in streams)
    n_sym = sum(s.shape[0] for s in e["sym"])
    assert E - n_sym * ETA < sb <= E + FLUSH_BITS * len(streams) + n_sym * ETA       # the coder's window, stream by stream
    fb = 8 * len(bitstream.write_file(1, *e["v1"][:3]))
    print(f"\n{name}: worst |p_net - p_codec| {worst:.1e}; loss {bits:.1f} bits, fp64 surrogate {S:.1f}, exact {E:.1f} "
          f"(|exact - surrogate| {abs(E - S):.1f} <= bound {bound:.1f}), streams {sb}, file {fb}; loss / exact - 1 "
          f"{100 * (bits / E - 1):+.3f} %, streams / exact - 1 {100 * (sb / E - 1):+.3f} %, file / loss - 1 {100 * (fb / bits - 1):+.3f} %")


@pytest.mark.parametrize("name", ["trained5", "trained3"])
def test_whole_network_gradients_against_fp64(ckpts, dev, name, monkeypatch):
    """test_train's fp64 check of the loss and every parameter's gradient, on trained weights (5 K points of the training
    distribution)"""
    from gauspcc_b200 import train as T
    from gauspcc_b200.synth import hac_like_cloud
    ck = ckpts[name]
    net = T.GausPcgcNet(ck["K"], state_dict=ck["sd"]).to(dev)
    check_network_gradients(net, torch.tensor(hac_like_cloud(5_000, seed=21, extent_log2=TRAIN_EXT - 1), device=dev), monkeypatch,
                            tag=f"{name}: ")
