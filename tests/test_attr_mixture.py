"""HAC++'s mixture coder (encoder_gaussian_mixed[_chunk] / decoder_gaussian_mixed[_chunk], HAC/utils/encodings_cuda.py:178-314)
and the Bernoulli mask coder (encoder / decoder, :435-500) without a per-symbol CDF table: arithmetic.mixture_* / row_* against
the table sequence the reference runs (calculate_cdf per component, `* prob`, summed in list order, clamped, then
arithmetic_encode / arithmetic_decode), restated here on the library's table entry points (pinned to the reference extension by
tests/golden/attr_golden.npz) and, when oracle/_ref/arithmetic.so was built, on the reference extension itself.  Streams, per-chunk
byte counts and `.b` files must be identical, and decodes exact."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 10000                                                               # encodings_cuda.py:6
QS = np.array([0.25, 0.5, 1.0], np.float32)


# ------------------------------------------------------------------------------------------------ CPU
def test_declared_in_header_and_binding():
    from gauspcc_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gpcgc.h")).read()
    for n in ["gpc_mixture_encode", "gpc_mixture_decode", "gpc_row_encode", "gpc_row_decode"]:
        assert n in _lib.SIGNATURES and n + "(" in hdr


def test_python_signatures():
    import inspect
    from gauspcc_b200 import arithmetic
    for fn, args in [("mixture_encode", ["sym", "mean", "scale", "prob", "Q", "min_value", "max_value", "chunk_size"]),
                     ("mixture_decode", ["mean", "scale", "prob", "Q", "in_cache_all", "in_cnt_all", "min_value", "max_value",
                                         "chunk_size"]),
                     ("row_encode", ["sym", "row", "chunk_size"]),
                     ("row_decode", ["row", "in_cache_all", "in_cnt_all", "N", "chunk_size"])]:
        assert list(inspect.signature(getattr(arithmetic, fn)).parameters) == args


def test_fused_mixture_routing():
    import torch
    from gauspcc_b200.encodings_cuda import _takes_fused_mixture as fused
    n = 7
    v = [torch.zeros(n) for _ in range(5)]
    probs = torch.softmax(torch.zeros(n, 3), 1)
    assert fused(n, v[:1], v[:1], v[:1]) and fused(n, v[:4], v[:4], v[:4])
    assert fused(n, v[:3], v[:3], [probs[:, k] for k in range(3)])                     # strided columns
    for dt in (torch.float16, torch.bfloat16):
        assert fused(n, v[:2], v[:2], [t.to(dt) for t in v[:2]])
    assert not fused(n, v, v, v)                                                        # K = 5
    assert not fused(n, [], [], [])
    assert not fused(n, v[:2], v[:2], [v[0], v[1].double()])                           # float64 prob: the table path's error
    assert not fused(n, v[:2], v[:2], [v[0], torch.zeros(1)])                          # a broadcasting prob
    assert not fused(n, v[:2], v[:2], [v[0], v[1].view(n, 1)])
    assert not fused(n, v[:2], [v[0], torch.zeros(n + 1)], v[:2])
    assert not fused(n, v[:2], v[:1], v[:2])                                           # lists of different lengths
    assert not fused(n + 1, v[:2], v[:2], v[:2])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ref_ext():
    from oracle import build_ref_arithmetic
    return build_ref_arithmetic.load_module()                               # None unless built (GPC_REFERENCE_ROOT at build time)


def _mix_case(n, K, seed, apart=20, per_symbol_q=True, prob_dtype=None, same=False):
    """Inputs of a K-component mixture: component means `apart` bins to either side of a common centre (so symbols drawn from a
    minor component land below or above the decoder's window around the major one), a clamped (1e-12) and a very wide scale on
    some rows, probs as the strided columns of a softmax [n, K], x drawn from a component chosen by those probs."""
    import torch
    rng = np.random.default_rng(seed)
    Q = rng.choice(QS, n) if per_symbol_q else np.full(n, 0.5, np.float32)
    centre = rng.normal(0, 3, n).astype(np.float32)
    off = (np.arange(K) - (K - 1) / 2) * 2 * apart
    means = [(centre + off[k] * Q).astype(np.float32) for k in range(K)]
    scales = []
    for k in range(K):
        s = (np.abs(rng.normal(1, 0.5, n)) + 0.05).astype(np.float32) * Q
        s[k::7] = 1e-12                                                     # clamped to 1e-9 (arithmetic_kernel.cu:22)
        s[(k + 3)::11] *= 40
        scales.append(s.astype(np.float32))
    logits = torch.tensor(rng.normal(0, 1.5, (n, K)).astype(np.float32), device="cuda")
    probs = torch.softmax(logits.to(prob_dtype) if prob_dtype is not None else logits, 1)
    comp = torch.multinomial(probs.float(), 1, generator=torch.Generator(device="cuda").manual_seed(seed)).view(-1).cpu().numpy()
    pick = np.arange(n)
    m, s = np.stack(means)[comp, pick], np.stack(scales)[comp, pick]
    x = (m + np.minimum(s, 3 * Q) * rng.normal(size=n)).astype(np.float32)
    if same:
        x[:] = x[0]                                                         # one symbol value: Lp = 2
    dev = lambda a: torch.tensor(a, device="cuda")                          # noqa: E731
    return dev(x), [dev(a) for a in means], [dev(a) for a in scales], [probs[:, k] for k in range(K)], dev(Q.astype(np.float32))


def _table(ext, means, scales, probs, Q, mn, mx):
    """encodings_cuda.py:211-226 on `ext`'s calculate_cdf"""
    import torch
    lower = ext.calculate_cdf(means[0], scales[0], Q, mn, mx) * probs[0].unsqueeze(-1)
    for m, s, p in zip(means[1:], scales[1:], probs[1:]):
        lower += ext.calculate_cdf(m, s, Q, mn, mx) * p.unsqueeze(-1)
    return torch.clamp(lower, min=0.0, max=1.0)


def _check_streams(x, means, scales, probs, Q, ref_ext):
    """fused stream == table stream byte for byte, and both decoders give the symbols back; returns (sym, Lp)"""
    import torch
    from gauspcc_b200 import arithmetic as A
    xi = torch.round(x / Q)
    mn, mx = int(xi.min()), int(xi.max())
    Lp = mx - mn + 2
    sym = (xi - mn).to(torch.int16)
    n = sym.numel()
    lower = _table(A, means, scales, probs, Q, mn, mx)
    t_stream, t_cnt = A.arithmetic_encode(sym, lower, CHUNK, n, Lp)
    M, S, P = (torch.stack([t.float() for t in ts]) for ts in (means, scales, probs))
    f_stream, f_cnt = A.mixture_encode(sym, M, S, P, Q, mn, mx, CHUNK)
    assert torch.equal(f_cnt, t_cnt) and torch.equal(f_stream, t_stream)
    assert torch.equal(A.mixture_decode(M, S, P, Q, f_stream, f_cnt, mn, mx, CHUNK), sym)
    assert torch.equal(A.arithmetic_decode(lower, f_stream, f_cnt, CHUNK, n, Lp), sym)
    if ref_ext is not None:
        r_lower = _table(ref_ext, means, scales, probs, Q, mn, mx)
        assert torch.equal(r_lower, lower)
        r_stream, r_cnt = ref_ext.arithmetic_encode(sym, r_lower, CHUNK, n, Lp)
        assert torch.equal(r_cnt, f_cnt) and torch.equal(r_stream, f_stream)
    return sym, Lp


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 9999, 10001, 123457])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_mixture_stream_matches_table(K, n, ref_ext):
    x, means, scales, probs, Q = _mix_case(n, K, seed=10 * K + n % 7, per_symbol_q=n % 2 == 1)
    sym, Lp = _check_streams(x, means, scales, probs, Q, ref_ext)
    if K > 1 and n > 1000:
        # the bimodal input reaches below, inside and above the window of 32 candidates around the major component's mean
        import torch
        P = torch.stack(probs)
        major = torch.stack(means).gather(0, P.argmax(0, keepdim=True)).view(-1)
        xi = torch.round(x / Q)
        centre = torch.round(major / Q) - xi.min()
        d = sym.float() - centre
        assert (d < -16).any() and (d > 16).any() and (d.abs() <= 15).any()


@pytest.mark.gpu
def test_mixture_edge_alphabets_and_half_probs(ref_ext):
    # Lp = 2: every symbol equal
    x, means, scales, probs, Q = _mix_case(9999, 2, seed=1, per_symbol_q=False, same=True)
    assert _check_streams(x, means, scales, probs, Q, ref_ext)[1] == 2
    # Lp in the thousands: components 1500 bins apart
    x, means, scales, probs, Q = _mix_case(10001, 3, seed=2, apart=1500)
    assert _check_streams(x, means, scales, probs, Q, ref_ext)[1] > 3000
    # float16 probs (the table path promotes them to float32 in `lower * prob`)
    import torch
    x, means, scales, probs, Q = _mix_case(10001, 3, seed=3, prob_dtype=torch.float16)
    assert probs[0].dtype == torch.float16
    _check_streams(x, means, scales, probs, Q, ref_ext)


def _files(tmp_path, prefix):
    return {p.name: p.read_bytes() for p in sorted(tmp_path.iterdir()) if p.name.startswith(prefix)}


@pytest.mark.gpu
@pytest.mark.parametrize("K,scalar_q,half", [(1, True, False), (2, False, False), (3, True, True), (4, False, False)])
def test_mixed_chunk_files_match_table_path(K, scalar_q, half, tmp_path, monkeypatch):
    import torch
    from gauspcc_b200 import encodings_cuda as E
    n = 34567
    x, means, scales, probs, Q = _mix_case(n, K, seed=40 + K, per_symbol_q=not scalar_q, prob_dtype=torch.float16 if half else None)
    q = 0.5 if scalar_q else Q
    bits = E.encoder_gaussian_mixed_chunk(x, means, scales, probs, q, file_name=str(tmp_path / "fused.b"), chunk_size=15000)
    fused = _files(tmp_path, "fused_")
    assert list(fused) == ["fused_0.b", "fused_1.b", "fused_2.b"] and bits == 8 * sum(map(len, fused.values()))
    back = E.decoder_gaussian_mixed_chunk(means, scales, probs, q, file_name=str(tmp_path / "fused.b"), chunk_size=15000)
    assert torch.equal(back, torch.round(x / q) * q)
    with monkeypatch.context() as mp:                                       # the table sequence (_mixed_lower + table coder)
        mp.setattr(E, "_takes_fused_mixture", lambda *a: False)
        E.encoder_gaussian_mixed_chunk(x, means, scales, probs, q, file_name=str(tmp_path / "table.b"), chunk_size=15000)
        table_back = E.decoder_gaussian_mixed_chunk(means, scales, probs, q, file_name=str(tmp_path / "table.b"), chunk_size=15000)
    assert list(fused.values()) == list(_files(tmp_path, "table_").values())
    assert torch.equal(table_back, back)


@pytest.mark.gpu
def test_mixed_outside_fused_path_unchanged(tmp_path):
    import torch
    from gauspcc_b200 import encodings_cuda as E
    n = 12345
    x, means, scales, probs, Q = _mix_case(n, 5, seed=7)                   # K = 5: the table path, round trip as before
    f = str(tmp_path / "k5.b")
    E.encoder_gaussian_mixed(x, means, scales, probs, Q, file_name=f)
    assert torch.equal(E.decoder_gaussian_mixed(means, scales, probs, Q, file_name=f), torch.round(x / Q) * Q)
    x, means, scales, probs, Q = _mix_case(n, 2, seed=8)
    with pytest.raises(RuntimeError):                                       # a float64 first prob: a float64 table, refused by the coder
        E.encoder_gaussian_mixed(x, means, scales, [probs[0].double(), probs[1]], Q, file_name=str(tmp_path / "f64.b"))
    # a float64 later prob: `lower_all += lower` rounds into the float32 table, a sum the fused path does not restate
    p64 = [probs[0], probs[1].double()]
    E.encoder_gaussian_mixed(x, means, scales, p64, Q, file_name=f)
    assert torch.equal(E.decoder_gaussian_mixed(means, scales, p64, Q, file_name=f), torch.round(x / Q) * Q)


def _old_bernoulli_file(E, A, x, file_name):
    """encodings_cuda.py:435-467 with its [n, 3] table"""
    import torch
    x = x.detach().view(-1)
    prob_1 = (x.sum() / x.numel()).to(torch.float32)
    p = torch.zeros(x.numel(), dtype=torch.float32, device=x.device)
    p[...] = prob_1
    p_u = 1 - p.unsqueeze(-1)
    cdf = torch.cat([torch.zeros_like(p_u), p_u, torch.ones_like(p_u)], dim=-1)
    stream, cnt = A.arithmetic_encode(torch.floor(x).to(torch.int16), cdf, CHUNK, x.numel(), 3)
    return E._write(file_name, [prob_1.cpu().numpy().tobytes()], cnt, stream)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["p0.3", "zeros", "ones"])
def test_bernoulli_mask_files_match_table_path(kind, tmp_path):
    import torch
    from gauspcc_b200 import arithmetic as A, encodings_cuda as E
    n = 34567
    g = torch.Generator(device="cuda").manual_seed(5)
    mask = {"p0.3": (torch.rand(n, device="cuda", generator=g) < 0.3).float(), "zeros": torch.zeros(n, device="cuda"),
            "ones": torch.ones(n, device="cuda")}[kind]
    new, old = str(tmp_path / "new.b"), str(tmp_path / "old.b")
    bits = E.encoder(mask, file_name=new)
    assert bits == _old_bernoulli_file(E, A, mask, old)
    assert open(new, "rb").read() == open(old, "rb").read()
    assert torch.equal(E.decoder(n, new).to(torch.float32), mask)


@pytest.mark.gpu
def test_mixture_errors_and_truncated_stream():
    import torch
    from gauspcc_b200 import arithmetic as A
    from gauspcc_b200._lib import GpcError
    n = 64
    x, means, scales, probs, Q = _mix_case(n, 2, seed=11)
    xi = torch.round(x / Q)
    mn, mx = int(xi.min()), int(xi.max())
    sym = (xi - mn).to(torch.int16)
    for K in (0, 5):
        M = torch.zeros(K, n, device="cuda")
        with pytest.raises(GpcError):
            A.mixture_encode(sym, M, M + 1, M, Q, mn, mx, 16)
        with pytest.raises(GpcError):
            A.mixture_decode(M, M + 1, M, Q, torch.zeros(4, dtype=torch.uint8, device="cuda"),
                             torch.ones(4, dtype=torch.int32, device="cuda"), mn, mx, 16)
    M, S, P = (torch.stack(ts).float() for ts in (means, scales, probs))
    stream, cnt = A.mixture_encode(sym, M, S, P, Q, mn, mx, 16)
    assert torch.equal(A.mixture_decode(M, S, P, Q, stream, cnt, mn, mx, 16), sym)
    # a truncated stream decodes to garbage of the right length, without hanging or faulting
    out = A.mixture_decode(M, S, P, Q, stream[:1], torch.tensor([1, 0, 0, 0], dtype=torch.int32, device="cuda"), mn, mx, 16)
    assert out.shape == (n,)
