"""SURVEY 8f-4: HAC's chunked attribute coder (HAC/submodules/arithmetic.zip!arithmetic/arithmetic_kernel.cu, callers
HAC/utils/encodings_cuda.py:317-500) -- the library's kernels (csrc/attr_ac.cu) behind gauspcc_b200.arithmetic /
gauspcc_b200.encodings_cuda against the CPU oracle, against the stored tables and streams of tests/golden/attr_golden.npz
(tests/golden/make_attr_golden.py says where they come from) and, when oracle/_ref/arithmetic.so was built from the reference's
own sources (GPC_REFERENCE_ROOT at build time), against the reference extension itself on the same GPU: bytes, per-chunk counts
and decoded symbols must be identical."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 10000                                                               # encodings_cuda.py:6
CASES = [(1, 0, False), (9999, 1, False), (10000, 2, False), (10001, 3, True), (123457, 4, True)]       # n, seed, tiny_scale


def _case(n, seed, q=0.5, spread=3.0, tiny_scale=False):
    rng = np.random.default_rng(seed)
    mean = rng.normal(0, spread, n).astype(np.float32)
    scale = (np.abs(rng.normal(1, 0.5, n)) + 0.05).astype(np.float32)
    if tiny_scale:
        scale[::7] = 1e-12                                                  # clamped to 1e-9 (arithmetic_kernel.cu:22)
        scale[1::11] *= 40                                                  # and very wide rows: the decoder's search leaves its window
    Q = np.full(n, q, np.float32) if np.isscalar(q) else q.astype(np.float32)
    x = (mean + scale * rng.normal(size=n)).astype(np.float32)
    return x, mean, scale, Q


# ------------------------------------------------------------------------------------------------ CPU: the oracle itself
def test_oracle_attr_roundtrip_and_chunking():
    from oracle import oracle as O
    x, mean, scale, Q = _case(23456, 1)
    xi = np.rint(x / Q)
    mn, mx = int(xi.min()), int(xi.max())
    cdf = O.attr_cdf(mean, scale, Q, mn, mx)
    assert cdf.shape == (23456, mx - mn + 2) and (np.diff(cdf, axis=1) >= 0).all() and cdf.min() >= 0 and cdf.max() <= 1
    sym = (xi - mn).astype(np.int16)
    stream, cnt = O.attr_encode(sym, cdf, CHUNK)
    assert len(cnt) == 3 and cnt.sum() == len(stream)
    assert np.array_equal(O.attr_decode(cdf, stream, cnt, CHUNK), sym)
    # a chunk is an independent stream: coding the second chunk alone gives its bytes
    s2, c2 = O.attr_encode(sym[CHUNK:2 * CHUNK], cdf[CHUNK:2 * CHUNK], CHUNK)
    assert s2 == stream[cnt[0]:cnt[0] + cnt[1]] and c2[0] == cnt[1]
    # known answer: the Bernoulli coder of encodings_cuda.py:435-467 on 8 symbols with p(1) = 0.5 is the range coder's KAT
    cdf2 = np.tile(np.array([[0, 0.5, 1.0]], np.float32), (8, 1))
    v = O._attr_int_rows(cdf2)
    assert list(v[0]) == [0, 32768, 0]                                      # rn(1.0 * 65534) + 2 = 2^16 wraps: only ever read as c_high of the top symbol, 0x10000 by rule
    assert O.attr_encode(np.array([0, 1, 1, 0, 1, 0, 0, 1], np.int16), cdf2, CHUNK)[0].hex() == "6940"


def test_declared_in_header_and_binding():
    from gauspcc_b200 import _lib
    names = [n for n in _lib.SIGNATURES if n.startswith("gpc_attr_")]
    assert len(names) == 7
    hdr = open(os.path.join(ROOT, "include", "gpcgc.h")).read()
    for n in names:
        assert n + "(" in hdr


def test_python_boundary_matches_reference_names():
    import inspect
    from gauspcc_b200 import arithmetic, encodings_cuda as E
    assert E.chunk_size_cuda == 10000
    for fn, args in [("encoder_gaussian", ["x", "mean", "scale", "Q", "file_name"]),
                     ("decoder_gaussian", ["mean", "scale", "Q", "file_name"]),
                     ("encoder_gaussian_chunk", ["x", "mean", "scale", "Q", "file_name", "chunk_size"]),
                     ("decoder_gaussian_chunk", ["mean", "scale", "Q", "file_name", "chunk_size"]),
                     ("encoder_gaussian_mixed", ["x", "mean_list", "scale_list", "prob_list", "Q", "file_name"]),
                     ("decoder_gaussian_mixed", ["mean_list", "scale_list", "prob_list", "Q", "file_name"]),
                     ("encoder", ["x", "file_name"]), ("decoder", ["N_len", "file_name", "device"])]:
        assert list(inspect.signature(getattr(E, fn)).parameters) == args
    for fn, args in [("calculate_cdf", ["mean", "scale", "Q", "min_value", "max_value"]),
                     ("arithmetic_encode", ["sym", "cdf", "chunk_size", "N", "Lp"]),
                     ("arithmetic_decode", ["cdf", "in_cache_all", "in_cnt_all", "chunk_size", "N", "Lp"])]:
        assert list(inspect.signature(getattr(arithmetic, fn)).parameters) == args


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ref_ext():
    from oracle import build_ref_arithmetic
    return build_ref_arithmetic.load_module()                               # None unless built (GPC_REFERENCE_ROOT at build time)


@pytest.fixture(scope="module")
def ref_golden(golden_dir):
    return np.load(os.path.join(golden_dir, "attr_golden.npz"))


def _dev(*arrays):
    import torch
    return [torch.tensor(a, device="cuda") for a in arrays]


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed,tiny", CASES)
def test_gaussian_coder_vs_oracle_and_reference(n, seed, tiny, ref_ext, ref_golden):
    import torch
    from gauspcc_b200 import arithmetic as A
    from oracle import oracle as O
    x, mean, scale, Q = _case(n, seed, tiny_scale=tiny)
    xi = np.rint(x / Q)
    mn, mx = int(xi.min()), int(xi.max())
    Lp = mx - mn + 2
    sym = (xi - mn).astype(np.int16)
    d_sym, d_mean, d_scale, d_Q = _dev(sym, mean, scale, Q)
    # 1. the table: against the numpy restatement (float erfc implementations differ in the last bits)
    lower = A.calculate_cdf(d_mean, d_scale, d_Q, mn, mx)
    assert lower.shape == (n, Lp)
    assert np.abs(lower.cpu().numpy() - O.attr_cdf(mean, scale, Q, mn, mx)).max() <= 2e-6
    # 2. table coder: bytes and counts identical to the oracle fed with the same table
    stream, cnt = A.arithmetic_encode(d_sym, lower, CHUNK, n, Lp)
    o_stream, o_cnt = O.attr_encode(sym, lower.cpu().numpy(), CHUNK)
    assert np.array_equal(cnt.cpu().numpy(), o_cnt) and stream.cpu().numpy().tobytes() == o_stream
    dec = A.arithmetic_decode(lower, stream, cnt, CHUNK, n, Lp)
    assert dec.dtype == torch.int16 and np.array_equal(dec.cpu().numpy(), sym)
    # 3. the fused Gaussian path produces the same bytes without the table, and decodes them
    g_stream, g_cnt = A.gaussian_encode(d_sym, d_mean, d_scale, d_Q, mn, mx, CHUNK)
    assert torch.equal(g_cnt, cnt) and torch.equal(g_stream, stream)
    assert np.array_equal(A.gaussian_decode(d_mean, d_scale, d_Q, g_stream, g_cnt, mn, mx, CHUNK).cpu().numpy(), sym)
    # 4. the stored tables and streams (provenance in tests/golden/make_attr_golden.py), and the reference extension itself on
    # the same GPU when it was built from the reference's own sources
    tag = f"n{n}_s{seed}"
    rows = torch.from_numpy(ref_golden[tag + "_rows"]).cuda()
    assert np.array_equal(lower[rows].cpu().numpy(), ref_golden[tag + "_lower"])
    assert np.array_equal(cnt.cpu().numpy(), ref_golden[tag + "_cnt"]) and np.array_equal(stream.cpu().numpy(), ref_golden[tag + "_stream"])
    if ref_ext is not None:
        r_lower = ref_ext.calculate_cdf(d_mean, d_scale, d_Q, mn, mx)
        assert torch.equal(r_lower, lower)
        r_stream, r_cnt = ref_ext.arithmetic_encode(d_sym, r_lower, CHUNK, n, Lp)
        assert torch.equal(r_cnt, cnt) and torch.equal(r_stream, stream)
        assert torch.equal(ref_ext.arithmetic_decode(r_lower, stream, cnt, CHUNK, n, Lp), dec)


@pytest.mark.gpu
def test_attr_coder_errors_and_edges():
    import torch
    from gauspcc_b200 import arithmetic as A
    from gauspcc_b200._lib import GpcError
    cdf = torch.tensor([[0, 0.25, 0.5, 1.0]] * 5, dtype=torch.float32, device="cuda")
    with pytest.raises(GpcError):
        A.arithmetic_encode(torch.tensor([0, 1, 3, 0, 0], dtype=torch.int16, device="cuda"), cdf, CHUNK, 5, 4)   # symbol > Lp - 2
    with pytest.raises(RuntimeError):
        A.arithmetic_encode(torch.zeros(5, dtype=torch.int16), cdf.cpu(), CHUNK, 5, 4)                           # no CPU path
    # zero-width bins (two equal CDF entries) still code: the `+ symbol` keeps the integer CDF strictly increasing
    cdf0 = torch.tensor([[0, 0, 0, 1.0]] * 64, dtype=torch.float32, device="cuda")
    sym = torch.tensor([0, 1, 2, 2] * 16, dtype=torch.int16, device="cuda")
    stream, cnt = A.arithmetic_encode(sym, cdf0, 16, 64, 4)
    assert cnt.numel() == 4 and torch.equal(A.arithmetic_decode(cdf0, stream, cnt, 16, 64, 4), sym)
    # a truncated stream decodes to garbage of the right length, without hanging or faulting
    out = A.arithmetic_decode(cdf0, stream[:1], torch.tensor([1, 0, 0, 0], dtype=torch.int32, device="cuda"), 16, 64, 4)
    assert out.shape == (64,)


@pytest.mark.gpu
def test_encodings_cuda_files(tmp_path, ref_ext):
    """The drop-in of HAC/utils/encodings_cuda.py: round trips through .b files for every coder HAC / HAC++ call
    (gaussian_model.py:1171-1206, 1239-1310; HAC-plus gaussian_model.py:1315, 1499), and the bit counts they return."""
    import torch
    from gauspcc_b200 import encodings_cuda as E
    n = 34567
    x, mean, scale, Q = _case(n, 9, q=np.random.default_rng(3).choice([0.25, 0.5, 1.0], n))
    d_x, d_mean, d_scale, d_Q = _dev(x, mean, scale, Q)
    f = str(tmp_path / "feat.b")
    bits = E.encoder_gaussian(d_x, d_mean, d_scale, d_Q, file_name=f)
    assert bits == 8 * os.path.getsize(f)
    back = E.decoder_gaussian(d_mean, d_scale, d_Q, file_name=f)
    assert torch.equal(back, torch.round(d_x / d_Q) * d_Q)
    # scalar Q, chunked files (chunk_size symbols per file: name_<c>.b)
    bits = E.encoder_gaussian_chunk(d_x, d_mean, d_scale, 0.5, file_name=f, chunk_size=15000)
    files = sorted(p.name for p in tmp_path.iterdir() if p.name.startswith("feat_"))
    assert files == ["feat_0.b", "feat_1.b", "feat_2.b"] and bits == 8 * sum(os.path.getsize(tmp_path / p) for p in files)
    back = E.decoder_gaussian_chunk(d_mean, d_scale, 0.5, file_name=f, chunk_size=15000)
    assert torch.equal(back, torch.round(d_x / 0.5) * 0.5)
    # mixture of three Gaussians (HAC++)
    probs = torch.softmax(torch.randn(3, n, device="cuda"), 0)
    means = [d_mean, d_mean + 1.0, d_mean - 2.0]
    scales = [d_scale, d_scale * 2, d_scale * 0.5]
    g = str(tmp_path / "mix.b")
    bits = E.encoder_gaussian_mixed_chunk(d_x, means, scales, list(probs), d_Q, file_name=g, chunk_size=20000)
    back = E.decoder_gaussian_mixed_chunk(means, scales, list(probs), d_Q, file_name=g, chunk_size=20000)
    assert torch.equal(back, torch.round(d_x / d_Q) * d_Q) and bits > 0
    # Bernoulli masks
    mask = (torch.rand(n, device="cuda") < 0.3).to(torch.float32)
    h = str(tmp_path / "mask.b")
    bits = E.encoder(mask, file_name=h)
    assert bits == 8 * os.path.getsize(h)
    assert torch.equal(E.decoder(n, h).to(torch.float32), mask)
    assert bits < 0.95 * n                                                  # H(0.3) = 0.88 bit per symbol
