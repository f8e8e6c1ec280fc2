"""Generate tests/golden/attr_golden.npz from the reference's attribute coder (HAC/submodules/arithmetic.zip), on the five inputs of
tests/test_attr_coder.py::test_gaussian_coder_vs_oracle_and_reference.

    GPC_REFERENCE_ROOT=<checkout of the reference> python __graft_entry__.py      # builds oracle/_ref/arithmetic.so
    python tests/golden/make_attr_golden.py [out.npz]                             # needs a CUDA device

Per case it stores what the reference extension returns: a seeded sample of the rows of its table (calculate_cdf; the whole
table of the largest case is 552 MB), its byte stream and its per-chunk byte counts (arithmetic_encode).  It refuses to run
without the extension, and to save when this library's calculate_cdf / arithmetic_encode differ from the extension's anywhere.

Provenance of the committed file: it was recorded from this library's calculate_cdf + arithmetic_encode, at a commit whose
tests/test_attr_coder.py asserted those to be identical to the reference extension's, but without the extension at hand
when the file was written.  Running this script reproduces it from the extension itself; its arrays must come out the same."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

SAMPLE_ROWS = 64


def sample_rows(n, seed):
    """the table rows kept for case (n, seed): the first, the last and SAMPLE_ROWS seeded ones"""
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([[0, n - 1], rng.choice(n, min(n, SAMPLE_ROWS), replace=False)])).astype(np.int64)


def main(out):
    import torch
    from gauspcc_b200 import arithmetic as A
    from oracle import build_ref_arithmetic
    from test_attr_coder import CASES, CHUNK, _case
    ref = build_ref_arithmetic.load_module()
    if ref is None:
        sys.exit("the reference extension is not built (oracle/_ref/arithmetic.so): see the usage above")
    g = {}
    for n, seed, tiny in CASES:
        x, mean, scale, Q = _case(n, seed, tiny_scale=tiny)
        xi = np.rint(x / Q)
        mn, mx = int(xi.min()), int(xi.max())
        Lp = mx - mn + 2
        d_sym, d_mean, d_scale, d_Q = [torch.tensor(a, device="cuda") for a in ((xi - mn).astype(np.int16), mean, scale, Q)]
        lower = ref.calculate_cdf(d_mean, d_scale, d_Q, mn, mx)
        stream, cnt = ref.arithmetic_encode(d_sym, lower, CHUNK, n, Lp)
        ours = A.calculate_cdf(d_mean, d_scale, d_Q, mn, mx)
        o_stream, o_cnt = A.arithmetic_encode(d_sym, ours, CHUNK, n, Lp)
        if not (torch.equal(ours, lower) and torch.equal(o_cnt, cnt) and torch.equal(o_stream, stream)):
            sys.exit(f"case n={n} seed={seed}: the library's table or stream differs from the reference extension's; nothing written")
        rows = sample_rows(n, seed)
        tag = f"n{n}_s{seed}"
        g[tag + "_rows"] = rows
        g[tag + "_lower"] = lower[torch.from_numpy(rows).to(lower.device)].cpu().numpy()
        g[tag + "_stream"] = stream.cpu().numpy()
        g[tag + "_cnt"] = cnt.cpu().numpy()
    np.savez_compressed(out, **g)
    print(out, {k: v.shape for k, v in g.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "attr_golden.npz"))
