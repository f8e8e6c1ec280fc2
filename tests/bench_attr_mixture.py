"""(Lives under tests/ because it loads the reference extension from oracle/_ref: only tests/, smoke() and bench.py may touch oracle/.)
HAC++'s mixture coder on one GPU: the fused path (arithmetic.mixture_encode / mixture_decode, no table) against the table sequence
encoder_gaussian_mixed / decoder_gaussian_mixed run before it (calculate_cdf per component, `* prob`, summed, clamped, then
arithmetic_encode / arithmetic_decode) on the library's kernels and, when built, on the reference extension.

    python tests/bench_attr_mixture.py [n_symbols] [reps]       (default 10 000 000 = one file of encoder_gaussian_mixed_chunk, 5 reps)

Prints one JSON line: the card's name and power limit, then per K in (2, 3) CUDA-event times after one warm-up call, the peak of
torch.cuda.max_memory_allocated above what the inputs hold, and how often the fused decoder's first window of 32 candidates
decides the symbol for two choices of its centre.  Bytes and symbols are checked for identity before any timing.  The inputs
(10 M symbols, several hundred MB) are far larger than L2."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gauspcc_b200 import arithmetic as A

CHUNK = 10000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit": q[1]}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) / reps, 3), out


def peak_mb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    return round((torch.cuda.max_memory_allocated() - base) / 2**20, 1), out


def table(ext, M, S, P, Q, mn, mx):
    lower = ext.calculate_cdf(M[0], S[0], Q, mn, mx) * P[0].unsqueeze(-1)
    for k in range(1, M.shape[0]):
        lower += ext.calculate_cdf(M[k], S[k], Q, mn, mx) * P[k].unsqueeze(-1)
    return torch.clamp(lower, min=0.0, max=1.0)


def window_hits(sym, centre, max_symbol):
    """share of symbols the decoder's first window (attr_decode_chunks_kernel, CENTRED) decides without attr_search"""
    w0 = torch.clamp(centre - 15, max=max_symbol - 31).clamp(min=0)
    top = torch.clamp(max_symbol - w0, max=31)
    s = sym.long()
    miss = ((s < w0) & (w0 > 0)) | ((s >= w0 + top) & (w0 + top < max_symbol))
    return round(1.0 - miss.float().mean().item(), 4)


def run_k(K, n, reps, ref):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(K)
    q = 0.25
    Q = torch.full((n,), q, device=dev)
    # bimodal (K = 2) / trimodal (K = 3): components 40 bins apart around a common centre, as HAC++'s mixtures are when they help
    off = (torch.arange(K, device=dev, dtype=torch.float32) - (K - 1) / 2) * 40 * q
    centre = torch.randn(n, device=dev, generator=g) * 6 * q
    M = (centre[None] + off[:, None]).contiguous()
    S = ((torch.randn(K, n, device=dev, generator=g).abs() * 0.5 + 0.3) * 4 * q).contiguous()
    P = torch.softmax(torch.randn(n, K, device=dev, generator=g) * 1.5, 1).t().contiguous()
    comp = torch.multinomial(P.t(), 1, generator=g).view(1, -1)
    x = M.gather(0, comp)[0] + S.gather(0, comp)[0] * torch.randn(n, device=dev, generator=g)
    xi = torch.round(x / Q)
    mn, mx = int(xi.min()), int(xi.max())
    Lp = mx - mn + 2
    sym = (xi - mn).to(torch.int16)
    del x, comp, centre

    # identity first
    stream, cnt = A.mixture_encode(sym, M, S, P, Q, mn, mx, CHUNK)
    lower = table(A, M, S, P, Q, mn, mx)
    t_stream, t_cnt = A.arithmetic_encode(sym, lower, CHUNK, n, Lp)
    ok_stream = bool(torch.equal(stream, t_stream) and torch.equal(cnt, t_cnt))
    ok_sym = bool(torch.equal(A.mixture_decode(M, S, P, Q, stream, cnt, mn, mx, CHUNK), sym)
                  and torch.equal(A.arithmetic_decode(lower, stream, cnt, CHUNK, n, Lp), sym))
    del lower, t_stream, t_cnt
    assert ok_stream and ok_sym

    major = M.gather(0, P.argmax(0, keepdim=True))[0]
    hits = {"major_component_mean": window_hits(sym, torch.round(major / Q).long() - mn, Lp - 2),
            "mixture_mean": window_hits(sym, torch.round((M * P).sum(0) / Q).long() - mn, Lp - 2)}

    def enc_fused():
        return A.mixture_encode(sym, M, S, P, Q, mn, mx, CHUNK)

    def dec_fused():
        return A.mixture_decode(M, S, P, Q, stream, cnt, mn, mx, CHUNK)

    def enc_table(ext=A):
        return ext.arithmetic_encode(sym, table(ext, M, S, P, Q, mn, mx), CHUNK, n, Lp)

    def dec_table(ext=A):
        return ext.arithmetic_decode(table(ext, M, S, P, Q, mn, mx), stream, cnt, CHUNK, n, Lp)

    res = {"K": K, "n_symbols": n, "Lp": Lp, "bits_per_symbol": round(8 * stream.numel() / n, 3), "identical_stream": ok_stream,
           "identical_symbols": ok_sym, "first_window_hit_rate": hits}
    for name, enc, dec in [("fused", enc_fused, dec_fused), ("table", enc_table, dec_table)]:
        te, _ = timed(enc, reps)
        td, _ = timed(dec, reps)
        me, _ = peak_mb(enc)
        md, _ = peak_mb(dec)
        res[name] = {"enc_ms": te, "dec_ms": td, "enc_peak_MB": me, "dec_peak_MB": md}
    if ref is None:
        res["reference_table"] = "oracle/_ref/arithmetic.so not built"
    else:
        r_stream, r_cnt = enc_table(ref)
        same = bool(torch.equal(r_stream, stream) and torch.equal(r_cnt, cnt) and torch.equal(dec_table(ref), sym))
        te, _ = timed(lambda: enc_table(ref), max(1, reps // 2))
        td, _ = timed(lambda: dec_table(ref), max(1, reps // 2))
        me, _ = peak_mb(lambda: enc_table(ref))
        md, _ = peak_mb(lambda: dec_table(ref))
        res["reference_table"] = {"enc_ms": te, "dec_ms": td, "enc_peak_MB": me, "dec_peak_MB": md, "identical": same}
    res["speedup_vs_table"] = {"enc": round(res["table"]["enc_ms"] / res["fused"]["enc_ms"], 2),
                               "dec": round(res["table"]["dec_ms"] / res["fused"]["dec_ms"], 2)}
    return res


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    from oracle import build_ref_arithmetic
    ref = build_ref_arithmetic.load_module()
    line = {"metric": "HAC++ mixture coder: fused vs table sequence (device-timed ms, peak MB above the inputs)", "card": card(),
            "chunk_size": CHUNK, "runs": [run_k(K, n, reps, ref) for K in (2, 3)]}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
