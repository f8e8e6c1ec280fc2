"""Drop-in for the coder half of HAC/utils/encodings_cuda.py (:317-500 and the mixed variants :178-314): the same function
names, arguments, return values and `.b` file layout (float32 min, float32 max, int32 len(cnt bytes), cnt int32[chunks], stream),
so files written by either side are read by the other.

    HAC/scene/gaussian_model.py:37   from utils.encodings_cuda import encoder_gaussian_chunk, decoder_gaussian_chunk, encoder, decoder

No coder here builds the reference's lower[N][Lp] table on the paths HAC and HAC++ take: the single-Gaussian coders evaluate
each symbol's CDF entries on the fly (arithmetic.gaussian_encode / gaussian_decode), the mixture coders do the same for up to
four components (arithmetic.mixture_encode / mixture_decode), and the Bernoulli mask coder codes every symbol against one
shared row [0, 1 - p, 1] (arithmetic.row_encode / row_decode).  The bytes are those of the table path.  Mixture calls the fused
path cannot reproduce bit for bit (more than four components, components not 1-D of the symbols' length, probabilities that are
not float32 / float16 / bfloat16) still build the table with the reference's element-wise torch arithmetic (_mixed_lower).
"""
from __future__ import annotations

import numpy as np
import torch

from . import arithmetic

chunk_size_cuda = 10000                                                     # encodings_cuda.py:6


def _q_tensor(Q, like):
    if not isinstance(Q, torch.Tensor):
        Q = torch.tensor([Q], dtype=like.dtype, device=like.device).repeat(like.shape[0])
    return Q


def _f32(t):
    return t.detach().to(torch.float32).contiguous()


def _write(file_name, header, cnt_torch, byte_stream_torch):
    cnt_bytes = cnt_torch.cpu().numpy().tobytes()
    byte_stream_bytes = byte_stream_torch.cpu().numpy().tobytes()
    with open(file_name, 'wb') as fout:
        for h in header:
            fout.write(h)
        fout.write(np.array([len(cnt_bytes)]).astype(np.int32).tobytes())
        fout.write(cnt_bytes)
        fout.write(byte_stream_bytes)
    return (len(byte_stream_bytes) + len(cnt_bytes)) * 8 + 32 * (len(header) + 1)


def _read(file_name, n_header, device="cuda"):
    with open(file_name, 'rb') as fin:
        header = [np.frombuffer(fin.read(4), dtype=np.float32).copy() for _ in range(n_header)]
        len_cnt_bytes = int(np.frombuffer(fin.read(4), dtype=np.int32)[0])
        cnt = torch.tensor(np.frombuffer(fin.read(len_cnt_bytes), dtype=np.int32).copy(), device=device)
        stream = torch.tensor(np.frombuffer(fin.read(), dtype=np.uint8).copy(), device=device)
    return header, cnt, stream


def _quantise(x, Q):
    x_int_round = torch.round(x / Q)                                        # encodings_cuda.py:342
    mm = torch.stack([x_int_round.min(), x_int_round.max()]).cpu()          # one transfer for both
    return x_int_round, mm[0], mm[1]


def encoder_gaussian(x, mean, scale, Q, file_name='tmp.b'):
    """encodings_cuda.py:335-373"""
    assert file_name.endswith('.b')
    assert len(x.shape) == 1
    Q = _q_tensor(Q, mean)
    x_int_round, min_value, max_value = _quantise(x, Q)
    sym = (x_int_round - min_value.to(x.device)).to(torch.int16)
    stream, cnt = arithmetic.gaussian_encode(sym.contiguous(), _f32(mean), _f32(scale), _f32(Q), int(min_value), int(max_value),
                                             chunk_size_cuda)
    return _write(file_name, [min_value.to(torch.float32).numpy().tobytes(), max_value.to(torch.float32).numpy().tobytes()], cnt, stream)


def decoder_gaussian(mean, scale, Q, file_name='tmp.b'):
    """encodings_cuda.py:394-432"""
    assert file_name.endswith('.b')
    assert len(mean.shape) == 1
    assert mean.shape == scale.shape
    Q = _q_tensor(Q, mean)
    (mn, mx), cnt, stream = _read(file_name, 2, mean.device)
    sym = arithmetic.gaussian_decode(_f32(mean), _f32(scale), _f32(Q), stream, cnt, int(mn[0]), int(mx[0]), chunk_size_cuda)
    x = sym.to(torch.float32) + float(mn[0])
    return x * Q


def _chunked(N, chunk_size):
    return [(c, slice(c * chunk_size, c * chunk_size + chunk_size)) for c in range(int(np.ceil(N / chunk_size)))]


def encoder_gaussian_chunk(x, mean, scale, Q, file_name='tmp.b', chunk_size=1000_0000):
    """encodings_cuda.py:317-332: one file per 10 M symbols, `name_<c>.b`"""
    assert file_name.endswith('.b')
    assert len(x.shape) == 1
    x, mean, scale = x.view(-1), mean.view(-1), scale.view(-1)
    is_t = isinstance(Q, torch.Tensor)
    if is_t:
        Q = Q.view(-1)
    return sum(encoder_gaussian(x[s], mean[s], scale[s], Q[s] if is_t else Q, file_name.replace('.b', f'_{str(c)}.b'))
               for c, s in _chunked(x.shape[0], chunk_size))


def decoder_gaussian_chunk(mean, scale, Q, file_name='tmp.b', chunk_size=1000_0000):
    """encodings_cuda.py:375-391"""
    assert file_name.endswith('.b')
    mean_v, scale_v = mean.view(-1), scale.view(-1)
    is_t = isinstance(Q, torch.Tensor)
    if is_t:
        Q = Q.view(-1)
    out = [decoder_gaussian(mean_v[s], scale_v[s], Q[s] if is_t else Q, file_name.replace('.b', f'_{str(c)}.b'))
           for c, s in _chunked(mean_v.shape[0], chunk_size)]
    return torch.cat(out, dim=0).type_as(mean)


_FUSED_PROB_DTYPES = (torch.float32, torch.float16, torch.bfloat16)      # exact in float32, as torch's promotion in `lower * prob`


def _takes_fused_mixture(n, mean_list, scale_list, prob_list):
    """True when arithmetic.mixture_* gives the bytes of the table _mixed_lower builds: 1 to 4 components, every mean / scale /
    prob a 1-D tensor of length n (no broadcasting) and every prob float32, float16 or bfloat16."""
    k = len(mean_list)
    if not 1 <= k <= 4 or len(scale_list) != k or len(prob_list) != k:
        return False
    if not all(isinstance(t, torch.Tensor) and tuple(t.shape) == (n,) for t in (*mean_list, *scale_list, *prob_list)):
        return False
    return all(p.dtype in _FUSED_PROB_DTYPES for p in prob_list)


def _stack_f32(ts):
    return torch.stack([t.detach().to(torch.float32) for t in ts])      # [K, n], contiguous


def _mixed_lower(mean_list, scale_list, prob_list, Q, min_value, max_value):
    lower_all = None                                                        # encodings_cuda.py:211-226
    for mean, scale, prob in zip(mean_list, scale_list, prob_list):
        lower = arithmetic.calculate_cdf(_f32(mean), _f32(scale), _f32(Q), min_value, max_value) * prob.unsqueeze(-1)
        if lower_all is None:
            lower_all = lower
        else:
            lower_all += lower
    return torch.clamp(lower_all, min=0.0, max=1.0)


def encoder_gaussian_mixed(x, mean_list, scale_list, prob_list, Q, file_name='tmp.b'):
    """encodings_cuda.py:203-250"""
    assert file_name.endswith('.b')
    assert len(x.shape) == 1
    Q = _q_tensor(Q, x)
    assert x.shape == mean_list[0].shape == scale_list[0].shape == prob_list[0].shape == Q.shape
    x_int_round, min_value, max_value = _quantise(x, Q)
    sym = (x_int_round - min_value.to(x.device)).to(torch.int16)
    if _takes_fused_mixture(x.shape[0], mean_list, scale_list, prob_list):
        stream, cnt = arithmetic.mixture_encode(sym.contiguous(), _stack_f32(mean_list), _stack_f32(scale_list), _stack_f32(prob_list),
                                                _f32(Q), int(min_value), int(max_value), chunk_size_cuda)
    else:
        lower = _mixed_lower(mean_list, scale_list, prob_list, Q, int(min_value), int(max_value))
        stream, cnt = arithmetic.arithmetic_encode(sym.contiguous(), lower, chunk_size_cuda, int(lower.shape[0]), int(lower.shape[1]))
    return _write(file_name, [min_value.to(torch.float32).numpy().tobytes(), max_value.to(torch.float32).numpy().tobytes()], cnt, stream)


def decoder_gaussian_mixed(mean_list, scale_list, prob_list, Q, file_name='tmp.b'):
    """encodings_cuda.py:277-314"""
    assert file_name.endswith('.b')
    m0 = mean_list[0]
    Q = _q_tensor(Q, m0)
    assert mean_list[0].shape == scale_list[0].shape == prob_list[0].shape == Q.shape
    (mn, mx), cnt, stream = _read(file_name, 2, m0.device)
    if _takes_fused_mixture(m0.numel(), mean_list, scale_list, prob_list):
        sym = arithmetic.mixture_decode(_stack_f32(mean_list), _stack_f32(scale_list), _stack_f32(prob_list), _f32(Q), stream, cnt,
                                        int(mn[0]), int(mx[0]), chunk_size_cuda)
    else:
        lower = _mixed_lower(mean_list, scale_list, prob_list, Q, int(mn[0]), int(mx[0]))
        sym = arithmetic.arithmetic_decode(lower, stream, cnt, chunk_size_cuda, int(lower.shape[0]), int(lower.shape[1]))
    x = sym.to(m0.device).to(torch.float32) + float(mn[0])
    return x * Q


def encoder_gaussian_mixed_chunk(x, mean_list, scale_list, prob_list, Q, file_name='tmp.b', chunk_size=1000_0000):
    """encodings_cuda.py:178-200"""
    assert file_name.endswith('.b')
    assert len(x.shape) == 1
    x = x.view(-1)
    ml, sl, pl = [m.view(-1) for m in mean_list], [s.view(-1) for s in scale_list], [p.view(-1) for p in prob_list]
    is_t = isinstance(Q, torch.Tensor)
    if is_t:
        Q = Q.view(-1)
    return sum(encoder_gaussian_mixed(x[s], [m[s] for m in ml], [v[s] for v in sl], [p[s] for p in pl], Q[s] if is_t else Q,
                                      file_name.replace('.b', f'_{str(c)}.b')) for c, s in _chunked(x.shape[0], chunk_size))


def decoder_gaussian_mixed_chunk(mean_list, scale_list, prob_list, Q, file_name='tmp.b', chunk_size=1000_0000):
    """encodings_cuda.py:253-274"""
    assert file_name.endswith('.b')
    ml, sl, pl = [m.view(-1) for m in mean_list], [s.view(-1) for s in scale_list], [p.view(-1) for p in prob_list]
    is_t = isinstance(Q, torch.Tensor)
    if is_t:
        Q = Q.view(-1)
    out = [decoder_gaussian_mixed([m[s] for m in ml], [v[s] for v in sl], [p[s] for p in pl], Q[s] if is_t else Q,
                                  file_name.replace('.b', f'_{str(c)}.b')) for c, s in _chunked(ml[0].shape[0], chunk_size)]
    return torch.cat(out, dim=0).type_as(mean_list[0])


def _bernoulli_row(prob_1, device):
    p = torch.as_tensor(prob_1, dtype=torch.float32, device=device).reshape(1)     # encodings_cuda.py:439-446: every row of the
    return torch.cat([torch.zeros_like(p), 1 - p, torch.ones_like(p)])             # reference's [n, 3] table is [0, 1 - p, 1]


def encoder(x, file_name='tmp.b'):
    """encodings_cuda.py:435-467: a {0, 1} tensor under one global Bernoulli probability"""
    assert file_name[-2:] == '.b'
    x = x.detach().view(-1)
    prob_1 = x.sum() / x.numel()
    sym = torch.floor(x).to(torch.int16)
    stream, cnt = arithmetic.row_encode(sym.contiguous(), _bernoulli_row(prob_1.to(torch.float32), x.device), chunk_size_cuda)
    return _write(file_name, [prob_1.to(torch.float32).cpu().numpy().tobytes()], cnt, stream)


def decoder(N_len, file_name='tmp.b', device='cuda'):
    """encodings_cuda.py:470-500"""
    assert file_name[-2:] == '.b'
    (prob_1,), cnt, stream = _read(file_name, 1, device)
    return arithmetic.row_decode(_bernoulli_row(prob_1, device), stream, cnt, N_len, chunk_size_cuda)
