"""Bring-up check + timing of the TMA / tcgen05 conv (spconv_um.cu) against a torch fp64 reference built from the dense kernel map and
against the mma.sync conv (v6d) on the levels of a synthetic scene.  Run on the GPU box:  python tools/um_check.py [npts]"""
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gauspcc_b200 import _lib
from gauspcc_b200.codec import UM_TILE_ROWS, DeviceWeights, GausPcgcCodec, _ptr
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import make_synthetic_state_dict


def main():
    npts = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
    min_rows = int(os.environ.get("UM_MIN_ROWS", 3000))
    dev = torch.device("cuda:0")
    w = DeviceWeights(make_synthetic_state_dict(), dev)
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    wp = torch.empty_like(w.convs)
    _lib.check(lib.gpc_spconv_pack_weights_um(_ptr(w.convs), w.convs.shape[0], _ptr(wp), st), "pack_um")
    xyz = torch.tensor(hac_like_cloud(npts, 0), dtype=torch.float32, device=dev)
    codec = GausPcgcCodec(w, dev)
    keys, meta = codec.pack_keys(xyz)
    mm = meta.cpu().numpy()[2:8]
    leaf = codec.sort_unique(keys, mm.astype(np.uint32))
    levels = codec.build_pyramid(leaf, mm.astype(np.int64))
    print("levels:", [l.n for l in levels], flush=True)
    widx = 3
    for li, lv in enumerate(levels):
        n = lv.n
        if n < min_rows:
            continue
        dense = codec.dense_map(lv.keys)
        g = torch.Generator(device=dev).manual_seed(li)
        x = torch.randn((n, 32), device=dev, generator=g)
        res = torch.randn((n, 32), device=dev, generator=g)
        xs = codec.split_rows(x)
        xj = torch.empty_like(x)
        codec._call("gpc_rows_join", _ptr(xs), n, _ptr(xj), codec._stream())          # what the split rows really hold
        # fp64 reference on the split-row values
        ref = torch.zeros((n, 32), dtype=torch.float64, device=dev)
        W64 = w.convs[widx].double()
        for k in range(125):
            m = dense[k]
            hit = m >= 0
            if hit.any():
                ref[hit] += xj[m[hit].long()].double() @ W64[k]
        ref_relu = torch.relu(ref + res.double())
        n_pairs_real = int((dense >= 0).sum())
        # v6d timing
        km6b = codec.build_kmap(lv.keys, family="v6")
        y6 = codec.conv(x, widx, km6b, residual=res, relu=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            codec.conv(x, widx, km6b, residual=res, relu=True, out=y6)
        e1.record(); torch.cuda.synchronize()
        ms6 = e0.elapsed_time(e1) / reps
        err6 = float((y6.double() - torch.relu((ref - xj.double().new_zeros(1)) + res.double())).abs().max())
        tr = UM_TILE_ROWS
        km = codec._um_map(dense, n, tr)
        poff = km.pair_off
        y = torch.full((n, 32), float("nan"), device=dev)
        ys = torch.zeros((n, 32), dtype=torch.int32, device=dev)
        order = km.tile_order if os.environ.get("UM_ORDER", "1") != "0" else None
        args = (_ptr(xs), _ptr(wp[widx]), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(poff), n, tr, _ptr(order), _ptr(res), 1, _ptr(y), _ptr(ys), 0, 0, st)
        rc = lib.gpc_spconv_fwd_um(*args)
        _lib.check(rc, "um")
        torch.cuda.synchronize()
        err = float((y.double() - ref_relu).abs().max())
        yj = torch.empty_like(y)
        codec._call("gpc_rows_join", _ptr(ys), n, _ptr(yj), codec._stream())
        err_s = float((yj - y).abs().max())
        scale = float(ref_relu.abs().max())
        # determinism + row-range launches
        y2 = torch.empty_like(y)
        args2 = list(args); args2[10] = _ptr(y2); args2[11] = None
        half = (n // 2) // tr * tr
        a = list(args2); a[12], a[13] = 0, half
        _lib.check(lib.gpc_spconv_fwd_um(*a), "um rows a")
        a = list(args2); a[12], a[13] = half, 0
        _lib.check(lib.gpc_spconv_fwd_um(*a), "um rows b")
        torch.cuda.synchronize()
        same = bool(torch.equal(y2, y))
        e0.record()
        for _ in range(reps):
            lib.gpc_spconv_fwd_um(*args2)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        clk = ms * 1e-3 * 1.9e9 * 148 / max(n_pairs_real, 1)
        if os.environ.get("UM_PROF", "1") != "0":
            lib.gpc_debug_conv_um_profile(None, 1)
            a = list(args2); a[9] = 1 | 256
            _lib.check(lib.gpc_spconv_fwd_um(*a), "um prof")
            buf = (C.c_uint64 * 16)()
            lib.gpc_debug_conv_um_profile(C.cast(buf, C.c_void_p), 1)
            ch, ctas = max(buf[11], 1), max(buf[15], 1)
            names = ["e.items", "p.empty_g", "p.issue", "m.full_w", "m.full_g", "m.empty_d", "m.issue", "e.loop", "e.full_d", "e.ldtm_issue", "e.rmw"]
            print(f"   prof tile={tr}: chunks/cta={ch / ctas:.0f} " + " ".join(f"{nm}={buf[i] / ch:.0f}" for i, nm in enumerate(names))
                  + f" | per cta: total={buf[12] / ctas:.0f} setup={buf[13] / ctas:.0f} writeout={buf[14] / ctas:.0f}", flush=True)
        print(f"n={n:8d} p/r={n_pairs_real / n:5.1f} tile={tr:4d} entries/pairs={km.n_pairs / max(n_pairs_real, 1):.2f} "
              f"um {ms:.3f} ms ({clk:.1f} clk/pair)  v6d {ms6:.3f} ms  err={err:.2e} (v6d {err6:.2e}, scale {scale:.1f}) "
              f"split-out err={err_s:.2e} rows-identical={same}", flush=True)


if __name__ == "__main__":
    main()
