"""Training on the GPU (gauspcc_b200/train.py, csrc/spconv_grad.cu): the weight-gradient kernel and the mirrored-weight input gradient
against fp64, SparseConvFn against torch fp64 autograd, the network's code length against the codec's own probabilities and bytes,
whole-network gradients against an fp64 restatement of SURVEY.md Appendix A, a short training run and `cli train`.

Bounds: the gradients run the forward's arithmetic (bf16 hi / lo split, three terms, fp32 accumulation), so the fp64 bound of
tests/test_row_ranges.py applies per element, relative to the sum of magnitudes of the products that make it up:
|got - ref| <= 2 * 2^-16 * absref."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

BOUND_C = 2.0
V6_CONFIGS = [(8, 47), (16, 46), (32, 46), (64, 42), (64, 48), (128, 48)]      # (tile_rows, variant): every mma.sync tiling
LEVELS = [(1_000, 9), (30_000, 12), (200_000, 14)]                            # (rows, extent_log2 of the hac-like cloud)
WIDX = 7


@pytest.fixture(scope="module")
def env():
    from gauspcc_b200 import train as T
    from gauspcc_b200.codec import GausPcgcCodec
    from gauspcc_b200.weights import CONV_KEYS, make_synthetic_state_dict
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    geo = {k: GausPcgcCodec(T._Geometry(k), dev) for k in (3, 5)}
    W = {k: T._to125(make_synthetic_state_dict(5, 32, k)[CONV_KEYS[WIDX]].to(dev)) for k in (3, 5)}
    return {"T": T, "dev": dev, "geo": geo, "W": W}


_LEVELS = {}


def level(env, n, ext, k):
    """sorted keys, dense map [125, n], random x / dy and the fp64 references of dW and dx of one level, computed once"""
    key = (n, k)
    if key in _LEVELS:
        return _LEVELS[key]
    from gauspcc_b200.synth import hac_like_cloud
    codec, dev = env["geo"][k], env["dev"]
    keys, _ = codec.pack_keys(torch.tensor(hac_like_cloud(n, seed=n, extent_log2=ext), device=dev))
    keys = torch.sort(keys).values
    dense = codec.dense_map(keys)
    g = torch.Generator(device=dev).manual_seed(n + k)
    x = torch.randn((n, 32), generator=g, device=dev)
    dy = torch.randn((n, 32), generator=g, device=dev)
    x64, d64, W64 = x.double(), dy.double(), env["W"][k].double()
    dW = torch.zeros((125, 32, 32), dtype=torch.float64, device=dev)
    dW_abs, dx, dx_abs = torch.zeros_like(dW), torch.zeros_like(x64), torch.zeros_like(x64)
    for kk in range(125):
        o = (dense[kk] >= 0).nonzero().squeeze(1)
        if o.numel() == 0:
            continue
        i = dense[kk][o].long()
        dW[kk] = x64[i].t() @ d64[o]
        dW_abs[kk] = x64[i].abs().t() @ d64[o].abs()
        dx.index_add_(0, i, d64[o] @ W64[kk].t())                   # dx[i] += dy[o] W[k]^T over the pairs (o, i) of offset k
        dx_abs.index_add_(0, i, d64[o].abs() @ W64[kk].abs().t())
    lv = dict(keys=keys, dense=dense, n=n, x=x, dy=dy, dW=dW, dW_abs=dW_abs, dx=dx, dx_abs=dx_abs)
    _LEVELS[key] = lv
    return lv


def within(got, ref, absref):
    err = (got.double() - ref).abs()
    ratio = float((err / absref.clamp(min=1e-30)).max())
    return bool((err <= BOUND_C * 2.0 ** -16 * absref + 1e-30).all()), ratio


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("n,ext", LEVELS)
def test_wgrad_against_fp64(env, n, ext, k):
    T, codec = env["T"], env["geo"][k]
    lv = level(env, n, ext, k)
    absent = lv["dW_abs"].flatten(1).amax(1) == 0
    if k == 3:
        outer = torch.ones(125, dtype=torch.bool, device=env["dev"])
        outer[list(T.K5_OF_K3)] = False
        assert bool(absent[outer].all())                            # a 3^3 map has no pair outside the inner cube
    for tr, var in V6_CONFIGS:
        km = codec._v6_map(lv["dense"], n, tr, var)
        dW = T.conv_wgrad(lv["x"], lv["dy"], km)
        ok, ratio = within(dW, lv["dW"], lv["dW_abs"])
        assert ok, f"tile_rows {tr}: worst |err| / absref {ratio * 2 ** 16:.3f} * 2^-16"
        assert bool((dW[absent] == 0).all()) and not bool(torch.signbit(dW[absent]).any())   # absent offsets: exact +0
        assert torch.equal(T.conv_wgrad(lv["x"], lv["dy"], km), dW)                          # same bits on every call
        print(f"wgrad n={n} K={k} tile_rows={tr}: worst |err| / absref {ratio * 2 ** 16:.3f} * 2^-16")


def test_wgrad_padding_contributes_nothing(env):
    """entries of the padding (all ones) add nothing: the same pairs in a stream with a different padding pattern (other tile
    heights pad other segments) give dW within rounding, and a level whose rows have no neighbours but themselves gives x^T dy"""
    T, codec, dev = env["T"], env["geo"][5], env["dev"]
    keys, _ = codec.pack_keys(torch.tensor([[8 * i, 0, 0] for i in range(37)], dtype=torch.int32, device=dev))
    keys = torch.sort(keys).values
    dense = codec.dense_map(keys)
    x, dy = torch.randn((37, 32), device=dev), torch.randn((37, 32), device=dev)
    for tr, var in V6_CONFIGS:
        dW = T.conv_wgrad(x, dy, codec._v6_map(dense, 37, tr, var))
        ref = x.double().t() @ dy.double()
        assert bool(((dW[62].double() - ref).abs() <= BOUND_C * 2.0 ** -16 * (x.double().abs().t() @ dy.double().abs())).all())
        others = torch.cat([dW[:62], dW[63:]])
        assert bool((others == 0).all())


def test_wgrad_rejects_bad_arguments(env):
    from gauspcc_b200 import _lib
    lib = _lib.load()
    assert lib.gpc_spconv_wgrad_v6(None, None, None, None, 100, 24, None, None, 0, None) == -1
    assert lib.gpc_spconv_wgrad_v6(None, None, None, None, 100, 64, None, None, 0, None) == -4      # workspace too small
    assert lib.gpc_spconv_wgrad_workspace_bytes(100, 64) == 125 * 32 * 32 * 4


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("n,ext", LEVELS)
def test_dgrad_through_the_mirrored_pack(env, n, ext, k):
    T, codec = env["T"], env["geo"][k]
    lv = level(env, n, ext, k)
    dense = lv["dense"]
    # the identity the input gradient rests on: nbr_k(o) = i  <=>  nbr_{124-k}(i) = o
    for kk in range(125):
        o = (dense[kk] >= 0).nonzero().squeeze(1)
        assert torch.equal(dense[124 - kk][dense[kk][o].long()].long(), o), f"offset {kk}"
        assert int((dense[kk] >= 0).sum()) == int((dense[124 - kk] >= 0).sum())
    for tr, var in V6_CONFIGS:
        km = codec._v6_map(dense, n, tr, var)
        dx = T.conv_dgrad(lv["dy"], env["W"][k], km)
        ok, ratio = within(dx, lv["dx"], lv["dx_abs"])
        assert ok, f"tile_rows {tr}: worst |err| / absref {ratio * 2 ** 16:.3f} * 2^-16"
        assert torch.equal(T.conv_dgrad(lv["dy"], env["W"][k], km), dx)
        print(f"dgrad n={n} K={k} tile_rows={tr}: worst |err| / absref {ratio * 2 ** 16:.3f} * 2^-16")


def conv64_dense(x, W125, dense):
    """sum_k x[nbr_k(o)] W[k] in the dtype of x, differentiable: the rows of all 125 offsets gathered at once"""
    n = x.shape[0]
    xp = torch.cat([x, x.new_zeros((1, x.shape[1]))])
    idx = torch.where(dense >= 0, dense.long(), torch.full_like(dense, n, dtype=torch.int64)).t()     # [n, 125]
    return torch.einsum("nkc,kcd->nd", xp[idx], W125)


@pytest.mark.parametrize("k", [5, 3])
def test_sparse_conv_fn_against_fp64_autograd(env, k):
    """y = ReLU(conv(x, W) + r) and a linear loss: both gradients and the residual's, against fp64 autograd of the dense-map conv.
    The ReLU mask of the reference is the kernel's own (an fp32 sum within 2^-16 of zero may fall on either side; that it agrees
    with the fp64 sign everywhere else is checked)"""
    T, codec, dev = env["T"], env["geo"][k], env["dev"]
    from gauspcc_b200.synth import hac_like_cloud
    keys, _ = codec.pack_keys(torch.tensor(hac_like_cloud(20_000, seed=1, extent_log2=12), device=dev))
    keys = torch.sort(keys).values
    km = codec.build_kmap(keys, family="v6")
    dense = codec.dense_map(keys)
    g = torch.Generator(device=dev).manual_seed(k)
    n = keys.shape[0]
    x0, r0, c = (torch.randn((n, 32), generator=g, device=dev) for _ in range(3))
    Wk0 = env["W"][k][list(T.K5_OF_K3)] if k == 3 else env["W"][k]
    x, r, Wk = (t.clone().requires_grad_() for t in (x0, r0, Wk0))
    pre = T.SparseConvFn.apply(x, Wk, km) + r
    (torch.relu(pre) * c).sum().backward()
    x64, r64, Wk64 = (t.double().requires_grad_() for t in (x0, r0, Wk0))
    W125 = T._to125(Wk64) if k == 3 else Wk64
    pre64 = conv64_dense(x64, W125, dense) + r64
    absref = conv64_dense(x0.double().abs(), T._to125(Wk0.double().abs()) if k == 3 else Wk0.double().abs(), dense) + r0.double().abs()
    ok, ratio = within(pre.detach(), pre64.detach(), absref)
    assert ok, ratio
    mask = pre.detach() > 0
    assert bool(((pre64.detach() > 0) == mask)[pre64.detach().abs() > BOUND_C * 2.0 ** -16 * absref].all())
    ((pre64 * mask) * c.double()).sum().backward()
    for name, a, b in (("x", x, x64), ("W", Wk, Wk64), ("r", r, r64)):
        rel = float((a.grad.double() - b.grad).norm() / b.grad.norm())
        print(f"SparseConvFn K={k} d{name}: relative L2 error {rel:.2e}")
        assert rel <= 1e-4, (name, rel)


@pytest.fixture(scope="module")
def clouds():
    from gauspcc_b200.synth import hac_like_cloud
    return {n: hac_like_cloud(n, seed=11, extent_log2=ext) for n, ext in ((20_000, 13), (100_000, 15))}


@pytest.mark.parametrize("n", [20_000, 100_000])
def test_network_forward_matches_the_codec(env, clouds, n):
    """the per-stage probabilities equal encode(..., collect=True)'s; the code length is within 1 % of the streams' bytes (the
    range coder's overhead and the rounding of the integer CDF rows are the gap)"""
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.weights import make_synthetic_state_dict
    T, dev = env["T"], env["dev"]
    sd = make_synthetic_state_dict(5)
    codec = GausPcgcCodec(DeviceWeights(sd, dev), dev)
    xyz = torch.tensor(clouds[n], device=dev)
    _, _, streams, aux = codec.encode(xyz, collect=True)
    net = T.GausPcgcNet(5, state_dict=sd).to(dev)
    with torch.no_grad():
        out = net(xyz, collect=True)
    assert len(out["probs"]) == len(aux["probs"]) == len(streams)
    worst = max(float((p - q).abs().max()) for p, q in zip(out["probs"], aux["probs"]))
    assert worst <= 1e-5, worst
    stream_bits = 8 * sum(len(s) for s in streams)
    gap = float(out["bits"]) / stream_bits - 1
    print(f"\nN={n}: worst |p - p_codec| {worst:.2e}; network {float(out['bits']):.0f} bits vs streams {stream_bits} bits ({100 * gap:+.3f} %)")
    assert abs(gap) <= 0.01


def reference_bits(P, levels, geo, K, relu_inputs):
    """Appendix A in float64 torch on dense maps, the network's parameters P (fp64 leaves): the code length of the streams under
    the coder's probabilities (p * (65536 - A) + 1) / 65536.
    relu_inputs: the fp32 network's ReLU inputs, in the order it applied them (this function applies its ReLUs in the same order).
    Each ReLU keeps the units the network kept: a pre-activation within rounding of zero can fall on either side in fp32, and one
    unit on the other side gates its whole gradient.  Returns (bits, units whose fp64 sign differs, their largest |fp64 value|
    relative to the largest |value| of their tensor)."""
    from gauspcc_b200 import weights as Wm
    from gauspcc_b200.codec import CTX_SHIFT, STAGE_MASK, STAGE_SHIFT
    from gauspcc_b200.train import K5_OF_K3, _octant

    def Wc(i):
        w = P[Wm.CONV_KEYS[i]]
        if K == 3:
            full = w.new_zeros((125, 32, 32))
            full = full.index_copy(0, torch.tensor(K5_OF_K3, device=w.device), w)
            return full
        return w

    flips = [0, 0.0]

    def relu(x):
        x32 = next(relu_inputs)
        assert x32.shape == x.shape
        keep = x32 > 0
        other = keep != (x.detach() > 0)
        if other.any():
            flips[0] += int(other.sum())
            flips[1] = max(flips[1], float(x.detach()[other].abs().max() / x.detach().abs().max()))
        return x * keep

    def stack(x, ids, dense):
        x = relu(conv64_dense(x, Wc(ids[0]), dense))
        for a, b in ((ids[1], ids[2]), (ids[3], ids[4])):
            x = relu(conv64_dense(relu(conv64_dense(x, Wc(a), dense)), Wc(b), dense) + x)
        return x

    dense = [geo.dense_map(lv.keys) for lv in levels]
    bits = 0.0
    for d in range(len(levels) - 1):
        parent, gt = levels[d], levels[d + 1]
        _, cp = geo.expand(parent, gt.n)
        f = stack(P["prior_embedding.weight"][parent.occ.long()], Wm.PRIOR_CONVS, dense[d])
        oc = _octant(gt.keys)
        u = stack(f[cp.long()] + P["target_embedding.target_res_embedding.weight"][oc], Wm.TARGET_CONVS, dense[d + 1])
        occ = gt.occ.long()
        for i in range(4):
            f = u if i == 0 else u + P[f"pred_head_s{i}_emb.weight"][occ >> CTX_SHIFT[i]]
            c0, c1 = Wm.stage_convs(i)
            t = conv64_dense(relu(conv64_dense(f, Wc(c0), dense[d + 1])), Wc(c1), dense[d + 1])
            h = relu(t @ P[f"pred_head_s{i}.0.weight"].t() + P[f"pred_head_s{i}.0.bias"])
            p = torch.softmax(h @ P[f"pred_head_s{i}.2.weight"].t() + P[f"pred_head_s{i}.2.bias"], dim=1)
            sym = (occ >> STAGE_SHIFT[i]) & STAGE_MASK[i]
            A = Wm.STAGE_ALPHABETS[i]
            bits = bits - torch.log2((p.gather(1, sym[:, None]) * (65536 - A) + 1) / 65536).sum()   # the coder's probability
    assert next(relu_inputs, None) is None
    return bits, flips[0], flips[1]


@pytest.mark.parametrize("k", [5, 3])
def test_whole_network_gradients_against_fp64(env, k, monkeypatch):
    from gauspcc_b200.synth import hac_like_cloud
    T, dev = env["T"], env["dev"]
    net = T.GausPcgcNet(k, seed=5).to(dev)
    xyz = torch.tensor(hac_like_cloud(5_000, seed=21, extent_log2=11), device=dev)
    relu_inputs, relu = [], torch.relu
    monkeypatch.setattr(torch, "relu", lambda t: (relu_inputs.append(t.detach().double()), relu(t))[1])
    out = net(xyz)
    monkeypatch.undo()
    out["bits"].backward()
    levels = net.geometry(xyz)
    P64 = {n: p.detach().double().requires_grad_() for n, p in net.named_parameters()}
    ref, flips, flip_mag = reference_bits(P64, levels, net.codec(dev), k, iter(relu_inputs))
    units = sum(t.numel() for t in relu_inputs)
    assert flips <= 1e-3 * units and flip_mag <= 1e-3, (flips, units, flip_mag)       # only values within rounding of zero
    ref.backward()
    assert abs(float(out["bits"]) / float(ref) - 1) <= 1e-4, (float(out["bits"]), float(ref))
    worst = 0.0
    for n, p in net.named_parameters():
        g64 = P64[n].grad
        rel = float((p.grad.double() - g64).norm() / g64.norm())
        worst = max(worst, rel)
        assert rel <= 1e-3, (n, rel)
    print(f"\nK={k}: {out['levels']} levels, bits {float(out['bits']):.1f}; worst per-parameter relative L2 error {worst:.2e}; "
          f"{flips} of {units} ReLU units on the other side of zero in fp64 (at most {flip_mag:.1e} of their tensor's largest value)")


def _patches(T, seed, n=32_000, max_points=8_000):
    from gauspcc_b200.synth import hac_like_cloud
    xyz = torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=13))
    return xyz, [xyz[i] for i in T.partition(xyz, max_points)]


def test_training_lowers_the_rate_and_the_checkpoint_codes(env, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.weights import make_synthetic_state_dict, validate_state_dict
    T, dev = env["T"], env["dev"]
    cloud, _ = _patches(T, 31)
    ck = str(tmp_path / "trained.pth")
    sd, rows = T.train([cloud], ck, steps=200, seed=3, kernel_size=5, max_points=8_000)
    first = float(np.mean([r["bpp"] for r in rows[:20]]))
    last = float(np.mean([r["bpp"] for r in rows[-20:]]))
    print(f"\nbpp: first 20 steps {first:.4f}, last 20 steps {last:.4f}; {rows[-1]['time']:.1f} s for 200 steps")
    assert last < first
    validate_state_dict(torch.load(ck), 32, 5)
    init = str(tmp_path / "init.pth")
    torch.save(make_synthetic_state_dict(5), init)
    _, held = _patches(T, 77)
    xyz = held[0].to(dev)
    sizes = {}
    for name, path in (("init", init), ("trained", ck)):
        r = pcc_utils.compress_point_cloud(xyz, path, str(tmp_path / f"{name}.bin"), kernel_size=5)
        dec = pcc_utils.decompress_point_cloud(str(tmp_path / f"{name}.bin"), path, kernel_size=5)["point_cloud"]
        assert np.array_equal(np.unique(dec.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz.cpu().numpy(), axis=0))
        sizes[name] = r["file_size_bits"]
    print(f"held-out patch of {xyz.shape[0]} points: {sizes['init'] / xyz.shape[0]:.4f} bpp with the initial weights, "
          f"{sizes['trained'] / xyz.shape[0]:.4f} bpp trained")
    assert sizes["trained"] < sizes["init"]


@pytest.mark.parametrize("k", [5, 3])
def test_training_is_deterministic(env, k):
    T = env["T"]
    cloud, _ = _patches(T, 41, n=16_000, max_points=4_000)
    a, ra = T.train([cloud], steps=30, seed=8, kernel_size=k, max_points=4_000)
    b, rb = T.train([cloud], steps=30, seed=8, kernel_size=k, max_points=4_000)
    assert [r["bpp"] for r in ra] == [r["bpp"] for r in rb]
    assert list(a) == list(b) and all(torch.equal(a[n], b[n]) for n in a)
    init = T.GausPcgcNet(k, seed=5).state_dict()
    assert not torch.equal(a["prior_resnet.0.kernel"], init["prior_resnet.0.kernel"])
    c, _ = T.train([cloud], steps=30, seed=9, kernel_size=k, max_points=4_000)          # another patch order
    assert not all(torch.equal(a[n], c[n]) for n in a)


def test_cli_train_then_compress_and_decompress(env, tmp_path):
    from gauspcc_b200 import cli, plyio
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import validate_state_dict
    dev = env["dev"]
    src = tmp_path / "in"
    src.mkdir()
    clouds = [hac_like_cloud(6_000, seed=s, extent_log2=12) for s in (1, 2)]
    for s, c in enumerate(clouds):
        plyio.write_ply_ascii(torch.tensor(c, dtype=torch.float32, device=dev), str(src / f"s{s}.ply"))
    ck = str(tmp_path / "ck" / "net.pth")
    res = str(tmp_path / "res")
    assert cli.main(["train", "--input_glob", str(src), "--ckpt_out", ck, "--steps", "6", "--kernel_size", "3", "--posQ", "1",
                     "--is_data_pre_quantized", "--max_points", "4000", "--resultdir", res]) == 0
    validate_state_dict(torch.load(ck), 32, 3)
    log = open(os.path.join(res, "ue_4stage_conv_train_data2.csv")).read().splitlines()
    assert log[0] == "step,points,bpp,time" and len(log) == 7
    enc, dec = str(tmp_path / "enc"), str(tmp_path / "dec")
    assert cli.main(["compress", "--input_glob", str(src), "--output_folder", enc, "--ckpt", ck, "--posQ", "1",
                     "--is_data_pre_quantized", "--resultdir", res]) == 0
    assert cli.main(["decompress", "--input_glob", enc, "--output_folder", dec, "--ckpt", ck, "--is_data_pre_quantized",
                     "--resultdir", res]) == 0
    for s, c in enumerate(clouds):
        got = cli.read_points(os.path.join(dec, f"s{s}.ply.bin.ply")).astype(np.int32)
        assert np.array_equal(np.unique(got, axis=0), np.unique(c, axis=0))
