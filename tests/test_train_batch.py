"""Minibatch training on the GPU: the pair-balanced weight gradient (gpc_spconv_wgrad_v6_balanced, csrc/spconv_grad.cu) against fp64
and against gpc_spconv_wgrad_v6, GausPcgcNet.forward_batch (union octrees of patches) against each patch's own forward, batched
training runs and `cli train --batch_size`.

Bound of the weight gradient as tests/test_train.py: |got - ref| <= 2 * 2^-16 * sum |x| |dy| per element."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

BOUND_C = 2.0
V6_CONFIGS = [(8, 47), (16, 46), (32, 46), (64, 42), (64, 48), (128, 48)]
LEVELS = [1_000, 30_000, 200_000, 1_200_000]            # the last: a union of eight 150 K-point HAC-like patches


@pytest.fixture(scope="module")
def env():
    from gauspcc_b200 import train as T
    from gauspcc_b200.codec import GausPcgcCodec
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    return {"T": T, "dev": dev, "geo": {k: GausPcgcCodec(T._Geometry(k), dev) for k in (3, 5)}}


def level_keys(codec, n):
    """sorted unique keys of a HAC-like level of about n rows; 1.2 M rows: eight 150 K patches stacked along z, as a union level"""
    from gauspcc_b200.synth import hac_like_cloud
    dev = codec.dev
    if n < 1_000_000:
        xyz = torch.tensor(hac_like_cloud(n, seed=n, extent_log2={1_000: 9, 30_000: 12, 200_000: 14}[n]), device=dev)
    else:
        parts = []
        for s in range(8):
            p = torch.tensor(hac_like_cloud(150_000, seed=40 + s, extent_log2=16), device=dev)
            p[:, 2] += (s - 4) * (1 << 17)
            parts.append(p)
        xyz = torch.cat(parts)
    keys, _ = codec.pack_keys(xyz)
    return torch.unique(keys)


def fp64_wgrad(dense, x, dy):
    x64, d64 = x.double(), dy.double()
    dW = torch.zeros((125, 32, 32), dtype=torch.float64, device=x.device)
    dW_abs = torch.zeros_like(dW)
    for kk in range(125):
        o = (dense[kk] >= 0).nonzero().squeeze(1)
        if o.numel():
            i = dense[kk][o].long()
            dW[kk] = x64[i].t() @ d64[o]
            dW_abs[kk] = x64[i].abs().t() @ d64[o].abs()
    return dW, dW_abs


def worst(got, ref, absref):
    err = (got.double() - ref).abs()
    return bool((err <= BOUND_C * 2.0 ** -16 * absref + 1e-30).all()), float((err / absref.clamp(min=1e-30)).max())


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("n", LEVELS)
def test_balanced_wgrad_against_fp64(env, n, k):
    T, codec, dev = env["T"], env["geo"][k], env["dev"]
    keys = level_keys(codec, n)
    rows = keys.shape[0]
    dense = codec.dense_map(keys)
    g = torch.Generator(device=dev).manual_seed(n + k)
    x = torch.randn((rows, 32), generator=g, device=dev)
    dy = torch.randn((rows, 32), generator=g, device=dev)
    ref, absref = fp64_wgrad(dense, x, dy)
    absent = absref.flatten(1).amax(1) == 0
    worst_bal = worst_old = 0.0
    for tr, var in V6_CONFIGS:
        km = codec._v6_map(dense, rows, tr, var)
        dW = T.conv_wgrad(x, dy, km, balanced=True)
        ok, ratio = worst(dW, ref, absref)
        assert ok, f"rows {rows} tile_rows {tr}: worst |err| / absref {ratio * 2 ** 16:.3f} * 2^-16"
        worst_bal = max(worst_bal, ratio)
        assert bool((dW[absent] == 0).all()) and not bool(torch.signbit(dW[absent]).any())     # absent offsets: exact +0
        assert torch.equal(T.conv_wgrad(x, dy, km, balanced=True), dW)                          # same bits on every call
        old = T.conv_wgrad(x, dy, km)
        ok, ratio = worst(dW, old.double(), absref)
        assert ok, f"rows {rows} tile_rows {tr}: balanced vs gpc_spconv_wgrad_v6 {ratio * 2 ** 16:.3f} * 2^-16"
        worst_old = max(worst_old, ratio)
    print(f"\nbalanced wgrad rows={rows} K={k}: worst |err| / absref {worst_bal * 2 ** 16:.3f} * 2^-16 (fp64), "
          f"{worst_old * 2 ** 16:.3f} * 2^-16 against gpc_spconv_wgrad_v6")


def test_balanced_wgrad_centre_only_level(env):
    """rows without neighbours but themselves: dW[62] = x^T dy, every other offset +0"""
    T, codec, dev = env["T"], env["geo"][5], env["dev"]
    keys, _ = codec.pack_keys(torch.tensor([[8 * i, 0, 0] for i in range(1000)], dtype=torch.int32, device=dev))
    keys = torch.sort(keys).values
    dense = codec.dense_map(keys)
    x, dy = torch.randn((1000, 32), device=dev), torch.randn((1000, 32), device=dev)
    ref = x.double().t() @ dy.double()
    absref = x.double().abs().t() @ dy.double().abs()
    for tr, var in V6_CONFIGS:
        dW = T.conv_wgrad(x, dy, codec._v6_map(dense, 1000, tr, var), balanced=True)
        assert bool(((dW[62].double() - ref).abs() <= BOUND_C * 2.0 ** -16 * absref).all())
        others = torch.cat([dW[:62], dW[63:]])
        assert bool((others == 0).all()) and not bool(torch.signbit(others).any())


def test_balanced_wgrad_rejects_bad_arguments(env):
    from gauspcc_b200 import _lib
    lib = _lib.load()
    f = lib.gpc_spconv_wgrad_v6_balanced
    assert f(None, None, None, None, -1, 64, 0, None, None, 0, None) == -1                 # n < 0
    assert f(None, None, None, None, 100, 24, 100, None, None, 0, None) == -1               # not a tile height of the conv
    assert f(None, None, None, None, 100, 64, -8, None, None, 0, None) == -1                # negative entry count
    assert f(None, None, None, None, 100, 64, 800, None, None, 0, None) == -4               # workspace too small
    ws = lib.gpc_spconv_wgrad_balanced_workspace_bytes(100, 64, 800)
    assert f(None, None, None, None, 100, 64, 800, None, None, ws - 1, None) == -4
    assert lib.gpc_spconv_wgrad_balanced_workspace_bytes(0, 64, 0) == 0
    assert lib.gpc_spconv_wgrad_balanced_workspace_bytes(1_000_000, 128, 10_000_000) > \
        lib.gpc_spconv_wgrad_balanced_workspace_bytes(1_000_000, 128, 1_000_000)


def test_balanced_wgrad_stays_inside_its_workspace(env):
    """a workspace of exactly the queried size, followed by a guard region: on the 1.2 M-row union level nothing is written past
    it, and the result is the one a roomier workspace gives"""
    from gauspcc_b200 import _lib
    from gauspcc_b200.codec import _ptr
    T, codec, dev = env["T"], env["geo"][5], env["dev"]
    lib = _lib.load()
    keys = level_keys(codec, 1_200_000)
    rows = keys.shape[0]
    km = codec.build_kmap(keys, family="v6")
    x, dy = torch.randn((rows, 32), device=dev), torch.randn((rows, 32), device=dev)
    ws_b = int(lib.gpc_spconv_wgrad_balanced_workspace_bytes(rows, km.tile_rows, km.n_pairs))
    buf = torch.full((ws_b + 65536,), 0x5A, dtype=torch.uint8, device=dev)
    dW = torch.empty((125, 32, 32), device=dev)
    assert lib.gpc_spconv_wgrad_v6_balanced(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pairs), rows, km.tile_rows, km.n_pairs, _ptr(dW),
                                            _ptr(buf), ws_b, torch.cuda.current_stream(dev).cuda_stream) == 0
    torch.cuda.synchronize()
    assert bool((buf[ws_b:] == 0x5A).all())
    assert torch.equal(dW, T.conv_wgrad(x, dy, km, balanced=True))


# ---------------------------------------------------------------------------------------------------------------- forward_batch
def mixed_patches():
    """four patches of different sizes and depths, one far from the origin (recentred by geometry, as the encoder does)"""
    from gauspcc_b200.synth import hac_like_cloud
    a = hac_like_cloud(9_000, seed=1, extent_log2=13)
    b = hac_like_cloud(3_000, seed=2, extent_log2=10)
    c = hac_like_cloud(14_000, seed=3, extent_log2=14) + np.array([600_000, -500_000, 700_000], dtype=np.int32)
    d = hac_like_cloud(800, seed=4, extent_log2=8)
    return [torch.tensor(p) for p in (a, b, c, d)]


def grads(net):
    return {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}


def single_runs(T, dev, k, patches, tiling=None):
    """each patch through forward(xyz) alone: (summed bits, per patch its probability rows, summed gradients); tiling = (tile_rows,
    variant) forces one mma.sync tiling on every level instead of the size-dependent one"""
    net = T.GausPcgcNet(k, seed=5).to(dev)
    if tiling is not None:
        c = net.codec(dev)
        c.adaptive_tiles, c.tile_rows, c.v6_variant = False, tiling[0], tiling[1]
    bits, probs, tot = 0.0, [], None
    for p in patches:
        net.zero_grad(set_to_none=True)
        o = net(p, collect=True)
        o["bits"].backward()
        bits += float(o["bits"].detach())
        probs.append(o["probs"])
        g = grads(net)
        tot = g if tot is None else {n: tot[n] + g[n] for n in tot}
    return bits, probs, tot


def prob_gap(a, b):
    worst = 0.0
    for mine, theirs in zip(a, b):
        assert len(mine) == len(theirs)
        for x, y in zip(mine, theirs):
            assert x.shape == y.shape
            worst = max(worst, float((x - y).abs().max()))
    return worst


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))


def check_batch(T, dev, k, union_max_rows=None, expect_unions=0):
    """forward_batch against each patch's forward(xyz).  A union level takes its conv tiling from its own row count, so a patch's rows
    are summed in another fp32 order than in its own level (same neighbours, parents and weights).  How far that alone moves the
    probabilities and gradients is measured here: the single patches again with one other tiling forced on every level.  The union
    must stay within twice that spread (and within 2e-6 / 1e-4, the bounds for a batch whose tilings all match, where it is smaller)."""
    patches = [p.to(dev) for p in mixed_patches()]
    singles, probs1, ref_g = single_runs(T, dev, k, patches)
    _, probs_alt, alt_g = single_runs(T, dev, k, patches, tiling=(8, 47))
    net = T.GausPcgcNet(k, seed=5).to(dev)
    if union_max_rows is not None:
        net.union_max_rows = union_max_rows
    out = net.forward_batch(patches, collect=True)
    out["bits"].backward()
    assert out["unions"] == expect_unions if expect_unions else out["unions"] >= 2, out["unions"]
    assert out["patches"] == 4 and out["points"] == sum(int(p.shape[0]) for p in patches)
    rel_bits = abs(float(out["bits"]) / singles - 1)
    assert rel_bits <= 1e-5, rel_bits
    assert abs(float(out["bpp"]) - float(out["bits"]) / out["points"]) <= 1e-6 * float(out["bpp"])
    worst_p, floor_p = prob_gap(out["probs"], probs1), prob_gap(probs_alt, probs1)
    assert worst_p <= max(2e-6, 2 * floor_p), (worst_p, floor_p)
    g = grads(net)
    worst_g = floor_g = 0.0
    for n, r in ref_g.items():
        rel, floor = rel_l2(g[n], r), rel_l2(alt_g[n], r)
        worst_g, floor_g = max(worst_g, rel), max(floor_g, floor)
        assert rel <= max(1e-4, 2 * floor), (n, rel, floor)
    print(f"\nK={k} unions={out['unions']}: bits {float(out['bits']):.1f} vs per-patch sum {singles:.1f} (rel {rel_bits:.1e}); "
          f"worst |p - p_single| {worst_p:.1e} (another tiling alone: {floor_p:.1e}); worst per-parameter gradient relative L2 "
          f"{worst_g:.2e} (another tiling alone: {floor_g:.2e})")


@pytest.mark.parametrize("k", [5, 3])
def test_union_batch_matches_single_patches(env, k):
    check_batch(env["T"], env["dev"], k, expect_unions=1)


@pytest.mark.parametrize("k", [5, 3])
def test_several_unions_match_single_patches(env, k):
    """a row cap below the batch's rows: plan_unions splits it into two or more unions, which run in turn"""
    check_batch(env["T"], env["dev"], k, union_max_rows=16_000)


# ---------------------------------------------------------------------------------------------------------------- training
def _cloud(seed, n=16_000, ext=13):
    from gauspcc_b200.synth import hac_like_cloud
    return torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=ext))


@pytest.mark.parametrize("k", [5, 3])
def test_batched_training_is_deterministic(env, k):
    T = env["T"]
    cloud = _cloud(41)
    a, ra = T.train([cloud], steps=12, seed=8, kernel_size=k, max_points=2_000, batch_size=4)
    b, rb = T.train([cloud], steps=12, seed=8, kernel_size=k, max_points=2_000, batch_size=4)
    assert [r["bpp"] for r in ra] == [r["bpp"] for r in rb]
    assert all(torch.equal(a[n], b[n]) for n in a)
    assert all(r["points"] > 2_000 for r in ra)                                # four patches of ~2 000 points per step
    init = T.GausPcgcNet(k, seed=5).state_dict()
    assert not torch.equal(a["prior_resnet.0.kernel"], init["prior_resnet.0.kernel"])


def test_batch_size_one_is_the_default(env):
    T = env["T"]
    cloud = _cloud(41)
    a, ra = T.train([cloud], steps=10, seed=8, kernel_size=5, max_points=4_000)
    b, rb = T.train([cloud], steps=10, seed=8, kernel_size=5, max_points=4_000, batch_size=1)
    assert [(r["points"], r["bpp"]) for r in ra] == [(r["points"], r["bpp"]) for r in rb]
    assert all(torch.equal(a[n], b[n]) for n in a)
    with pytest.raises(ValueError):
        T.train([cloud], steps=1, max_points=4_000, batch_size=5)             # 4 patches


def test_batched_training_lowers_the_rate_and_the_checkpoint_codes(env, tmp_path):
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.weights import make_synthetic_state_dict
    T, dev = env["T"], env["dev"]
    cloud = _cloud(31, n=64_000)
    ck = str(tmp_path / "trained.pth")
    sd, rows = T.train([cloud], ck, steps=100, seed=3, kernel_size=5, max_points=4_000, batch_size=8)
    first = float(np.mean([r["bpp"] for r in rows[:10]]))
    last = float(np.mean([r["bpp"] for r in rows[-10:]]))
    print(f"\nB=8: bpp first 10 steps {first:.4f}, last 10 steps {last:.4f}; {rows[-1]['time']:.1f} s for 100 steps")
    assert last < first
    init = str(tmp_path / "init.pth")
    torch.save(make_synthetic_state_dict(5), init)
    held = _cloud(77, n=32_000)
    xyz = held[T.partition(held, 8_000)[0]].to(dev)
    sizes = {}
    for name, path in (("init", init), ("trained", ck)):
        r = pcc_utils.compress_point_cloud(xyz, path, str(tmp_path / f"{name}.bin"), kernel_size=5)
        dec = pcc_utils.decompress_point_cloud(str(tmp_path / f"{name}.bin"), path, kernel_size=5)["point_cloud"]
        assert np.array_equal(np.unique(dec.cpu().numpy().astype(np.int32), axis=0), np.unique(xyz.cpu().numpy(), axis=0))
        sizes[name] = r["file_size_bits"]
    print(f"held-out patch of {xyz.shape[0]} points: {sizes['init'] / xyz.shape[0]:.4f} bpp initial, "
          f"{sizes['trained'] / xyz.shape[0]:.4f} bpp trained")
    assert sizes["trained"] < sizes["init"]


def test_cli_train_batch_size_then_compress_and_decompress(env, tmp_path):
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
    assert cli.main(["train", "--input_glob", str(src), "--ckpt_out", ck, "--steps", "4", "--kernel_size", "3", "--posQ", "1",
                     "--is_data_pre_quantized", "--max_points", "2000", "--batch_size", "4", "--resultdir", res]) == 0
    validate_state_dict(torch.load(ck), 32, 3)
    log = open(os.path.join(res, "ue_4stage_conv_train_data2.csv")).read().splitlines()
    assert log[0] == "step,points,bpp,time" and len(log) == 5
    assert all(int(r.split(",")[1]) > 2_000 for r in log[1:])
    enc, dec = str(tmp_path / "enc"), str(tmp_path / "dec")
    assert cli.main(["compress", "--input_glob", str(src), "--output_folder", enc, "--ckpt", ck, "--posQ", "1",
                     "--is_data_pre_quantized", "--resultdir", res]) == 0
    assert cli.main(["decompress", "--input_glob", enc, "--output_folder", dec, "--ckpt", ck, "--is_data_pre_quantized",
                     "--resultdir", res]) == 0
    for s, c in enumerate(clouds):
        got = cli.read_points(os.path.join(dec, f"s{s}.ply.bin.ply")).astype(np.int32)
        assert np.array_equal(np.unique(got, axis=0), np.unique(c, axis=0))
