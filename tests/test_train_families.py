"""Training on the codec's sparse and tcgen05 conv families (gauspcc_b200/train.py, csrc/spconv_grad.cu): gpc_spconv_wgrad_sparse and
gpc_spconv_wgrad_um against fp64, the input gradient through each family's mirrored-weight forward, the mirror identity on the
families' own maps, SparseConvFn against fp64 autograd, GausPcgcNet(conv_families="codec") against the mma.sync network on union
levels that take all three families, and short "codec" training runs.

Bound of the gradients as tests/test_train.py: |got - ref| <= 2 * 2^-16 * sum of |products| per element."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

BOUND_C = 2.0
SIZES = [1_000, 150_000, 600_000, 1_200_000]
FAMILIES = ["sparse", "um"]


@pytest.fixture(scope="module")
def env():
    from gauspcc_b200 import train as T
    from gauspcc_b200.codec import GausPcgcCodec
    from gauspcc_b200.weights import CONV_KEYS, make_synthetic_state_dict
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    geo = {k: GausPcgcCodec(T._Geometry(k), dev) for k in (3, 5)}
    W = {k: T._to125(make_synthetic_state_dict(5, 32, k)[CONV_KEYS[7]].to(dev)) for k in (3, 5)}
    return {"T": T, "dev": dev, "geo": geo, "W": W}


def hac(n, seed, dev):
    from gauspcc_b200.synth import hac_like_cloud
    return torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=16), device=dev)


def cube(n, seed, dev):
    """n voxels drawn without repetition from a cube 3x their count (about 40 neighbours per row in 5^3)"""
    side = int(round((3 * n) ** (1 / 3))) + 1
    g = torch.Generator(device=dev).manual_seed(seed)
    idx = torch.randperm(side ** 3, generator=g, device=dev)[:n]
    return torch.stack([idx % side, (idx // side) % side, idx // (side * side)], 1).to(torch.int32)


def level_keys(codec, kind, n):
    """the shapes of profiles/r07_train_batch.md: a sparse HAC-like finest level (150 K-point patches stacked along z, as a union
    level) or a dense coarse level"""
    dev = codec.dev
    if kind == "dense":
        xyz = cube(n, n, dev)
    else:
        parts, left, s = [], n, 0
        while left > 0:
            p = hac(min(left, 150_000), 500 + s, dev)
            p[:, 2] += (s - 4) * (1 << 17)
            parts.append(p)
            left -= p.shape[0]
            s += 1
        xyz = torch.cat(parts)
    keys, _ = codec.pack_keys(xyz)
    return torch.unique(keys)


def fp64_refs(dense, x, dy, W):
    """dW, dx and the sums of magnitudes that bound them, in fp64 over the dense map"""
    x64, d64, W64 = x.double(), dy.double(), W.double()
    dW = torch.zeros((125, 32, 32), dtype=torch.float64, device=x.device)
    dW_abs, dx, dx_abs = torch.zeros_like(dW), torch.zeros_like(x64), torch.zeros_like(x64)
    for kk in range(125):
        o = (dense[kk] >= 0).nonzero().squeeze(1)
        if o.numel() == 0:
            continue
        i = dense[kk][o].long()
        dW[kk] = x64[i].t() @ d64[o]
        dW_abs[kk] = x64[i].abs().t() @ d64[o].abs()
        dx.index_add_(0, i, d64[o] @ W64[kk].t())
        dx_abs.index_add_(0, i, d64[o].abs() @ W64[kk].abs().t())
    return dW, dW_abs, dx, dx_abs


def within(got, ref, absref):
    err = (got.double() - ref).abs()
    return bool((err <= BOUND_C * 2.0 ** -16 * absref + 1e-30).all()), float((err / absref.clamp(min=1e-30)).max())


def map_triples(km, n):
    """the (offset, output row, input row) triples a sparse or tcgen05 map holds, sorted, as int64 keys (k * n + o) * n + i"""
    dev = km.seg.device
    if km.um_rows:
        q = torch.arange(km.n_pairs, device=dev)
        nbr = km.pair_nbr.long() & 0xFFFFFFFF
        real = nbr != 0xFFFFFFFF
        cell = torch.searchsorted(km.seg.long(), q, right=True) - 1
        k = cell % 126
        o = (cell // 126) * km.um_rows + (km.pair_off.long() >> 7)
        k, o, i = k[real], o[real], nbr[real]
    else:
        e = km.pairs[:km.n_pairs]
        nbr = e & 0xFFFFFFFF
        real = nbr != 0xFFFFFFFF
        q = torch.arange(km.n_pairs, device=dev)[real]
        cell = torch.searchsorted(km.seg.long(), q, right=True) - 1
        kk = cell % 125
        k = kk + (kk >= 62).long()
        dst = (e[real] >> 32) & 0xFFFFFFFF
        o = torch.searchsorted(km.rowptr.long(), dst, right=True) - 1      # the row whose contributions hold slot dst
        rows = torch.arange(n, device=dev)
        k = torch.cat([k, torch.full_like(rows, 62)])
        o, i = torch.cat([o, rows]), torch.cat([nbr[real], rows])
    return torch.sort((k * n + o) * n + i).values


def run_wgrad_raw(env, fam, km, x, dy, guard=65536):
    """the family's wgrad through the C ABI with a workspace of exactly the queried size followed by a canary region"""
    from gauspcc_b200 import _lib
    from gauspcc_b200.codec import _ptr
    lib, dev, n = _lib.load(), env["dev"], x.shape[0]
    st = torch.cuda.current_stream(dev).cuda_stream
    dW = torch.empty((125, 32, 32), device=dev)
    if fam == "um":
        ws_b = int(lib.gpc_spconv_wgrad_um_workspace_bytes(n, km.um_rows, km.n_pairs))
        buf = torch.full((ws_b + guard,), 0x5A, dtype=torch.uint8, device=dev)
        rc = lib.gpc_spconv_wgrad_um(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(km.pair_off), n, km.um_rows, km.n_pairs,
                                     _ptr(dW), _ptr(buf), ws_b, st)
    else:
        ws_b = int(lib.gpc_spconv_wgrad_sparse_workspace_bytes(n, km.n_pairs))
        buf = torch.full((ws_b + guard,), 0x5A, dtype=torch.uint8, device=dev)
        rc = lib.gpc_spconv_wgrad_sparse(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pairs), _ptr(km.rowptr), n, km.n_pairs, _ptr(dW),
                                         _ptr(buf), ws_b, st)
    assert rc == 0
    torch.cuda.synchronize()
    assert bool((buf[ws_b:] == 0x5A).all()), "the kernel wrote past its workspace"
    return dW


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kind", ["sparse", "dense"])
def test_family_gradients_against_fp64(env, kind, n, k):
    """on one level, both families' maps: the map holds exactly the dense map's pairs and is symmetric (nbr_k(o) = i <=>
    nbr_{124-k}(i) = o, what the input gradient rests on), wgrad and dgrad within the fp64 bound, absent offsets +0, the same bits
    on every call, and the workspace bound"""
    T, codec, dev = env["T"], env["geo"][k], env["dev"]
    keys = level_keys(codec, kind, n)
    rows = keys.shape[0]
    dense = codec.dense_map(keys)
    g = torch.Generator(device=dev).manual_seed(n + k)
    x = torch.randn((rows, 32), generator=g, device=dev)
    dy = torch.randn((rows, 32), generator=g, device=dev)
    W = env["W"][k]
    dW_ref, dW_abs, dx_ref, dx_abs = fp64_refs(dense, x, dy, W)
    absent = dW_abs.flatten(1).amax(1) == 0
    # the dense map's triples, and their mirror images
    o_all = [(dense[kk] >= 0).nonzero().squeeze(1) for kk in range(125)]
    kd = torch.cat([torch.full_like(o, kk) for kk, o in enumerate(o_all)])
    od = torch.cat(o_all)
    idn = torch.cat([dense[kk][o].long() for kk, o in enumerate(o_all)])
    want = torch.sort((kd * rows + od) * rows + idn).values
    mirror = torch.sort(((124 - kd) * rows + idn) * rows + od).values
    assert torch.equal(want, mirror)
    del o_all, kd, od, idn, mirror
    for fam in FAMILIES:
        km = codec.build_kmap(keys, family=fam)
        assert T.kmap_family(km) == fam
        assert torch.equal(map_triples(km, rows), want), f"{fam} map differs from the dense map"
        dW = T.conv_wgrad(x, dy, km)
        ok, ratio_w = within(dW, dW_ref, dW_abs)
        assert ok, f"{fam} wgrad rows {rows}: worst |err| / absref {ratio_w * 2 ** 16:.3f} * 2^-16"
        assert bool((dW[absent] == 0).all()) and not bool(torch.signbit(dW[absent]).any())       # absent offsets: exact +0
        assert torch.equal(T.conv_wgrad(x, dy, km), dW)                                          # same bits on every call
        assert torch.equal(run_wgrad_raw(env, fam, km, x, dy), dW)
        dx = T.conv_dgrad(dy, W, km)
        ok, ratio_x = within(dx, dx_ref, dx_abs)
        assert ok, f"{fam} dgrad rows {rows}: worst |err| / absref {ratio_x * 2 ** 16:.3f} * 2^-16"
        assert torch.equal(T.conv_dgrad(dy, W, km), dx)
        print(f"\n{kind} level rows={rows} K={k} {fam} map ({km.n_real / rows:.2f} pairs per row): worst |err| / absref wgrad "
              f"{ratio_w * 2 ** 16:.3f} * 2^-16, dgrad {ratio_x * 2 ** 16:.3f} * 2^-16")
        del km
    torch.cuda.empty_cache()


def test_family_wgrad_centre_only_and_padding(env):
    """rows without neighbours but themselves: dW[62] = x^T dy and every other offset +0, on both maps (the sparse map has no
    straggler at all, the tcgen05 map pads every centre cell); 8192 + 5 rows put a partial 8-row unit in a second block"""
    T, codec, dev = env["T"], env["geo"][5], env["dev"]
    n = 8192 + 5
    keys, _ = codec.pack_keys(torch.tensor([[8 * (i % 4096), 8 * (i // 4096), 0] for i in range(n)], dtype=torch.int32, device=dev))
    keys = torch.sort(keys).values
    x, dy = torch.randn((n, 32), device=dev), torch.randn((n, 32), device=dev)
    ref = x.double().t() @ dy.double()
    absref = x.double().abs().t() @ dy.double().abs()
    for fam in FAMILIES:
        km = codec.build_kmap(keys, family=fam)
        dW = T.conv_wgrad(x, dy, km)
        assert bool(((dW[62].double() - ref).abs() <= BOUND_C * 2.0 ** -16 * absref).all()), fam
        others = torch.cat([dW[:62], dW[63:]])
        assert bool((others == 0).all()) and not bool(torch.signbit(others).any()), fam


def test_family_wgrad_rejects_bad_arguments(env):
    from gauspcc_b200 import _lib
    lib = _lib.load()
    um, sp = lib.gpc_spconv_wgrad_um, lib.gpc_spconv_wgrad_sparse
    assert um(None, None, None, None, None, -1, 512, 0, None, None, 0, None) == -1              # n < 0
    assert um(None, None, None, None, None, 1000, 256, 32, None, None, 0, None) == -1           # not the tcgen05 tile height
    assert um(None, None, None, None, None, 1000, 512, 24, None, None, 0, None) == -1           # entries not whole 16-entry cells
    assert um(None, None, None, None, None, 1000, 512, -16, None, None, 0, None) == -1
    assert um(None, None, None, None, None, 1000, 512, 1 << 32, None, None, 0, None) == -1
    ws = lib.gpc_spconv_wgrad_um_workspace_bytes(1000, 512, 3200)
    assert um(None, None, None, None, None, 1000, 512, 3200, None, None, ws - 1, None) == -4     # workspace too small
    assert sp(None, None, None, None, None, -1, 0, None, None, 0, None) == -1
    assert sp(None, None, None, None, None, 40_000_000, 0, None, None, 0, None) == -1           # n * 124 >= 2^32
    assert sp(None, None, None, None, None, 1000, 12, None, None, 0, None) == -1                # entries not whole 8-entry units
    ws = lib.gpc_spconv_wgrad_sparse_workspace_bytes(1000, 800)
    assert sp(None, None, None, None, None, 1000, 800, None, None, ws - 1, None) == -4
    assert lib.gpc_spconv_wgrad_um_workspace_bytes(0, 512, 0) == 0
    assert lib.gpc_spconv_wgrad_sparse_workspace_bytes(0, 0) == 0
    assert lib.gpc_spconv_wgrad_sparse_workspace_bytes(1_000_000, 8_000_000) > lib.gpc_spconv_wgrad_sparse_workspace_bytes(1_000_000, 0)


def conv64_dense(x, W125, dense):
    n = x.shape[0]
    xp = torch.cat([x, x.new_zeros((1, x.shape[1]))])
    idx = torch.where(dense >= 0, dense.long(), torch.full_like(dense, n, dtype=torch.int64)).t()
    return torch.einsum("nkc,kcd->nd", xp[idx], W125)


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("fam", FAMILIES)
def test_sparse_conv_fn_against_fp64_autograd(env, fam, k):
    """y = ReLU(conv(x, W) + r) and a linear loss on a sparse or tcgen05 map: the three gradients against fp64 autograd of the
    dense-map conv (the ReLU mask is the kernel's own, as in tests/test_train.py)"""
    T, codec, dev = env["T"], env["geo"][k], env["dev"]
    keys, _ = codec.pack_keys(hac(20_000, 1, dev) // 8)
    keys = torch.unique(keys)
    km = codec.build_kmap(keys, family=fam)
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
        print(f"SparseConvFn {fam} ({km.n_real / n:.2f} pairs per row) K={k} d{name}: relative L2 error {rel:.2e}")
        assert rel <= 5e-6, (name, rel)


# ------------------------------------------------------------------------------------------------------------ whole network
def mixed_batch(dev):
    """two sparse HAC-like patches and two dense ones; with a row cap of 220 K the planner puts each pair in one union (deepest first),
    whose finest level is then a sparse or a dense level of about 200 K rows"""
    return [hac(100_000, 61, dev), hac(100_000, 62, dev), cube(100_000, 63, dev), cube(100_000, 64, dev)]


def grads(net):
    return {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}


def batch_run(T, dev, patches, families, tiling=None):
    net = T.GausPcgcNet(5, seed=5, conv_families=families).to(dev)
    net.union_max_rows = 220_000
    if tiling is not None:
        c = net.codec(dev)
        c.adaptive_tiles, c.tile_rows, c.v6_variant = False, tiling[0], tiling[1]
    out = net.forward_batch(patches, collect=True)
    out["bits"].backward()
    return out, grads(net)


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


def test_codec_families_match_the_mma_sync_network(env):
    """the same batch through conv_families="codec" and "v6": the codec's family rule gives its union levels all three families
    (checked on the reported counts); bits agree to 1e-5, probabilities and every parameter's gradient stay within twice what a
    change of mma.sync tiling alone moves them (measured here, as tests/test_train_batch.py's check_batch does)"""
    T, dev = env["T"], env["dev"]
    patches = mixed_batch(dev)
    ref, ref_g = batch_run(T, dev, patches, "v6")
    alt, alt_g = batch_run(T, dev, patches, "v6", tiling=(8, 47))
    got, got_g = batch_run(T, dev, patches, "codec")
    assert ref["families"]["sparse"] == ref["families"]["um"] == 0 and ref["families"]["v6"] > 0
    fams = got["families"]
    assert fams["v6"] > 0 and fams["sparse"] > 0 and fams["um"] > 0, fams
    assert got["unions"] == ref["unions"] >= 2
    rel_bits = abs(float(got["bits"].detach()) / float(ref["bits"].detach()) - 1)
    assert rel_bits <= 1e-5, rel_bits
    worst_p, floor_p = prob_gap(got["probs"], ref["probs"]), prob_gap(alt["probs"], ref["probs"])
    assert worst_p <= max(2e-6, 2 * floor_p), (worst_p, floor_p)
    worst_g = floor_g = 0.0
    for n, r in ref_g.items():
        rel, floor = rel_l2(got_g[n], r), rel_l2(alt_g[n], r)
        worst_g, floor_g = max(worst_g, rel), max(floor_g, floor)
        assert rel <= max(1e-4, 2 * floor), (n, rel, floor)
    print(f"\nfamilies {fams}, {got['unions']} unions: bits {float(got['bits'].detach()):.1f} vs {float(ref['bits'].detach()):.1f} "
          f"(rel {rel_bits:.1e}); "
          f"worst |p - p_v6| {worst_p:.1e} (another tiling alone: {floor_p:.1e}); worst per-parameter gradient relative L2 "
          f"{worst_g:.2e} (another tiling alone: {floor_g:.2e})")


def test_codec_families_single_patch_forward(env):
    """forward() on one patch with a finest level above 150 K rows: the codec's rule puts that level on the sparse conv; the bits
    match the mma.sync network's to 1e-5"""
    T, dev = env["T"], env["dev"]
    xyz = hac(200_000, 71, dev)
    v6 =T.GausPcgcNet(5, seed=5).to(dev)
    co = T.GausPcgcNet(5, seed=5, conv_families="codec").to(dev)
    with torch.no_grad():
        ov, oc = v6(xyz), co(xyz)
    assert ov["families"] == {"v6": ov["levels"] + 1, "sparse": 0, "um": 0}
    assert oc["families"]["sparse"] >= 1 and sum(oc["families"].values()) == oc["levels"] + 1
    assert abs(float(oc["bits"]) / float(ov["bits"]) - 1) <= 1e-5


# ------------------------------------------------------------------------------------------------------------ training
def train_clouds():
    from gauspcc_b200.synth import hac_like_cloud
    return [torch.tensor(hac_like_cloud(200_000, seed=31, extent_log2=16))]


def test_codec_training_is_deterministic_lowers_the_rate_and_codes(env, tmp_path):
    """four 50 K-point patches per step: their union's finest level (~200 K rows) runs the sparse conv and its gradients"""
    from gauspcc_b200 import pcc_utils
    from gauspcc_b200.weights import make_synthetic_state_dict
    T, dev = env["T"], env["dev"]
    clouds = train_clouds()
    net = T.GausPcgcNet(5, seed=5, conv_families="codec").to(dev)
    patches = [clouds[0][i].to(dev) for i in T.partition(clouds[0], 50_000)]
    with torch.no_grad():
        fams = net.forward_batch(patches)["families"]
    assert fams["sparse"] >= 1, fams
    ck = str(tmp_path / "codec.pth")
    a, ra = T.train(clouds, ck, steps=40, seed=3, kernel_size=5, max_points=50_000, batch_size=4, conv_families="codec")
    b, rb = T.train(clouds, steps=40, seed=3, kernel_size=5, max_points=50_000, batch_size=4, conv_families="codec")
    assert [r["bpp"] for r in ra] == [r["bpp"] for r in rb]
    assert all(torch.equal(a[n], b[n]) for n in a)
    v, _ = T.train(clouds, steps=40, seed=3, kernel_size=5, max_points=50_000, batch_size=4)
    assert not all(torch.equal(a[n], v[n]) for n in a)                      # other kernels, other sums
    first = float(np.mean([r["bpp"] for r in ra[:10]]))
    last = float(np.mean([r["bpp"] for r in ra[-10:]]))
    print(f"\ncodec families, B=4: bpp first 10 steps {first:.4f}, last 10 steps {last:.4f}; {ra[-1]['time']:.1f} s for 40 steps")
    assert last < first
    init = str(tmp_path / "init.pth")
    torch.save(make_synthetic_state_dict(5), init)
    from gauspcc_b200.synth import hac_like_cloud
    held = torch.tensor(hac_like_cloud(32_000, seed=77, extent_log2=13))
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


def test_v6_families_are_the_default(env):
    T = env["T"]
    from gauspcc_b200.synth import hac_like_cloud
    cloud = torch.tensor(hac_like_cloud(16_000, seed=41, extent_log2=13))
    a, ra = T.train([cloud], steps=10, seed=8, kernel_size=5, max_points=4_000)
    b, rb = T.train([cloud], steps=10, seed=8, kernel_size=5, max_points=4_000, conv_families="v6")
    assert [r["bpp"] for r in ra] == [r["bpp"] for r in rb]
    assert all(torch.equal(a[n], b[n]) for n in a)
    # patches below 150 K rows: the codec's rule is the mma.sync conv on every level, the same bits
    c, rc = T.train([cloud], steps=10, seed=8, kernel_size=5, max_points=4_000, conv_families="codec")
    assert all(torch.equal(a[n], c[n]) for n in a)


@pytest.mark.parametrize("k,sha", [(5, "3915714d027f28f29fe5dc720bc946d8540edb3b2a083cbfa51e7a9d0910a345"),
                                   (3, "19ecba2319073ae45a04efe5c70c65f3b9d69abe3f2bcf23634a430eb93a90af")])
def test_default_training_reproduces_the_recorded_checkpoint(env, k, sha):
    """the default determinism run (30 steps, seed 8, 4 000-point patches of a 16 000-point cloud) writes the checkpoint bytes
    recorded when minibatch training was introduced: torch.save of its state_dict to a byte buffer"""
    import hashlib
    import io
    from gauspcc_b200.synth import hac_like_cloud
    T = env["T"]
    cloud = torch.tensor(hac_like_cloud(16_000, seed=41, extent_log2=13))
    sd, _ = T.train([cloud], steps=30, seed=8, kernel_size=k, max_points=4_000)
    buf = io.BytesIO()
    torch.save(sd, buf)
    assert hashlib.sha256(buf.getvalue()).hexdigest() == sha


def test_cli_train_codec_families_then_compress_and_decompress(env, tmp_path):
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
                     "--is_data_pre_quantized", "--max_points", "2000", "--batch_size", "4", "--conv_families", "codec",
                     "--resultdir", res]) == 0
    validate_state_dict(torch.load(ck), 32, 3)
    enc, dec = str(tmp_path / "enc"), str(tmp_path / "dec")
    assert cli.main(["compress", "--input_glob", str(src), "--output_folder", enc, "--ckpt", ck, "--posQ", "1",
                     "--is_data_pre_quantized", "--resultdir", res]) == 0
    assert cli.main(["decompress", "--input_glob", enc, "--output_folder", dec, "--ckpt", ck, "--is_data_pre_quantized",
                     "--resultdir", res]) == 0
    for s, c in enumerate(clouds):
        got = cli.read_points(os.path.join(dec, f"s{s}.ply.bin.ply")).astype(np.int32)
        assert np.array_equal(np.unique(got, axis=0), np.unique(c, axis=0))
