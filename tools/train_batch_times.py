"""Minibatch training on one GPU (gauspcc_b200/train.py): step time and patches/s per batch size and patch size, the two weight
gradient kernels against the forward conv from 1 K to 1.2 M rows (the crossover behind train.WGRAD_BALANCED_MIN_ROWS), and the
held-out file bpp after the same wall-clock budget at batch size 1 and 8.  The card's name and power limit go beside the numbers.

    python tools/train_batch_times.py [--sizes 20000,60000,150000] [--batches 1,2,4,8,16] [--reps 5] [--budget 20] [--out FILE]"""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gauspcc_b200 import pcc_utils
from gauspcc_b200 import train as T
from gauspcc_b200.codec import GausPcgcCodec
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import CONV_KEYS, make_synthetic_state_dict

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="20000,60000,150000")
ap.add_argument("--batches", default="1,2,4,8,16")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--levels", default="1000,10000,50000,150000,300000,600000,1200000")
ap.add_argument("--budget", type=float, default=20.0, help="seconds of training per batch size in the rate comparison")
ap.add_argument("--patch", type=int, default=20000, help="patch size of the rate comparison")
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("train_batch_times.py measures on the GPU; no CUDA device")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
out = {"card": card, "torch": torch.__version__, "reps": a.reps, "steps": {}, "wgrad": [], "rate": {}}


def ev():
    return torch.cuda.Event(enable_timing=True)


def cloud(n, seed):
    # extent 2^16 as the HAC scenes: a patch of n points keeps the density of a full scene
    return torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=16), device=dev)


# ---- step time per (patch size, batch size): B distinct patches of n points, forward_batch (B > 1) or forward (B = 1)
for n in [int(s) for s in a.sizes.split(",")]:
    pool = [cloud(n, 1000 + n + s) for s in range(max(int(b) for b in a.batches.split(",")))]
    for B in [int(b) for b in a.batches.split(",")]:
        net = T.GausPcgcNet(5, seed=5).to(dev)
        opt = torch.optim.Adam(net.parameters(), lr=5e-4)
        ts = []
        for r in range(a.reps + 2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            opt.zero_grad(set_to_none=True)
            o = net(pool[0]) if B == 1 else net.forward_batch(pool[:B])
            o["bpp"].backward()
            opt.step()
            torch.cuda.synchronize()
            if r >= 2:
                ts.append(time.perf_counter() - t0)
        ms = float(np.median(ts)) * 1e3
        row = {"patch_points": n, "batch": B, "step_ms": round(ms, 1), "patches_per_s": round(B / ms * 1e3, 1),
               "unions": o.get("unions", 0)}
        out["steps"][f"{n}x{B}"] = row
        print(json.dumps(row), flush=True)


# ---- one conv's forward, old and balanced weight gradient on levels from 1 K to 1.2 M rows
def conv_us(fn, reps=5, inner=10):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(inner):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / inner * 1e3)
    return round(float(np.median(ts)), 1)


geo = GausPcgcCodec(T._Geometry(5), dev)
W125 = make_synthetic_state_dict(5)[CONV_KEYS[7]].to(dev).contiguous()
Wa = T.pack_frag(W125)


def sparse_level(n):
    """a HAC-like finest level: n points of 150 K-point patches stacked along z (a union level), about one neighbour per row"""
    parts, left, s = [], n, 0
    while left > 0:
        p = cloud(min(left, 150_000), 500 + s)
        p[:, 2] += (s - 4) * (1 << 17)
        parts.append(p)
        left -= p.shape[0]
        s += 1
    keys, _ = geo.pack_keys(torch.cat(parts))
    return torch.unique(keys)


def dense_level(n):
    """a coarse level: n voxels drawn without repetition from a cube 3x their count (about 40 neighbours per row)"""
    side = int(round((3 * n) ** (1 / 3))) + 1
    g = torch.Generator(device=dev).manual_seed(n)
    idx = torch.randperm(side ** 3, generator=g, device=dev)[:n]
    xyz = torch.stack([idx % side, (idx // side) % side, idx // (side * side)], 1).to(torch.int32)
    keys, _ = geo.pack_keys(xyz)
    return torch.unique(keys)


for kind, make in (("sparse", sparse_level), ("dense", dense_level)):
    for n in [int(s) for s in a.levels.split(",")]:
        keys = make(n)
        rows = int(keys.shape[0])
        km = geo.build_kmap(keys, family="v6")
        x = torch.randn((rows, 32), device=dev)
        dy = torch.randn((rows, 32), device=dev)
        row = {"level": kind, "rows": rows, "pairs_per_row": round(km.n_real / rows, 2), "tile_rows": km.tile_rows,
               "forward_us": conv_us(lambda: T.conv_v6(x, Wa, km)),
               "wgrad_us": conv_us(lambda: T.conv_wgrad(x, dy, km)),
               "wgrad_balanced_us": conv_us(lambda: T.conv_wgrad(x, dy, km, balanced=True))}
        out["wgrad"].append(row)
        print(json.dumps(row), flush=True)
        del keys, km, x, dy
        torch.cuda.empty_cache()

# ---- held-out file bpp after the same wall-clock budget at B = 1 and B = 8
tmp = tempfile.mkdtemp(prefix="gpcgc_train_batch_")
train_clouds = [cloud(150_000, s) for s in (1, 2, 3, 4)]
held_scene = cloud(150_000, 90)
held = [held_scene[i] for i in T.partition(held_scene, a.patch)][:4]
torch.save(make_synthetic_state_dict(5), os.path.join(tmp, "init.pth"))
for B in (1, 8):
    # the steps that fit the budget, from a short timed run of the same configuration
    _, probe = T.train(train_clouds, steps=10, seed=0, kernel_size=5, max_points=a.patch, batch_size=B)
    per_step = (probe[-1]["time"] - probe[1]["time"]) / 8
    steps = max(10, int(a.budget / per_step))
    ck = os.path.join(tmp, f"b{B}.pth")
    t0 = time.time()
    sd, rows = T.train(train_clouds, ck, steps=steps, seed=0, kernel_size=5, max_points=a.patch, batch_size=B)
    secs = time.time() - t0
    coded, pts = 0, 0
    for i, xyz in enumerate(held):
        r = pcc_utils.compress_point_cloud(xyz, ck, os.path.join(tmp, f"b{B}_{i}.bin"), kernel_size=5)
        dec = pcc_utils.decompress_point_cloud(r["output_path"], ck, kernel_size=5)["point_cloud"]
        assert torch.equal(torch.unique(dec.to(torch.int32), dim=0), torch.unique(xyz, dim=0)), "round trip is not lossless"
        coded += r["file_size_bits"]
        pts += xyz.shape[0]
    out["rate"][str(B)] = {"batch": B, "steps": steps, "seconds": round(secs, 1), "patches_seen": steps * B,
                           "bpp_last_10": round(float(np.mean([r["bpp"] for r in rows[-10:]])), 4),
                           "held_out_file_bpp": round(coded / pts, 4), "lossless": True}
    print(json.dumps(out["rate"][str(B)]), flush=True)
init_coded, pts = 0, 0
for i, xyz in enumerate(held):
    r = pcc_utils.compress_point_cloud(xyz, os.path.join(tmp, "init.pth"), os.path.join(tmp, f"init_{i}.bin"), kernel_size=5)
    init_coded += r["file_size_bits"]
    pts += xyz.shape[0]
out["rate"]["init_file_bpp"] = round(init_coded / pts, 4)
out["rate"]["setup"] = {"train_scenes": "4 x hac_like_cloud(150000, seeds 1-4, extent 2^16)", "patch_points": a.patch,
                        "budget_s": a.budget, "lr": 5e-4,
                        "held_out": f"first 4 kd-tree patches (<= {a.patch} points) of hac_like_cloud(150000, seed 90, extent 2^16)"}
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f)
print(json.dumps(out))
