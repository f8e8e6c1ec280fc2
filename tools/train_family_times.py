"""Training on the codec's conv families (GausPcgcNet.conv_families, gauspcc_b200/train.py) against the mma.sync conv everywhere, on
one GPU: one conv's forward, input gradient and weight gradient on sparse and dense levels of 150 K to 1.2 M rows (the shapes of
tools/train_batch_times.py), the step time of union batches, and the held-out file bpp after the same wall-clock budget (the
protocol of tools/train_batch_times.py at B = 8).  "v6" and "codec" alternate in one process.  The card's name and power limit go
beside the numbers.

    python tools/train_family_times.py [--levels 150000,600000,1200000] [--steps 150000x4,...] [--reps 5] [--budget 20]
                                       [--batch 8] [--out FILE]
(an empty --levels or --steps skips that part)"""
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
ap.add_argument("--levels", default="150000,600000,1200000")
ap.add_argument("--steps", default="150000x4,150000x8,150000x16,20000x16", help="patch points x batch size")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--budget", type=float, default=20.0, help="seconds of training per family in the rate comparison")
ap.add_argument("--patch", type=int, default=20000, help="patch size of the rate comparison")
ap.add_argument("--batch", type=int, default=8, help="batch size of the rate comparison")
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("train_family_times.py measures on the GPU; no CUDA device")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
out = {"card": card, "torch": torch.__version__, "reps": a.reps, "convs": [], "steps": {}, "rate": {}}
FAMS = ("v6", "codec")


def ev():
    return torch.cuda.Event(enable_timing=True)


def cloud(n, seed):
    return torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=16), device=dev)


# ---- one conv: forward, dgrad (the mirrored-weight forward), wgrad; v6 and the codec's family alternate rep by rep
geo = GausPcgcCodec(T._Geometry(5), dev)
W125 = make_synthetic_state_dict(5)[CONV_KEYS[7]].to(dev).contiguous()


def sparse_level(n):
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
    side = int(round((3 * n) ** (1 / 3))) + 1
    g = torch.Generator(device=dev).manual_seed(n)
    idx = torch.randperm(side ** 3, generator=g, device=dev)[:n]
    xyz = torch.stack([idx % side, (idx // side) % side, idx // (side * side)], 1).to(torch.int32)
    keys, _ = geo.pack_keys(xyz)
    return torch.unique(keys)


def timed(fns, reps, inner=10):
    """median microseconds of each fn over reps windows of `inner` calls, the fns taking turns window by window"""
    for fn in fns:
        for _ in range(3):
            fn()
    ts = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            e0, e1 = ev(), ev()
            e0.record()
            for _ in range(inner):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ts[j].append(e0.elapsed_time(e1) / inner * 1e3)
    return [round(float(np.median(t)), 1) for t in ts]


for kind, make in (("sparse", sparse_level), ("dense", dense_level)):
    for n in [int(s) for s in a.levels.split(",") if s]:
        keys = make(n)
        rows = int(keys.shape[0])
        maps = {"v6": geo.build_kmap(keys, family="v6"), "codec": geo.build_kmap(keys)}
        pack = T.WeightPack(W125, T.WGRAD_BALANCED_MIN_ROWS)
        pack.mirror(), pack.um(), pack.mirror_um()
        x = torch.randn((rows, 32), device=dev)
        dy = torch.randn((rows, 32), device=dev)
        fns = []
        for f in FAMS:
            km = maps[f]
            bal = T.kmap_family(km) == "v6" and rows >= T.WGRAD_BALANCED_MIN_ROWS
            fns += [lambda km=km: pack.conv(x, km), lambda km=km: pack.conv(dy, km, mirrored=True),
                    lambda km=km, bal=bal: T.conv_wgrad(x, dy, km, balanced=bal)]
        us = timed(fns, a.reps)
        for j, f in enumerate(FAMS):
            km = maps[f]
            row = {"level": kind, "rows": rows, "pairs_per_row": round(km.n_real / rows, 2), "families": f,
                   "kernel": T.kmap_family(km), "forward_us": us[3 * j], "dgrad_us": us[3 * j + 1], "wgrad_us": us[3 * j + 2]}
            row["total_us"] = round(row["forward_us"] + row["dgrad_us"] + row["wgrad_us"], 1)
            out["convs"].append(row)
            print(json.dumps(row), flush=True)
        del keys, maps, x, dy, fns
        torch.cuda.empty_cache()


# ---- step time per (patch size, batch size): the same B patches, v6 and codec alternating step by step
def step_fn(net, opt, batch):
    def run():
        opt.zero_grad(set_to_none=True)
        o = net.forward_batch(batch)
        o["bpp"].backward()
        opt.step()
        return o
    return run


for spec in [s for s in a.steps.split(",") if s]:
    n, B = (int(v) for v in spec.split("x"))
    batch = [cloud(n, 1000 + n + s) for s in range(B)]
    runs, fams = {}, {}
    for f in FAMS:
        net = T.GausPcgcNet(5, seed=5, conv_families=f).to(dev)
        runs[f] = step_fn(net, torch.optim.Adam(net.parameters(), lr=5e-4), batch)
    ts = {f: [] for f in FAMS}
    for r in range(a.reps + 2):
        for f in FAMS:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = runs[f]()
            torch.cuda.synchronize()
            if r >= 2:
                ts[f].append(time.perf_counter() - t0)
            fams[f] = o["families"]
    for f in FAMS:
        ms = float(np.median(ts[f])) * 1e3
        row = {"patch_points": n, "batch": B, "families": f, "step_ms": round(ms, 1), "patches_per_s": round(B / ms * 1e3, 1),
               "kernel_maps": fams[f], "unions": o["unions"]}
        out["steps"][f"{n}x{B}_{f}"] = row
        print(json.dumps(row), flush=True)
    del batch, runs
    torch.cuda.empty_cache()

# ---- held-out file bpp after the same wall-clock budget, v6 and codec
tmp = tempfile.mkdtemp(prefix="gpcgc_train_families_")
train_clouds = [cloud(150_000, s) for s in (1, 2, 3, 4)]
held_scene = cloud(150_000, 90)
held = [held_scene[i] for i in T.partition(held_scene, a.patch)][:4]
torch.save(make_synthetic_state_dict(5), os.path.join(tmp, "init.pth"))
for f in FAMS:
    _, probe = T.train(train_clouds, steps=10, seed=0, kernel_size=5, max_points=a.patch, batch_size=a.batch, conv_families=f)
    per_step = (probe[-1]["time"] - probe[1]["time"]) / 8
    steps = max(10, int(a.budget / per_step))
    ck = os.path.join(tmp, f"{f}.pth")
    t0 = time.time()
    sd, rows = T.train(train_clouds, ck, steps=steps, seed=0, kernel_size=5, max_points=a.patch, batch_size=a.batch, conv_families=f)
    secs = time.time() - t0
    coded, pts = 0, 0
    for i, xyz in enumerate(held):
        r = pcc_utils.compress_point_cloud(xyz, ck, os.path.join(tmp, f"{f}_{i}.bin"), kernel_size=5)
        dec = pcc_utils.decompress_point_cloud(r["output_path"], ck, kernel_size=5)["point_cloud"]
        assert torch.equal(torch.unique(dec.to(torch.int32), dim=0), torch.unique(xyz, dim=0)), "round trip is not lossless"
        coded += r["file_size_bits"]
        pts += xyz.shape[0]
    out["rate"][f] = {"families": f, "batch": a.batch, "steps": steps, "seconds": round(secs, 1), "patches_seen": steps * a.batch,
                      "bpp_last_10": round(float(np.mean([r["bpp"] for r in rows[-10:]])), 4),
                      "held_out_file_bpp": round(coded / pts, 4), "lossless": True}
    print(json.dumps(out["rate"][f]), flush=True)
init_coded, pts = 0, 0
for i, xyz in enumerate(held):
    r = pcc_utils.compress_point_cloud(xyz, os.path.join(tmp, "init.pth"), os.path.join(tmp, f"init_{i}.bin"), kernel_size=5)
    init_coded += r["file_size_bits"]
    pts += xyz.shape[0]
out["rate"]["init_file_bpp"] = round(init_coded / pts, 4)
out["rate"]["setup"] = {"train_scenes": "4 x hac_like_cloud(150000, seeds 1-4, extent 2^16)", "patch_points": a.patch,
                        "batch": a.batch, "budget_s": a.budget, "lr": 5e-4,
                        "held_out": f"first 4 kd-tree patches (<= {a.patch} points) of hac_like_cloud(150000, seed 90, extent 2^16)"}
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f)
print(json.dumps(out))
