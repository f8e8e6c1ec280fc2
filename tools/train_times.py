"""Training on one GPU (gauspcc_b200/train.py): CUDA-event medians of forward / backward / Adam step per patch size, the weight and
input gradient of one conv against the forward conv on the same level, and the ideal and coded bits per point of held-out
hac_like_cloud patches before and after N steps from the synthetic init.  The card's name and power limit go beside the numbers.

    python tools/train_times.py [--sizes 20000,60000,150000] [--reps 10] [--steps 300] [--out FILE]"""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gauspcc_b200 import pcc_utils
from gauspcc_b200 import train as T
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import CONV_KEYS, make_synthetic_state_dict

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="20000,60000,150000")
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--steps", type=int, default=300)
ap.add_argument("--patch", type=int, default=20000, help="patch size of the training run")
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("train_times.py measures on the GPU; no CUDA device")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
out = {"card": card, "torch": torch.__version__, "reps": a.reps, "sizes": {}}


def ev():
    return torch.cuda.Event(enable_timing=True)


def cloud(n, seed):
    # extent 2^16 as the HAC scenes: a patch of n points keeps the density of a full scene
    return torch.tensor(hac_like_cloud(n, seed=seed, extent_log2=16), device=dev)


# ---- forward / backward / step per patch size
for n in [int(s) for s in a.sizes.split(",")]:
    net = T.GausPcgcNet(5, seed=5).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=5e-4)
    xyz = cloud(n, 100 + n)
    fw, bw, st = [], [], []
    for r in range(a.reps + 2):
        e = [ev() for _ in range(4)]
        torch.cuda.synchronize()
        e[0].record()
        o = net(xyz)
        e[1].record()
        opt.zero_grad(set_to_none=True)
        o["bpp"].backward()
        e[2].record()
        opt.step()
        e[3].record()
        torch.cuda.synchronize()
        if r >= 2:
            fw.append(e[0].elapsed_time(e[1])); bw.append(e[1].elapsed_time(e[2])); st.append(e[2].elapsed_time(e[3]))
    # one conv on the finest level: forward, input gradient (pack of the mirrored weights + forward kernel), weight gradient
    lv = net.geometry(xyz)[-1]
    km = lv.kmap
    W125 = net.state_dict()[CONV_KEYS[7]].contiguous()
    Wa = T.pack_frag(W125)
    x = torch.randn((lv.n, 32), device=dev)
    dy = torch.randn((lv.n, 32), device=dev)
    conv = {}
    for name, fn in (("forward", lambda: T.conv_v6(x, Wa, km)), ("dgrad", lambda: T.conv_dgrad(dy, W125, km)),
                     ("wgrad", lambda: T.conv_wgrad(x, dy, km))):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(5):
            e0, e1 = ev(), ev()
            e0.record()
            for _ in range(20):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / 20 * 1e3)
        conv[name + "_us"] = round(float(np.median(ts)), 1)
    out["sizes"][str(n)] = {"points": n, "levels": o["levels"], "bpp": round(float(o["bpp"].detach()), 4),
                            "forward_ms": round(float(np.median(fw)), 2), "backward_ms": round(float(np.median(bw)), 2),
                            "adam_ms": round(float(np.median(st)), 3),
                            "step_ms": round(float(np.median(np.array(fw) + np.array(bw) + np.array(st))), 2),
                            "finest_level": {"rows": lv.n, "true_pairs": km.n_real, "tile_rows": km.tile_rows, "variant": km.v6_variant,
                                             **conv}}
    print(json.dumps({n: out["sizes"][str(n)]}), flush=True)

# ---- bpp on held-out patches before and after training from the synthetic init
tmp = tempfile.mkdtemp(prefix="gpcgc_train_")
train_clouds = [cloud(150_000, s) for s in (1, 2, 3, 4)]
held_scene = cloud(150_000, 90)
held = [held_scene[i] for i in T.partition(held_scene, a.patch)][:4]
t0 = time.time()
sd, rows = T.train(train_clouds, os.path.join(tmp, "trained.pth"), steps=a.steps, seed=0, kernel_size=5, max_points=a.patch)
train_s = time.time() - t0
torch.save(make_synthetic_state_dict(5), os.path.join(tmp, "init.pth"))
evals = {}
for name, state in (("init", make_synthetic_state_dict(5)), ("trained", sd)):
    net = T.GausPcgcNet(5, state_dict=state).to(dev)
    ideal, coded, pts = 0.0, 0, 0
    for i, xyz in enumerate(held):
        with torch.no_grad():
            ideal += float(net(xyz)["bits"])
        r = pcc_utils.compress_point_cloud(xyz, os.path.join(tmp, name + ".pth"), os.path.join(tmp, f"{name}{i}.bin"), kernel_size=5)
        dec = pcc_utils.decompress_point_cloud(r["output_path"], os.path.join(tmp, name + ".pth"), kernel_size=5)["point_cloud"]
        assert torch.equal(torch.unique(dec.to(torch.int32), dim=0), torch.unique(xyz, dim=0)), "round trip is not lossless"
        coded += r["file_size_bits"]
        pts += xyz.shape[0]
    evals[name] = {"ideal_bpp": round(ideal / pts, 4), "file_bpp": round(coded / pts, 4)}
out["training"] = {"train_scenes": "4 x hac_like_cloud(150000, seeds 1-4, extent 2^16)", "patch_points": a.patch, "steps": a.steps,
                   "lr": 5e-4, "seconds": round(train_s, 1), "ms_per_step": round(train_s / a.steps * 1e3, 1),
                   "bpp_first_20": round(float(np.mean([r["bpp"] for r in rows[:20]])), 4),
                   "bpp_last_20": round(float(np.mean([r["bpp"] for r in rows[-20:]])), 4),
                   "held_out": f"first 4 kd-tree patches (<= {a.patch} points) of hac_like_cloud(150000, seed 90, extent 2^16)", **evals}
print(json.dumps({"training": out["training"]}), flush=True)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f)
print(json.dumps(out))
