"""BASELINE config[4] on one GPU: the per-scene loop (compress_point_cloud / decompress_point_cloud, one file after another) against
the batch API (compress_point_clouds / decompress_point_clouds, one union octree), in the same process, alternating.

    python tools/batch_union.py [--scenes 32] [--reps 3] [--gpu-coder-chunk N] [--out profiles/r03_batch_union.json]

Scene sizes are log-uniform in [100 K, 600 K] anchors with the seeds of tools/batch_scenes.py.  Every repetition checks that both
paths write identical bytes and that the batch decode equals the per-file decode (and the input, as a set).  Prints one JSON line:
end-to-end Mpoints/s, encode / decode wall time and launches per batch for both paths, with the GPU's name and power limit.

--gpu-coder-chunk N (> 0): both paths write container version 2 with chunks of N symbols (the per-scene version-2 loop against the
version-2 batch, same checks), and the version-1 batch runs beside them in the same alternation as "batch_v1" (its own files, so
its bytes are checked against nothing; its decode is checked against the version-2 loop's rows).
"""
import argparse, json, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gauspcc_b200 import pcc_utils
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import save_synthetic_checkpoint


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=32)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gpu-coder-chunk", type=int, default=0)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(0)
    sizes = np.exp(rng.uniform(np.log(100e3), np.log(600e3), a.scenes)).astype(np.int64)
    tmp = tempfile.mkdtemp(prefix="gpcgc_union_")
    ckpt = save_synthetic_checkpoint(os.path.join(tmp, "GausPcgc", "best_model_ue_4stage_conv.pt"))
    clouds = [torch.tensor(hac_like_cloud(int(n), seed=i), dtype=torch.float32, device=dev) for i, n in enumerate(sizes)]
    n_pts = int(sizes.sum())
    codec = pcc_utils._codec(ckpt, 32, 5)
    bc = pcc_utils._batch(codec)
    lp = [os.path.join(tmp, "loop", f"{i}.bin") for i in range(a.scenes)]
    bp = [os.path.join(tmp, "batch", f"{i}.bin") for i in range(a.scenes)]
    b1p = [os.path.join(tmp, "batch_v1", f"{i}.bin") for i in range(a.scenes)]
    chunk = a.gpu_coder_chunk

    def run_loop():
        l0 = int(codec.lib.gpc_launch_count())
        torch.cuda.synchronize(dev); t0 = time.perf_counter()
        for x, p in zip(clouds, lp):
            pcc_utils.compress_point_cloud(x, ckpt, p, gpu_coder_chunk=chunk)
        torch.cuda.synchronize(dev); t1 = time.perf_counter()
        l1 = int(codec.lib.gpc_launch_count())
        dec = [pcc_utils.decompress_point_cloud(p, ckpt)["point_cloud"] for p in lp]
        torch.cuda.synchronize(dev); t2 = time.perf_counter()
        return t1 - t0, t2 - t1, l1 - l0, int(codec.lib.gpc_launch_count()) - l1, dec

    dec_stats = {}                                                           # per batch run: BatchCodec.last_stats of its decode

    def run_batch(paths=bp, ck=chunk, name="batch"):
        l0 = int(codec.lib.gpc_launch_count())
        torch.cuda.synchronize(dev); t0 = time.perf_counter()
        pcc_utils.compress_point_clouds(clouds, ckpt, paths, gpu_coder_chunk=ck)
        torch.cuda.synchronize(dev); t1 = time.perf_counter()
        l1 = int(codec.lib.gpc_launch_count())
        dec = [d["point_cloud"] for d in pcc_utils.decompress_point_clouds(paths, ckpt)]
        torch.cuda.synchronize(dev); t2 = time.perf_counter()
        dec_stats[name] = {k: bc.last_stats.get(k) for k in ("unions", "stage_round_trips")}
        return t1 - t0, t2 - t1, l1 - l0, int(codec.lib.gpc_launch_count()) - l1, dec

    runs = [("loop", run_loop), ("batch", run_batch)]
    if chunk:
        runs.append(("batch_v1", lambda: run_batch(b1p, 0, "batch_v1")))
    for _, fn in runs:                                                        # warm-up: modules, allocator, pinned buffers
        fn()
    res = {name: [] for name, _ in runs}
    for rep in range(a.reps):
        for name, fn in runs:
            enc, dec, le, ld, rows = fn()
            res[name].append((enc, dec, le, ld))
            if name == "loop":
                loop_rows = rows
            else:
                for i in range(a.scenes):
                    if name == "batch":
                        with open(lp[i], "rb") as f1, open(bp[i], "rb") as f2:
                            assert f1.read() == f2.read(), f"scene {i}: batch bytes differ from the single call's"
                    assert torch.equal(rows[i], loop_rows[i]), f"scene {i}: {name} decode differs from the single decode"
                    if rep == 0:
                        got = np.unique(rows[i].cpu().numpy().astype(np.int64), axis=0)
                        assert np.array_equal(got, np.unique(clouds[i].cpu().numpy().astype(np.int64), axis=0)), f"scene {i}: not lossless"

    def summ(v):
        enc = float(np.median([r[0] for r in v])); dec = float(np.median([r[1] for r in v]))
        return {"enc_s": round(enc, 4), "dec_s": round(dec, 4), "e2e_mpts_s": round(n_pts / (enc + dec) / 1e6, 3),
                "enc_s_all": [round(r[0], 4) for r in v], "dec_s_all": [round(r[1], 4) for r in v],
                "launches_enc": v[-1][2], "launches_dec": v[-1][3]}

    out = {"config": f"{a.scenes} synthetic scenes, sizes log-uniform 100K-600K (seeds of tools/batch_scenes.py), 1 GPU",
           "gpu": gpu_info(), "points": n_pts, "reps": a.reps, "bytes_identical": True, "decode_identical": True, "lossless": True,
           "unions_dec": dec_stats["batch"]["unions"]}
    if chunk:
        out["gpu_coder_chunk"] = chunk
        out["decode_stats"] = dec_stats
    for name, _ in runs:
        out[name] = summ(res[name])
    out["speedup_e2e"] = round(out["batch"]["e2e_mpts_s"] / out["loop"]["e2e_mpts_s"], 3)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
