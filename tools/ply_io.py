"""ASCII PLY I/O on the GPU (csrc/textio.cu, gauspcc_b200/plyio.py) against the Python it replaces, and the file tools end to end.

    python tools/ply_io.py [--sizes 1000000,3000000] [--reps 3] [--scenes 32] [--cli-reps 2] [--out profiles/r05_ply_io.json]

1. Write and read of PLY files of synth.hac_like_cloud(n, 0) rows, as integer voxel rows (`123.0`) and as CLI-scaled rows
   `(c * 16 - 131072) * 0.001` (17-digit reprs): the GPU writer (plyio.write_ply_ascii, file written) against the row-by-row
   Python writer, and the GPU reader (plyio.read_points_device) against cli.read_points.  One process, alternating, after a
   warm-up; bytes and rows are checked equal.  Seconds per call, median of --reps.
2. `python -m gauspcc_b200.cli compress / decompress` over a folder of --scenes ASCII PLY files (log-uniform 100 K - 600 K points,
   the seeds of tools/batch_scenes.py, CLI-scaled rows) with --batch 1 and --batch <scenes>, alternating; wall time of the whole
   folder per run (files read, coded, written), identical .bin / .ply bytes checked.
Prints one JSON line with the GPU's name and power limit.
"""
import argparse, filecmp, json, os, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gauspcc_b200 import cli, plyio
from gauspcc_b200.synth import hac_like_cloud
from gauspcc_b200.weights import save_synthetic_checkpoint


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def save_ply_ascii_geo(coords, path):
    """the Python writer decompress_point_cloud used before (kit/io.py:36-49)"""
    coords = coords.astype(np.float32)
    with open(path, 'w') as f:
        f.write('ply\nformat ascii 1.0\n')
        f.write(f'element vertex {coords.shape[0]}\n')
        f.write('property float x\nproperty float y\nproperty float z\nend_header\n')
        for p in coords:
            f.write(f'{p[0]} {p[1]} {p[2]}\n')


def scaled(c):
    return ((c.astype(np.int64) * 16 - 131072) * 0.001).astype(np.float32)


def timed(fn, dev):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize(dev)
    return time.perf_counter() - t0, r


def io_rows(n, kind, reps, tmp, dev):
    c = hac_like_cloud(n, seed=0)
    pts = c.astype(np.float32) if kind == "int" else scaled(c)
    pts_d = torch.from_numpy(pts).to(dev)
    hp, gp = os.path.join(tmp, "host.ply"), os.path.join(tmp, "gpu.ply")
    plyio.write_ply_ascii(pts_d, gp)                                        # warm-up
    plyio.read_points_device(gp, dev)
    t = {k: [] for k in ("write_host", "write_gpu", "read_host", "read_gpu")}
    for _ in range(reps):
        t["write_host"].append(timed(lambda: save_ply_ascii_geo(pts, hp), dev)[0])
        t["write_gpu"].append(timed(lambda: plyio.write_ply_ascii(pts_d, gp), dev)[0])
        dt, ref = timed(lambda: cli.read_points(hp), dev)
        t["read_host"].append(dt)
        dt, got = timed(lambda: plyio.read_points_device(gp, dev), dev)
        t["read_gpu"].append(dt)
        assert filecmp.cmp(hp, gp, shallow=False), "GPU PLY bytes differ from the Python writer's"
        assert np.array_equal(got.cpu().numpy(), ref), "GPU rows differ from cli.read_points"
    med = {k: float(np.median(v)) for k, v in t.items()}
    return {"rows": n, "kind": kind, "bytes": os.path.getsize(gp), **{k + "_s": v for k, v in med.items()},
            "write_speedup": med["write_host"] / med["write_gpu"], "read_speedup": med["read_host"] / med["read_gpu"]}


def cli_folder(n_scenes, reps, tmp, dev):
    rng = np.random.default_rng(0)
    sizes = np.exp(rng.uniform(np.log(100e3), np.log(600e3), n_scenes)).astype(np.int64)
    src = os.path.join(tmp, "scenes")
    os.makedirs(src)
    for i, n in enumerate(sizes):
        plyio.write_ply_ascii(torch.from_numpy(scaled(hac_like_cloud(int(n), seed=i))).to(dev), os.path.join(src, f"{i:03d}.ply"))
    ckpt = save_synthetic_checkpoint(os.path.join(tmp, "GausPcgc", "best_model_ue_4stage_conv.pt"))
    common = ["--ckpt", ckpt, "--kernel_size", "5"]
    res = {1: {"compress": [], "decompress": []}, n_scenes: {"compress": [], "decompress": []}}

    def run(batch, rep):
        enc, dec = os.path.join(tmp, f"enc{batch}_{rep}"), os.path.join(tmp, f"dec{batch}_{rep}")
        b = ["--batch", str(batch)]
        t, _ = timed(lambda: cli.main(["compress", "--input_glob", src, "--output_folder", enc] + common + b), dev)
        res[batch]["compress"].append(t)
        t, _ = timed(lambda: cli.main(["decompress", "--input_glob", enc, "--output_folder", dec] + common + b), dev)
        res[batch]["decompress"].append(t)
        return enc, dec

    run(1, "warm"); run(n_scenes, "warm")
    for k in res:
        for v in res[k].values():
            v.clear()
    for rep in range(reps):
        e1, d1 = run(1, rep)
        en, dn = run(n_scenes, rep)
        for a, b in ((e1, en), (d1, dn)):
            names = sorted(os.listdir(a))
            assert names == sorted(os.listdir(b)) and all(filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False)
                                                          for f in names), f"{a} != {b}"
        for d in (e1, d1, en, dn):
            shutil.rmtree(d)
    n_pts = int(sizes.sum())
    out = {"scenes": n_scenes, "points": n_pts, "text_bytes": sum(os.path.getsize(os.path.join(src, f)) for f in os.listdir(src))}
    for batch, r in res.items():
        for step, ts in r.items():
            m = float(np.median(ts))
            out[f"batch{batch}_{step}_s"] = m
            out[f"batch{batch}_{step}_files_per_s"] = n_scenes / m
            out[f"batch{batch}_{step}_mpts_per_s"] = n_pts / m / 1e6
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,3000000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scenes", type=int, default=32)
    ap.add_argument("--cli-reps", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    tmp = tempfile.mkdtemp(prefix="gpcgc_plyio_")
    try:
        io = [io_rows(int(n), kind, a.reps, tmp, dev) for n in a.sizes.split(",") for kind in ("int", "cli")]
        folder = cli_folder(a.scenes, a.cli_reps, tmp, dev) if a.scenes > 0 else None
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    res = {"gpu": gpu_info(), "io": io, "cli_folder": folder}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
