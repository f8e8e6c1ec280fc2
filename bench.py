#!/usr/bin/env python
"""bench.py -- GausPcgc encode+decode throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--points P] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one scene: device-resident voxel anchors -> pyramid ->
kernel maps -> 18 sparse convs + 4 heads per level -> CDF rows (encode), then the same on the decode
side driven by the decoded symbols.  Workload at N=1: BASELINE config[1], 1M synthetic anchors with
the sparse-global/dense-local HAC++ distribution.  At N>1 the path shards by scene: every rank codes
its own copy of THE SAME scene (seed 0 on every rank: the max over ranks then measures the box, not the
luck of a rank's scene), no data-path collective, one small all_gather of per-scene results
("scaling": "weak").

value    = Mpoints/s, CUDA-event time of K steps (encode + decode device stages; CDFs stay in HBM;
           the decode side is fed the true symbols from HBM instead of the host range decoder, the
           device work is identical -- tests/test_gpu_parity.py proves the real decode is lossless).
           Nothing else is recorded inside the timed region.
e2e      = same metric through the public API (pcc_utils.compress_point_cloud /
           decompress_point_cloud) with HOST input, host range coder, file write/read and the result
           read back to the host, wall clock.  This is the number to hold against the reference arm.
roofline = the dominant kernel family of the step (the sparse conv of the big dense levels), from a SEPARATE
           profiled step after the timed region: algorithmic bytes (SURVEY.md 8d) / CUDA-event time of exactly
           those launches; `traffic` = measured dram bytes per launch of the same kernel from the committed
           ncu capture (profiles/r02_conv_um_dram.json).  `per_stage` lists every stage of the step the same way.
--impl reference: the reference algorithm on the host cores (CPU oracle port; the reference's own
           dependencies torchsparse/torchac are not installable offline) on the SAME workload when the
           run fits the time budget, else on the largest sample that does (config.sample_points says which).
--dump-outputs DIR: after the timed steps, what the last of them computed, as DIR/<name>.npy (float32, or float64 where
           float32 cannot hold an integer exactly): base_xyz, base_occ, occupancy (every coded level, coarse -> fine),
           cdf_bounds_stage<i> (c_low, c_high of the range coder's interval per row of stage i, coarse -> fine) and points
           (the decoded cloud).  The scene and weights are seeded, so two builds run with the same arguments can be compared
           array for array.  Above DUMP_BYTES every array keeps the same fraction of its rows, picked with a fixed seed.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mpoints/s GausPcgc encode+decode (device-timed)"
UNIT = "Mpoints/s"
DTYPE = "bf16x3-split/f32-acc"        # every product is hi.hi + hi.lo + lo.hi of bf16 halves (16 mantissa bits), fp32 accumulation
REF_BUDGET_S = 330.0                  # the reference arm's whole run (warm-up + steps) stays within a few minutes
CPU_BASELINE_S = 15.0                 # the cpu_baseline leg of the repo arm: one bounded sample
DUMP_BYTES = 60_000_000               # --dump-outputs: array bytes at most (with the .npy headers, under 64 MB)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def _workload(points: int) -> str:
    return f"GausPcgc encode/decode, {points} synthetic anchors (sparse-global/dense-local HAC++ distribution)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def _nvml(self):
        """NVML handle for fast sampling (a query is ~1 ms; an nvidia-smi process is ~0.4 s, one sample per timed region)"""
        try:
            import pynvml
            pynvml.nvmlInit()
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            return None, None

    def run(self):
        nv, h = self._nvml()
        while not self.stop_flag.is_set():
            try:
                if nv is not None:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    act = lambda bit: "Active" if r & bit else "Not Active"
                    self.samples.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                                         act(0x8), act(0x40), act(0x20), act(0x4)])     # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.05 if nv is not None else 0.2)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) >= 6 and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------- the reference algorithm on the host cores
def _host_threads() -> int:
    """All the cores this process may use.  torchrun exports OMP_NUM_THREADS=1 to its ranks; the oracle's OpenMP runtime is told the
    real number explicitly (libgomp is the runtime the oracle's shared library links)."""
    n = len(os.sched_getaffinity(0))
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except OSError:
        pass
    return n


def _oracle_roundtrip(xyz, w):
    from oracle import oracle as O
    t0 = time.perf_counter()
    blob = O.encode(xyz, w)
    dec = O.decode(blob, w)
    dt = time.perf_counter() - t0
    assert dec.shape[0] == xyz.shape[0], "oracle round trip lost points"
    return dt


def cpu_reference(points: int, steps: int, warmup: int, budget_s: float):
    """The CPU oracle port (reference algorithm, all host cores) on `points` anchors of the bench scene if warm-up + steps fit the
    budget, else on the largest sample that does.  -> (Mpoints/s, s per step, cores, sample points)"""
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import make_synthetic_state_dict, state_dict_to_numpy
    cores = _host_threads()
    w = state_dict_to_numpy(make_synthetic_state_dict())
    cal_n = min(points, 20_000)
    cal = _oracle_roundtrip(hac_like_cloud(cal_n, 0), w)                 # calibration: seconds per point on this box (also warms the library)
    per_point = cal / cal_n
    fit = int(budget_s / max(steps + warmup, 1) / per_point * 0.9)        # the oracle is a little super-linear: keep some slack
    sample = points if fit >= points else max(cal_n, fit // 10_000 * 10_000)
    xyz = hac_like_cloud(sample, 0)
    times = []
    for it in range(warmup + steps):
        dt = _oracle_roundtrip(xyz, w)
        if it >= warmup:
            times.append(dt)
    sec = float(np.mean(times))
    return sample / sec / 1e6, sec, cores, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                                           # one CPU arm per box: the host cores are shared by the ranks
    val, sec, cores, sample = cpu_reference(args.points, args.steps, args.warmup, REF_BUDGET_S)
    note = (f"{sample} anchors of the bench scene per step (encode+decode, lossless checked)"
            + ("" if sample == args.points else f": the full {args.points}-anchor config does not fit {REF_BUDGET_S:.0f} s for "
               f"{args.warmup}+{args.steps} steps on {cores} cores"))
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 5), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload(args.points) + ", reference algorithm (CPU port) on the box's host cores", "sample_points": sample,
                   "same_config": sample == args.points,
                   "box_level": "one scene at a time on all host cores; the value is the whole box's CPU throughput whatever --gpus says"},
        "cpu_baseline": {"value": round(val, 5), "unit": UNIT, "cores": cores, "kind": "port", "sample": note},
        "e2e": {"value": round(val, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- the repo arm
def _exact_float(a: np.ndarray) -> np.ndarray:
    if a.dtype.kind == "f":
        return a.astype(np.float32 if a.dtype.itemsize <= 4 else np.float64)
    return a.astype(np.float32 if a.size == 0 or int(np.abs(a.astype(np.int64)).max()) < (1 << 24) else np.float64)


def dump_outputs(path: str, out: dict):
    """Write what one step computed (step(keep=...)) as path/<name>.npy; see --dump-outputs in the module docstring."""
    import torch
    lohi = [t.cpu().numpy().view(np.uint32) for t in out["lohi"]]      # [4 * level + stage], levels coarse -> fine
    arrays = {"base_xyz": out["base_xyz"], "base_occ": out["base_occ"],
              "occupancy": torch.cat(out["occupancy"]).cpu().numpy() if out["occupancy"] else np.zeros(0, np.uint8)}
    for i in range(4):
        w = np.concatenate(lohi[i::4]) if lohi else np.zeros(0, np.uint32)
        arrays[f"cdf_bounds_stage{i}"] = np.stack([w & 0xFFFF, w >> 16], axis=1)
    arrays["points"] = out["points"].cpu().numpy()
    arrays = {k: _exact_float(np.asarray(v)) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.shape[0] * DUMP_BYTES // total
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference does not run it")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from gauspcc_b200.shard import pin_rank
    n_cpus = pin_rank(local, world)                                 # before torch / the codec size their thread pools

    import torch
    import torch.distributed as dist
    from gauspcc_b200 import pcc_utils, shard
    from gauspcc_b200.codec import DeviceWeights, GausPcgcCodec
    from gauspcc_b200.synth import hac_like_cloud
    from gauspcc_b200.weights import make_synthetic_state_dict, save_synthetic_checkpoint

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    sd = make_synthetic_state_dict()
    codec = GausPcgcCodec(DeviceWeights(sd, dev), dev)
    xyz = hac_like_cloud(args.points, seed=0)                        # the same scene on every rank (weak scaling by scene)
    x_dev = torch.tensor(xyz, dtype=torch.float32, device=dev)       # resident in HBM before the timed region
    from gauspcc_b200.pcc_utils import calculate_morton_order
    x_dev = x_dev[calculate_morton_order(x_dev)]                     # as HAC hands it over (gaussian_model.py:1108-1109)

    def step(keep=None):
        """one encode + decode; returns only scalars: a step must not keep the previous step's device buffers alive (the caching
        allocator would cudaMalloc a second and third working set inside the timed region: 149-203 ms per step instead of 135).
        keep (a dict, only on the last timed step) receives the arrays a caller of the path gets back, for --dump-outputs.  With
        --dump-outputs every step keeps its CDF words to the end, so the warm-up sizes the allocator's pool for the timed steps."""
        bx, bo, _, aux = codec.encode(x_dev, download=False, keep_lohi=bool(args.dump_outputs))
        n_enc = codec.launches
        occs = [lv.occ for lv in aux["levels"][1:]]
        out = codec.decode(bx, bo, [b""] * (4 * len(occs)), forced_occ=occs)
        if keep is not None:
            keep.update(base_xyz=bx, base_occ=bo, occupancy=occs, lohi=aux["lohi"], points=out)
        return int(out.shape[0]), n_enc + codec.launches, (int(len(aux["levels"]) - 1), int(sum(l.n for l in aux["levels"][1:])))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    codec.conv_profile = None
    for _ in range(args.warmup):
        n_out, _, _ = step()
    assert n_out == args.points
    barrier()
    sampler = ClockSampler(local)
    if not os.environ.get("BENCH_NO_SAMPLER"):
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    last = {} if args.dump_outputs and rank == 0 else None
    t_wall0 = time.perf_counter()
    e0.record(torch.cuda.current_stream(dev))
    for it in range(args.steps):
        n_out, nl, (n_levels, n_symbol_rows) = step(last if it == args.steps - 1 else None)
        launches += nl
    e1.record(torch.cuda.current_stream(dev))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.stop_flag.set()
    if sampler.is_alive():
        sampler.join()
    if last is not None:
        dump_outputs(args.dump_outputs, last)
        last = None
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # max over ranks
        res = shard.gather_results(torch.tensor([[args.points, int(ms * 1e3)]], dtype=torch.int64, device=dev), world,
                                   [[r] for r in range(world)])
        total_points = int(res[:, 0].sum().item())
    else:
        total_points = args.points
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = total_points / (ms_per_step / 1e3) / 1e6

    # ---- per-stage profile: two extra steps OUTSIDE the timed region, one CUDA-event pair per stage instance
    stages = {}
    if rank == 0 and not args.no_profile:
        n_prof = 2
        codec.conv_profile = []
        step()                                                       # creates the events of the pool
        codec.prewarm_profile_events(2 * len(codec.conv_profile) + 64)
        codec.conv_profile = []
        for _ in range(n_prof):
            codec._ev_next = 0
            pre = len(codec.conv_profile)
            step()
            torch.cuda.synchronize(dev)
            for p in codec.conv_profile[pre:]:
                st = stages.setdefault(p[5], {"ms": 0.0, "bytes": 0, "flops": 0, "launches": 0, "instances": 0})
                st["ms"] += p[0].elapsed_time(p[1]) / n_prof
                st["bytes"] += p[2] / n_prof
                st["flops"] += p[3] / n_prof
                st["launches"] += p[4] / n_prof
                st["instances"] += 1 / n_prof
        codec.conv_profile = None

    # ---- e2e through the public API, host buffers in, host result out (rank-local scene, wall clock)
    e2e = e2e_v2 = None
    if not args.no_e2e:
        tmp = tempfile.mkdtemp(prefix="gpcgc_bench_")
        ckpt = save_synthetic_checkpoint(os.path.join(tmp, "GausPcgc", "best_model_ue_4stage_conv.pt"))
        x_host = x_dev.cpu().pin_memory()
        binp = os.path.join(tmp, f"xyz_pcc_{rank}.bin")
        n_e2e = max(1, min(args.steps, 3))
        walls = []
        for it in range(1 + n_e2e):
            barrier()
            t0 = time.perf_counter()
            r = pcc_utils.compress_point_cloud(x_host, ckpt, binp)
            d2h_enc = codec_stats(pcc_utils)
            d = pcc_utils.decompress_point_cloud(binp, ckpt)
            dec_stats = codec_stats(pcc_utils)
            pts_host = d["point_cloud"].cpu()                        # the step's result read back to the host
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            if it > 0:
                walls.append(dt)
        rows = int(d2h_enc.get("rows", 0))
        tw = torch.tensor([float(np.mean(walls))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        e2e = {"value": round(total_points / float(tw.item()) / 1e6, 4), "unit": UNIT,
               "h2d_bytes_per_step": int(x_host.numel() * 4 + rows * 4),                       # input + decoded symbols
               "d2h_bytes_per_step": int(rows * 4 * 4 + rows * 2 * 28 + pts_host.numel() * 4),  # enc (c_low,c_high) words + dec CDF rows + result
               "enc_s": round(r["enc_time"], 4), "dec_s": round(d["dec_time"], 4), "bpp": round(r["bpp"], 3),
               "dec_host_ac_s": round(dec_stats.get("host_ac_s", 0.0), 4), "dec_gpu_wait_s": round(dec_stats.get("gpu_wait_s", 0.0), 4),
               "dec_gpu_s": round(dec_stats.get("gpu_ms", 0.0) / 1e3, 4), "dec_wavefront_levels": int(dec_stats.get("wave_levels", 0)),
               "ac_threads": codec_threads(pcc_utils), "cpus_per_rank": n_cpus}
        assert pts_host.shape[0] == args.points
        # the same round trip with the opt-in container version 2 (SURVEY 8f-3: occupancy streams coded on the GPU in chunks of 2048
        # symbols; no host range coder, only compressed bytes cross PCIe; NOT the reference bitstream -- reported beside e2e, never as it)
        walls2 = []
        for it in range(1 + n_e2e):
            barrier()
            t0 = time.perf_counter()
            r2 = pcc_utils.compress_point_cloud(x_host, ckpt, binp + ".v2", gpu_coder_chunk=2048)
            d2 = pcc_utils.decompress_point_cloud(binp + ".v2", ckpt)
            pts2 = d2["point_cloud"].cpu()
            torch.cuda.synchronize(dev)
            if it > 0:
                walls2.append(time.perf_counter() - t0)
        assert torch.equal(pts2, pts_host)
        tw2 = torch.tensor([float(np.mean(walls2))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tw2, op=dist.ReduceOp.MAX)
        e2e_v2 = {"value": round(total_points / float(tw2.item()) / 1e6, 4), "unit": UNIT,
                  "container": "version 2: GPU chunk coder, 2048 symbols per chunk (opt-in; not readable by the reference)",
                  "enc_s": round(r2["enc_time"], 4), "dec_s": round(d2["dec_time"], 4), "bpp": round(r2["bpp"], 3),
                  "h2d_bytes_per_step": int(x_host.numel() * 4 + r2["file_size_bits"] // 8),
                  "d2h_bytes_per_step": int(r2["file_size_bits"] // 8 + pts_host.numel() * 4)}

    if rank == 0:
        peaks, peak_kind = _peaks()
        line = {
            "metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": _workload(args.points) + ", 1 scene per B200", "points_per_gpu": args.points, "levels": n_levels,
                       "symbol_rows": n_symbol_rows, "same_scene_on_every_rank": True,
                       "l2": "working set (>= 128 MB feature arrays per level) exceeds the 126 MB L2; no explicit flush",
                       "parallelism": f"scene-sharded x{world}", "wall_ms_per_step": round(t_wall * 1e3 / args.steps, 2)},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
        }
        if stages:
            per_stage, tot_ms = [], sum(v["ms"] for v in stages.values())
            for name, v in sorted(stages.items(), key=lambda kv: -kv[1]["ms"]):
                gbs = v["bytes"] / (v["ms"] / 1e3) / 1e9 if v["ms"] > 0 else 0.0
                per_stage.append({"stage": name, "ms_per_step": round(v["ms"], 3), "share": round(v["ms"] / tot_ms, 4),
                                  "algorithmic_mb": round(v["bytes"] / 1e6, 1), "gbs": round(gbs, 1), "frac": round(gbs / peaks["hbm_gbs"], 4),
                                  "launches": int(round(v["launches"])) or int(round(v["instances"]))})
            dom_name = per_stage[0]["stage"]
            dom = stages[dom_name]
            achieved = dom["bytes"] / (dom["ms"] / 1e3) / 1e9
            traffic, traffic_src = None, None
            tpath = os.path.join(ROOT, "profiles", "r02_conv_um_dram.json")
            if dom_name == "conv_um" and os.path.exists(tpath):
                tj = json.load(open(tpath))
                traffic, traffic_src = int(tj["dram_bytes_per_launch_mean"]), "profiles/r02_conv_um_dram.json (ncu --set full, same kernel, same scene)"
            kernels = {"conv_um": "spconv_um_kernel<512, 64, ...> (tcgen05.mma + TMA gather4 / tile loads, big dense levels)",
                       "conv_sparse": "sp_centre_kernel + sp_straggler_kernel (sparse big levels)", "conv_v6": "spconv_fwd_v6 / v6d (mma.sync, coarse levels)"}
            line["roofline"] = {"kernel": kernels.get(dom_name, dom_name), "bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"],
                                "peak_kind": peak_kind + " (burst copy figure)", "unit": "GB/s", "frac": round(achieved / peaks["hbm_gbs"], 4),
                                "traffic": traffic, "traffic_source": traffic_src,
                                "algorithmic_bytes_per_launch": int(dom["bytes"] / max(dom["launches"], 1)),
                                "avg_launch_ms": round(dom["ms"] / max(dom["launches"], 1), 4), "launches_per_step": int(round(dom["launches"])),
                                "share_of_profiled_step": per_stage[0]["share"],
                                "tflops_effective_fp32": round(dom["flops"] / (dom["ms"] / 1e3) / 1e12, 2),
                                "note": "measured in two separate profiled steps (one CUDA-event pair per group of convs on a level) after the timed "
                                        "region, on ONE stream: the profile switches off the overlap of independent levels / kernel-map builds "
                                        "on side streams that the timed step uses, so per_stage sums to more than ms_per_step; the kernel is bound "
                                        "by its warp-specialised pipeline (hand-off latency between the roles), not by HBM: profiles/r02_conv_um.md"}
            line["per_stage"] = per_stage
        if e2e:
            line["e2e"] = e2e
            line["e2e_v2"] = e2e_v2
        if not args.no_cpu_baseline:
            val, sec, cores, sample = cpu_reference(args.points, 1, 0, CPU_BASELINE_S)
            line["cpu_baseline"] = {"value": round(val, 5), "unit": UNIT, "cores": cores, "kind": "port", "same_config": sample == args.points,
                                    "sample": f"{sample} anchors of the bench scene, encode+decode once ({sec:.1f} s) on {cores} host threads"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def codec_stats(pcc_utils_mod):
    for c in pcc_utils_mod._CODECS.values():
        return dict(c.last_stats)
    return {}


def codec_threads(pcc_utils_mod):
    for c in pcc_utils_mod._CODECS.values():
        return c.pool._max_workers
    return 0


if __name__ == "__main__":
    main()
