"""Device time of svnicp_map_evaluate (VoxelHashMap.Evaluate) at configs[1] size: a 64-beam scan (~143 k points) against a
saturated 1 m / 20-point local map built from synth.make_scan drives.

python scripts/map_evaluate_speed.py [--calls N] [--json OUT]

Cases: the full scan at M = 1, 8, 64 poses, and the down-sampled scan (uniform 0.5 m then 1.5 m, as synth.make_problem's
downsample) at M = 1, 64, 1000, each with and without the Gauss-Newton system.  Per call: CUDA events around the blocking call
(the map runs on its own stream and the call returns when its results are on the host, so this is the call's wall time: pose
upload, kernels, result copies).  Per kernel: torch.profiler in a separate pass (k_map_eval, the nearest-point pass, and
k_eval_fin).  Also prints queries (source points x poses) per second, the map's live voxels and points, and the card name and
power limit of the run.  Needs the GPU: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 0xC0FFEE
MAX_DIST = 3.0  # bench.WORKLOAD["max_dist"]


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=0, help="timed calls per case (default: 100 / 20 / 5 by size)")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import svn_icp_b200 as sv
    from svn_icp_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("map_evaluate_speed: no CUDA device (this measurement has no CPU fallback)")
    name, limit = card()
    print(f"card: {name}; power limit, max SM clock: {limit}", flush=True)
    world = synth.make_world(SEED)
    m = sv.VoxelHashMap(1.0, 100.0, 20)
    for k in range(12):  # the drive up to the scored scan, every scan inserted at its ground-truth pose
        pts, (R, t) = synth.make_scan(world, k, "64", SEED)
        m.AddPointCloud(pts.astype(np.float32), R, t)
    src, (Rg, tg) = synth.make_scan(world, 12, "64", SEED)
    src = src.astype(np.float32)
    down = synth.uniform_downsample(synth.uniform_downsample(src.astype(np.float64), 0.5), 1.5).astype(np.float32)
    rng = np.random.default_rng(1)
    R0, t0 = Rg @ synth.rot_from_rotvec(rng.normal(0, 0.002, 3)), tg + rng.normal(0, [0.05, 0.05, 0.02])
    poses = lambda M: np.concatenate([np.zeros((6, 1)), synth.init_particles(max(M - 1, 1), rng)], axis=1)[:, :M]  # noqa: E731
    res = dict(card=name, power_limit_and_max_clock=limit, map_voxels=m.Size(), map_points=m.PointCount(), n_full=len(src),
               n_down=len(down), max_dist=MAX_DIST, cases=[])
    print(f"map: {m.Size()} voxels, {m.PointCount()} points ({m.PointCount() / m.Size():.1f} per voxel); scan {len(src)} points, "
          f"down-sampled {len(down)}", flush=True)
    cases = [("full", src, 1), ("full", src, 8), ("full", src, 64), ("down", down, 1), ("down", down, 64), ("down", down, 1000)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = torch.cuda.current_stream()
    for label, cloud, M in cases:
        x = poses(M)
        work = len(cloud) * M
        for system in (True, False):
            n = args.calls or (100 if work < 2e6 else 20 if work < 2e7 else 5)
            for _ in range(2):
                m.Evaluate(cloud, R0, t0, x, MAX_DIST, want_system=system)
            ts = []
            for _ in range(n):
                ev0.record(st)
                m.Evaluate(cloud, R0, t0, x, MAX_DIST, want_system=system)
                ev1.record(st)
                ev1.synchronize()
                ts.append(ev0.elapsed_time(ev1))
            ts = np.array(ts)
            e = m.Evaluate(cloud, R0, t0, x[:, 0], MAX_DIST)
            row = dict(scan=label, n=len(cloud), M=M, system=system, calls=n, call_ms_median=float(np.median(ts)),
                       call_ms_min=float(ts.min()), queries_per_s_call=work / (np.median(ts) * 1e-3),
                       fitness_pose0=float(e["fitness"]), rmse_pose0=float(e["rmse"]))
            res["cases"].append(row)
            print(f"{label:4s} n={len(cloud):6d} M={M:5d} system={int(system)}: per call {row['call_ms_median']:.4f} ms median, "
                  f"{row['call_ms_min']:.4f} ms min ({n} calls); {row['queries_per_s_call'] / 1e6:.1f} M queries/s", flush=True)
    # kernel times: a separate, profiled pass
    from torch.profiler import ProfilerActivity, profile
    for label, cloud, M in cases:
        x = poses(M)
        for system in (True, False):
            reps = 10 if len(cloud) * M < 2e7 else 2
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    m.Evaluate(cloud, R0, t0, x, MAX_DIST, want_system=system)
            tot = {}
            for ev in prof.events():
                if ev.device_type.name != "CUDA":
                    continue
                key = "k_map_eval" if "k_map_eval<" in ev.name or "k_map_evalI" in ev.name else \
                      "k_eval_fin" if "k_eval_fin" in ev.name else "k_map_eval_prep" if "k_map_eval_prep" in ev.name else None
                if key:
                    tot[key] = tot.get(key, 0.0) + (getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0))
            per = {k: v / reps for k, v in tot.items()}
            row = next(r for r in res["cases"] if r["scan"] == label and r["M"] == M and r["system"] == system)
            row["kernel_us_per_call"] = per
            kq = per.get("k_map_eval", float("nan"))
            row["queries_per_s_kernel"] = len(cloud) * M / (kq * 1e-6)
            print(f"{label:4s} n={len(cloud):6d} M={M:5d} system={int(system)}: " +
                  ", ".join(f"{k} {v:.1f} us" for k, v in sorted(per.items())) +
                  f" per call; {row['queries_per_s_kernel'] / 1e9:.2f} G queries/s in k_map_eval", flush=True)
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
