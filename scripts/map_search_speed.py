"""Device time of svnicp_map_search (VoxelHashMap.Search) against the loop a caller would otherwise write: svnicp_map_evaluate
over the same grid poses in blocks of 32 (no Gauss-Newton system) and a ranking on the host.

python scripts/map_search_speed.py [--reps N] [--json OUT]

Map: the DESIGN 10b map (12 scans of the 64-beam sensor at 1 m / 20 points).  Cases: the down-sampled scan (uniform 0.5 m then
1.5 m, ~900 points) on a 41 x 41 x 1 x 1 x 1 x 72 grid (+-10 m at 0.5 m, 360 deg at 5 deg: 121 032 poses), and the full
scan (~143 k points) on a 21 x 21 x 1 x 1 x 1 x 9 grid (+-2.5 m at 0.25 m, +-8 deg at 2 deg: 3 969 poses); each at k = 1 and
k = 1024.  Per call: CUDA events around the blocking call, search and loop alternated in one process; both must give the same counts and winners.  Per kernel:
torch.profiler in a separate pass (k_map_search_count, k_map_search_topk, k_map_search_prep).  Prints the card name and power
limit of the run.  Needs the GPU: there is no CPU fallback."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from map_evaluate_speed import MAX_DIST, SEED, card  # noqa: E402

EV_BLOCK = 32  # poses per block of svnicp_map_evaluate


def evaluate_loop(m, cloud, R0, t0, x, k):
    """what a caller without svnicp_map_search does: blocks of 32 poses through Evaluate, then a host ranking"""
    M = x.shape[1]
    counts = np.zeros(M, dtype=np.int64)
    for j in range(0, M, EV_BLOCK):
        counts[j:j + EV_BLOCK] = m.Evaluate(cloud, R0, t0, x[:, j:j + EV_BLOCK], MAX_DIST, want_system=False)["inliers"]
    return counts, np.lexsort((np.arange(M), -counts))[:k]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3, help="alternated (search, loop) pairs per case")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import svn_icp_b200 as sv
    from svn_icp_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("map_search_speed: no CUDA device (this measurement has no CPU fallback)")
    name, limit = card()
    print(f"card: {name}; power limit, max SM clock: {limit}", flush=True)
    world = synth.make_world(SEED)
    m = sv.VoxelHashMap(1.0, 100.0, 20)
    for k in range(12):
        pts, (R, t) = synth.make_scan(world, k, "64", SEED)
        m.AddPointCloud(pts.astype(np.float32), R, t)
    src, (Rg, tg) = synth.make_scan(world, 12, "64", SEED)
    src = src.astype(np.float32)
    down = synth.uniform_downsample(synth.uniform_downsample(src.astype(np.float64), 0.5), 1.5).astype(np.float32)
    print(f"map: {m.Size()} voxels, {m.PointCount()} points; scan {len(src)} points, down-sampled {len(down)}", flush=True)
    big = ((41, 41, 1, 1, 1, 72), (0.5, 0.5, 0.0, 0.0, 0.0, np.deg2rad(5.0)))
    small = ((21, 21, 1, 1, 1, 9), (0.25, 0.25, 0.0, 0.0, 0.0, np.deg2rad(2.0)))
    cases = [("down", down, big, 1), ("down", down, big, 1024), ("full", src, small, 1), ("full", src, small, 1024)]
    res = dict(card=name, power_limit_and_max_clock=limit, map_voxels=m.Size(), map_points=m.PointCount(), n_full=len(src),
               n_down=len(down), max_dist=MAX_DIST, cases=[])
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = torch.cuda.current_stream()

    def timed(f):
        ev0.record(st)
        out = f()
        ev1.record(st)
        ev1.synchronize()
        return ev0.elapsed_time(ev1), out

    for label, cloud, (counts, steps), k in cases:
        M = int(np.prod(counts))
        x = sv.search_grid_poses(counts, steps, np.arange(M))
        m.Search(cloud, Rg, tg, counts, steps, MAX_DIST, top_k=k)  # warm-up
        t_s, t_l = [], []
        for _ in range(args.reps):
            ts, r = timed(lambda: m.Search(cloud, Rg, tg, counts, steps, MAX_DIST, top_k=k, want_counts=True))
            tl, (cl, il) = timed(lambda: evaluate_loop(m, cloud, Rg, tg, x, k))
            t_s.append(ts)
            t_l.append(tl)
        agree = bool(np.array_equal(r["counts"].reshape(-1), cl) and np.array_equal(r["index"], il))
        q = len(cloud) * M
        row = dict(scan=label, n=len(cloud), grid=list(counts), M=M, k=k, reps=args.reps, search_ms=float(np.median(t_s)),
                   loop_ms=float(np.median(t_l)), speedup=float(np.median(t_l) / np.median(t_s)),
                   search_queries_per_s=q / (np.median(t_s) * 1e-3), agree=agree, best_count=int(r["count"][0]))
        res["cases"].append(row)
        print(f"{label:4s} n={len(cloud):6d} M={M:6d} k={k:4d}: search {row['search_ms']:.2f} ms "
              f"({row['search_queries_per_s'] / 1e9:.2f} G queries/s), evaluate loop {row['loop_ms']:.2f} ms, "
              f"x{row['speedup']:.1f}; counts and winners agree: {agree}; best count {row['best_count']}", flush=True)
    from torch.profiler import ProfilerActivity, profile
    for label, cloud, (counts, steps), k in cases:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.Search(cloud, Rg, tg, counts, steps, MAX_DIST, top_k=k)
        per = {}
        for ev in prof.events():
            if ev.device_type.name != "CUDA":
                continue
            for key in ("k_map_search_count", "k_map_search_topk", "k_map_search_prep", "k_map_eval"):
                if key in ev.name and not (key == "k_map_eval" and "k_map_eval_prep" in ev.name):
                    per[key] = per.get(key, 0.0) + (getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0))
                    break
        row = next(r for r in res["cases"] if r["scan"] == label and r["k"] == k)
        row["kernel_us_per_call"] = per
        M = int(np.prod(counts))
        row["count_kernel_queries_per_s"] = len(cloud) * M / (per.get("k_map_search_count", float("nan")) * 1e-6)
        print(f"{label:4s} M={M:6d} k={k:4d}: " + ", ".join(f"{kk} {v:.0f} us" for kk, v in sorted(per.items())) +
              f"; {row['count_kernel_queries_per_s'] / 1e9:.2f} G queries/s in k_map_search_count", flush=True)
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    if not all(r["agree"] for r in res["cases"]):
        raise SystemExit("map_search_speed: search and evaluate loop disagree")


if __name__ == "__main__":
    main()
