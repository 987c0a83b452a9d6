"""Device time of svnicp_map_search (VoxelHashMap.Search) against the loop a caller would otherwise write: svnicp_map_evaluate
over the same grid poses in blocks of 32 (no Gauss-Newton system) and a ranking on the host.

python scripts/map_search_speed.py [--reps N] [--json OUT] [--pruned-only]

Map: the DESIGN 10b map (12 scans of the 64-beam sensor at 1 m / 20 points).  Cases: the down-sampled scan (uniform 0.5 m then
1.5 m, ~900 points) on a 41 x 41 x 1 x 1 x 1 x 72 grid (+-10 m at 0.5 m, 360 deg at 5 deg: 121 032 poses), and the full
scan (~143 k points) on a 21 x 21 x 1 x 1 x 1 x 9 grid (+-2.5 m at 0.25 m, +-8 deg at 2 deg: 3 969 poses); each at k = 1 and
k = 1024.  Per call: CUDA events around the blocking call, search and loop alternated in one process; both must give the same counts and winners.  Per kernel:
torch.profiler in a separate pass (k_map_search_count, k_map_search_topk, k_map_search_prep).  Then the pruned path
(want_counts=False) against the exhaustive one (want_counts=True) on the same rows, a coarse grid below the selection rule and
the whole map without a prior (see pruned_cases); both must return the same winners.  Prints the card name and power limit of
the run.  Needs the GPU: there is no CPU fallback."""
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
    ap.add_argument("--pruned-only", action="store_true", help="only the pruned-against-exhaustive cases")
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

    for label, cloud, (counts, steps), k in ([] if args.pruned_only else cases):
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
    for label, cloud, (counts, steps), k in ([] if args.pruned_only else cases):
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
    res["pruned"] = pruned_cases(sv, synth, m, world, down, Rg, tg, big, small, src, timed, args.reps)
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    if not all(r["agree"] for r in res["cases"]):
        raise SystemExit("map_search_speed: search and evaluate loop disagree")
    if not all(r["agree"] and r["violations"] in (0, -1) for r in res["pruned"]):
        raise SystemExit("map_search_speed: the pruned and exhaustive paths disagree")


def pruned_cases(sv, synth, m, world, down, Rg, tg, big, small, full, timed, reps):
    """The same search with want_counts=False (the pruned path where the grid allows blocks) and want_counts=True (every pose
    counted), alternated: the DESIGN 10d rows, a coarse grid whose blocks fall below the selection rule's size, and the whole
    map without a prior (scan 14 down-sampled, the map's x-y extent at 0.25 m, full yaw at 2 deg, max_dist = 0.25)."""
    snap = m.Export()
    v = m.voxel_size_
    lo, hi = snap.voxels.min(0)[:2] * v, (snap.voxels.max(0)[:2] + 1) * v
    s14, (R14, t14) = synth.make_scan(world, 14, "64", SEED)
    d14 = synth.uniform_downsample(synth.uniform_downsample(s14.astype(np.float64), 0.5), 1.5).astype(np.float32)
    R0, t0 = np.eye(3), np.array([0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), t14[2]])
    whole = ((int((hi[0] - lo[0]) / 0.25) + 1, int((hi[1] - lo[1]) / 0.25) + 1, 1, 1, 1, 180),
             (0.25, 0.25, 0.0, 0.0, 0.0, np.deg2rad(2.0)))
    coarse = ((21, 21, 1, 1, 1, 72), (1.5, 1.5, 0.0, 0.0, 0.0, np.deg2rad(5.0)))
    cases = [("down", down, Rg, tg, big, 1, MAX_DIST, reps), ("down", down, Rg, tg, big, 1024, MAX_DIST, reps),
             ("full", full, Rg, tg, small, 1, MAX_DIST, reps), ("full", full, Rg, tg, small, 1024, MAX_DIST, reps),
             ("down", down, Rg, tg, coarse, 1, MAX_DIST, reps), ("down", down, Rg, tg, big, 1, 0.25, reps),
             ("whole", d14, R0, t0, whole, 1, 0.25, 1), ("whole", d14, R0, t0, whole, 5, 0.25, 1)]
    rows = []
    for label, cloud, Ra, ta, (counts, steps), k, md, nrep in cases:
        M = int(np.prod(counts))
        m.Search(cloud, Ra, ta, counts, steps, md, top_k=k)  # warm-up
        t_p, t_e = [], []
        for _ in range(nrep):
            tp, rp = timed(lambda: m.Search(cloud, Ra, ta, counts, steps, md, top_k=k))
            info = m.SearchInfo()
            te, re_ = timed(lambda: m.Search(cloud, Ra, ta, counts, steps, md, top_k=k, want_counts=True))
            t_p.append(tp)
            t_e.append(te)
        agree = all(np.array_equal(rp[f], re_[f]) for f in ("index", "poses", "count", "fitness", "rmse"))
        row = dict(scan=label, n=len(cloud), grid=list(counts), steps=[float(x) for x in steps], M=M, k=k, max_dist=md, reps=nrep,
                   pruned_ms=float(np.median(t_p)), exhaustive_ms=float(np.median(t_e)), agree=agree,
                   winners=[int(g) for g in rp["index"][:5]], best_count=int(rp["count"][0]), **info,
                   fraction_counted=info["poses_counted"] / M)
        if info["path"] == 1:  # the bound pass alone: the same bound queries as a count pass over the block centres
            row["bound_share"] = bound_share(sv, m, cloud, Ra, ta, counts, steps, md, k, info)
        rows.append(row)
        print(f"{label:5s} n={len(cloud):6d} M={M:9d} k={k:4d} max_dist={md:5.2f}: path {info['path']}, pruned {row['pruned_ms']:.2f} ms, "
              f"exhaustive {row['exhaustive_ms']:.2f} ms, x{row['exhaustive_ms'] / row['pruned_ms']:.2f}; "
              f"{info['blocks']} blocks of {info['poses_per_block']}, {info['blocks_counted']} counted, "
              f"fraction of poses counted {row['fraction_counted']:.4f}, bound share {row.get('bound_share', 0):.2f}, "
              f"violations {info['violations']}; winners {row['winners']} agree: {agree}", flush=True)
    return rows


def bound_share(sv, m, cloud, R0, t0, counts, steps, md, k, info):
    """share of the pruned call's device time spent in the bound pass (torch.profiler: k_map_search_count launches over
    block centres and the sort, against the whole call)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.Search(cloud, R0, t0, counts, steps, md, top_k=k)
    bound = total = 0.0
    seen_expand = False
    for ev in sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start):
        t = getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0)
        total += t
        seen_expand |= "k_map_search_expand" in ev.name
        if not seen_expand and any(x in ev.name for x in ("k_map_search_count", "k_map_search_bound_prep", "k_map_search_keys", "k_radix",
                                                            "k_scan_block_sums", "k_max_abs_finite")):
            bound += t
    return bound / total if total > 0 else float("nan")


if __name__ == "__main__":
    main()
