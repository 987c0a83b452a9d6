"""Time of svnicp_map_refine (VoxelHashMap.Refine) against the loop a caller writes without it, on one GPU.

python scripts/map_refine_speed.py [--calls N] [--skip-host-loop] [--skip-e2e] [--json OUT]

Map: scans 0-11 of the 64-beam drive at 1 m / 20 points (DESIGN 10b).  Scans: scan 14 down-sampled on the host (uniform 0.5 m then
1.5 m, ~900 points) and in full (~143 k points).  max_dist = 3, 30 iterations, tol = 0, from poses within +-0.5 m / +-5 deg of
the truth.  Cases M = 1, 8, 64, 1024 (1024 on the small scan only).
  per call   CUDA events around the blocking call, median of --calls; alternated in the same process with the host loop:
             Evaluate with the system (blocks of 32 poses inside the call), then the fp64 oracle's update per pose on the host
             (tests/map_refine_oracle.c), 30 times.  The final poses of both must agree within 1e-9.
  kernels    torch.profiler in a separate pass: total device time of k_map_refine_eval, k_eval_fin and k_map_refine_step.
  e2e        whole-map Search (top 5, 0.25 m^2) + Refine at 3 then 1 m^2 on the 0.5 m scan, against Search + a fine Search + SVN-ICP
             registration from the winner (64 particles), on scan 14 against the saved map: wall time and error to the truth.
The seeding A/B runs this script against a build with -DSVN_RF_SEED=0 (SVNICP_B200_LIB selects the library).  Prints the card
name, power limit and max SM clock of the run.  Needs the GPU: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 0xC0FFEE
MAX_DIST = 3.0
ITERS = 30


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def timed(fn, calls):
    import torch
    ts = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), out


def host_loop(m, src, Rg, tg, x0):
    from test_map_refine_cpu import refine_update
    x = x0.copy()
    for _ in range(ITERS):
        ev = m.Evaluate(src, Rg, tg, x, MAX_DIST)
        x = np.stack([refine_update(x[:, j], ev["H"][j], ev["b"][j])[0] for j in range(x.shape[1])], axis=1)
    return x


def exp_so3(w):
    from test_map_refine_cpu import so3_exp
    return so3_exp(w)[0]


def e2e(m, world, pts, Rg, tg, sv, synth):
    import torch
    snap = m.Export()
    v = m.voxel_size_
    lo, hi = snap.voxels.min(0)[:2] * v, (snap.voxels.max(0)[:2] + 1) * v
    pre = sv.ScanPreprocessor(len(pts))
    p1, n1 = pre.downsample_uniform(pts.astype(np.float32), 0.5)
    p2, n2 = pre.downsample_uniform(p1, 1.5, n=n1, on_device=True)
    R0, t0 = np.eye(3), np.array([0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), tg[2]])
    counts = (int((hi[0] - lo[0]) / 0.5) + 1, int((hi[1] - lo[1]) / 0.5) + 1, 1, 1, 1, 90)
    steps = (0.5, 0.5, 0.0, 0.0, 0.0, np.deg2rad(4.0))
    src = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)).cuda()

    def err(R, t):
        return float(np.linalg.norm(t - tg)), float(np.linalg.norm(R @ Rg.T - np.eye(3)))

    def refine_route():
        s = m.SearchDevice(p2, n2, False, R0, t0, counts, steps, 0.25, top_k=5)
        r1 = m.RefineDevice(p1, n1, False, R0, t0, s["poses"], 3.0, iterations=ITERS)
        r2 = m.RefineDevice(p1, n1, False, R0, t0, r1["poses"], 1.0, iterations=ITERS)
        x = r2["poses"][:, np.lexsort((np.arange(5), -r2["inliers"]))[0]]
        return err(R0 @ exp_so3(x[3:]), t0 + R0 @ x[:3])

    def three_stage():
        s = m.SearchDevice(p2, n2, False, R0, t0, counts, steps, 0.25, top_k=5)
        best = s["poses"][:, 0]
        Rw, tw = R0 @ exp_so3(best[3:]), t0 + R0 @ best[:3]
        fine = m.SearchDevice(p2, n2, False, Rw, tw, (9, 9, 1, 1, 1, 9), (0.125, 0.125, 0.0, 0.0, 0.0, np.deg2rad(0.5)), 0.25)
        xf = fine["poses"][:, 0]
        Rb, tb = Rw @ exp_so3(xf[3:]), tw + Rw @ xf[:3]
        rng = np.random.default_rng(5)
        icp = sv.SVNICP(sv.SteinICPParam(iterations=30, KNN_count=32, max_dist=MAX_DIST, lr=1.0, SVN_full_grad=True),
                        synth.init_particles(64, rng))
        ptr, n_t = m.GetMapDevice(tb, 110.0)
        icp.add_cloud_device(src.data_ptr(), len(pts), ptr, n_t, synth.init_particles(64, rng))
        icp.set_initial_mean(Rb, tb)
        icp.stein_align()
        x = icp.get_transformation()
        return err(Rb @ exp_so3(x[3:]), tb + Rb @ x[:3])

    out = {}
    for name, fn in (("search+refine", refine_route), ("search+fine search+registration", three_stage)) * 2:
        torch.cuda.synchronize()
        t = time.perf_counter()
        e = fn()
        torch.cuda.synchronize()
        out.setdefault(name, []).append((time.perf_counter() - t) * 1e3)
        out[name + " error"] = e
    for name in ("search+refine", "search+fine search+registration"):
        print(f"e2e {name}: {min(out[name]):.1f} ms (best of 2 after the first), error {out[name + ' error'][0]:.4f} m / "
              f"{out[name + ' error'][1]:.2e}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=7)
    ap.add_argument("--skip-host-loop", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import svn_icp_b200 as sv
    from svn_icp_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("map_refine_speed: no CUDA device (this measurement has no CPU fallback)")
    name, limit = card()
    print(f"card: {name}; power limit, max SM clock: {limit}; library {sv.LIB_PATH}", flush=True)
    world = synth.make_world(SEED)
    m = sv.VoxelHashMap(1.0, 100.0, 20)
    for k in range(12):
        pts, (R, t) = synth.make_scan(world, k, "64", SEED)
        m.AddPointCloud(pts.astype(np.float32), R, t)
    pts, (Rg, tg) = synth.make_scan(world, 14, "64", SEED)
    full = pts.astype(np.float32)
    down = synth.uniform_downsample(synth.uniform_downsample(pts.astype(np.float64), 0.5), 1.5).astype(np.float32)
    rng = np.random.default_rng(1)
    results = []
    for label, src, Ms in (("small", down, (1, 8, 64, 1024)), ("full", full, (1, 8, 64))):
        for M in Ms:
            x0 = np.concatenate([rng.uniform(-0.5, 0.5, (3, M)), rng.uniform(-np.deg2rad(5), np.deg2rad(5), (3, M))])
            call = lambda: m.Refine(src, Rg, tg, x0, MAX_DIST, iterations=ITERS, tol=0.0)  # noqa: E731
            call()
            calls = args.calls if len(src) * M < 2e7 else max(3, args.calls // 2)
            row = dict(scan=label, n=len(src), M=M)
            if args.skip_host_loop:
                row["refine_ms"], r = timed(call, calls)
            else:
                hl = lambda: host_loop(m, src, Rg, tg, x0)  # noqa: E731
                ta, tb = [], []
                for _ in range(max(3, calls // 2)):  # alternated
                    t1, r = timed(call, 1)
                    t2, xh = timed(hl, 1)
                    ta.append(t1)
                    tb.append(t2)
                row["refine_ms"], row["host_loop_ms"] = float(np.median(ta)), float(np.median(tb))
                row["max_dx_vs_host_loop"] = float(np.abs(r["poses"] - xh).max())
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                call()
                torch.cuda.synchronize()
            ker = {}
            for e in prof.key_averages():
                for k in ("k_map_refine_eval", "k_eval_fin", "k_map_refine_step"):
                    if k in e.key:
                        ker[k] = ker.get(k, 0.0) + e.device_time_total / 1e3  # ms
            row["kernels_ms"] = ker
            results.append(row)
            print(json.dumps(row), flush=True)
    out = dict(card=name, limit=limit, lib=sv.LIB_PATH, rows=results)
    if not args.skip_e2e:
        out["e2e"] = e2e(m, world, pts, Rg, tg, sv, synth)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(out, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
