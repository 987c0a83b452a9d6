"""Device time of svnicp_evaluate at configs[1] (bench.make_problem(1000): 64-beam scan, ~143 k points, K = 100).

python scripts/evaluate_speed.py [--calls N] [--json OUT]

After one 1000-particle scan, times evaluate() for M = 1 (the result pose), 64 and 1000 (particles), each with and without
the Gauss-Newton system.  Per call: CUDA events on the handle's stream around the whole call (pose upload, kernels, result
copies).  Per kernel: torch.profiler in a separate pass (k_eval_corr, the table-streaming pass).  For M = 1 the table pass
moves 16 * N_s * (K + 1) bytes (the float4 candidate rows and the source points; the table is 232 MB, larger than L2, so every
call streams it from HBM) and is compared with the 6.46 TB/s copy bandwidth measured on this project's B200 (DESIGN.md).
Prints the card name and power limit of the run.  Needs the GPU: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_BW = 6.46e12  # bytes/s, measured device-to-device copy rate of a B200 (DESIGN.md, k_filter row)


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
    ap.add_argument("--calls", type=int, default=0, help="timed calls per case (default: 200 / 40 / 6 for M = 1 / 64 / 1000)")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import bench
    import svn_icp_b200 as sv

    if not torch.cuda.is_available():
        raise SystemExit("evaluate_speed: no CUDA device (this measurement has no CPU fallback)")
    name, limit = card()
    print(f"card: {name}; power limit, max SM clock: {limit}", flush=True)
    W = bench.WORKLOAD
    P = W["particles"]
    pb, _ = bench.make_problem(P)
    stream = torch.cuda.Stream()
    icp = sv.SVNICP(sv.SteinICPParam(iterations=W["iterations"], KNN_count=W["K"], max_dist=W["max_dist"], lr=W["lr"],
                                     SVN_full_grad=W["svn_full_grad"]), pb.init_pose)
    icp.set_stream(stream.cuda_stream)
    icp.add_cloud(pb.source, pb.target, pb.init_pose)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    n_s, K = len(pb.source), W["K"]
    parts = icp.get_particles().reshape(6, P)
    cases = {1: icp.get_transformation()[:, None], 64: parts[:, :64].copy(), 1000: parts[:, :1000].copy()}
    calls = {1: 200, 64: 40, 1000: 6}
    res = dict(card=name, power_limit_and_max_clock=limit, n_s=n_s, K=K, scan_ms=icp.get_timing()["total_ms"], cases=[])
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for M, poses in cases.items():
        for system in (True, False):
            n = args.calls or calls[M]
            for _ in range(2):
                icp.evaluate(poses, want_system=system)
            ts = []
            for _ in range(n):
                ev0.record(stream)
                icp.evaluate(poses, want_system=system)
                ev1.record(stream)
                ev1.synchronize()
                ts.append(ev0.elapsed_time(ev1))
            ts = np.array(ts)
            row = dict(M=M, system=system, calls=n, call_ms_median=float(np.median(ts)), call_ms_min=float(ts.min()))
            res["cases"].append(row)
            print(f"M={M:5d} system={int(system)}: per call {row['call_ms_median']:.4f} ms median, {row['call_ms_min']:.4f} ms min "
                  f"({n} calls)", flush=True)
    # kernel times: a separate, profiled pass
    from torch.profiler import ProfilerActivity, profile
    for M in (1, 64, 1000):
        for system in (True, False):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(calls[M] // 2 or 1):
                    icp.evaluate(cases[M], want_system=system)
            ks = [e for e in prof.events() if e.device_type.name == "CUDA" and "k_eval_corr" in e.name]
            us = np.array([getattr(e, "device_time", None) or getattr(e, "cuda_time", np.nan) for e in ks]) if ks else np.array([np.nan])
            n_pass = -(-M // 32)
            per_call = float(np.median(us)) * n_pass
            line = f"M={M:5d} system={int(system)}: k_eval_corr {np.median(us):.1f} us per pass x {n_pass} passes = {per_call:.1f} us per call"
            row = next(r for r in res["cases"] if r["M"] == M and r["system"] == system)
            row["corr_us_per_pass"] = float(np.median(us))
            if M == 1:
                bytes_moved = 16.0 * n_s * (K + 1)
                bw = bytes_moved / (np.median(us) * 1e-6)
                row.update(bytes=bytes_moved, bytes_per_s=bw, fraction_of_copy_bw=bw / COPY_BW)
                line += f"; {bytes_moved / 1e6:.1f} MB -> {bw / 1e12:.2f} TB/s = {100 * bw / COPY_BW:.1f} % of {COPY_BW / 1e12:.2f} TB/s"
            print(line, flush=True)
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
