#!/usr/bin/env python
"""bench.py -- scans/sec of the SVN-ICP registration inner loop on N B200s (one process per GPU).

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--config 1|2|3|4]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one scan: add_cloud -> set_initial_mean -> stein_align -> getters (the call sequence of the
reference's caller, OdometryPipeline.cpp:582-607) on BASELINE.json configs[1]: synthetic 64-beam LiDAR scan
(~120k points) against its voxel-hash local map, 1000 particles, 30 iterations, early stop off, K = 100.
  value       scans/sec with the clouds already resident in HBM (device pointers), CUDA-event timed, max over ranks
  e2e         the same scan through the public API with HOST (pinned) clouds: H2D copies and result D2H inside the timing
  roofline    correspondence+reduction pass (k_filter + k_gn): algorithmic bytes / measured device time vs measured HBM peak
  cpu_baseline  the CPU checker timed on this box's host cores on a bounded sample (reported baseline, not the target)
  check       N > 1: rank 0 repeats the last scan on an unsharded handle and reports |sharded - single| (asserted <= 1e-7)
With N > 1 the particles are sharded across the ranks (strong scaling of the same scan; one record exchange per iteration).
--impl reference times the reference's own CPU implementation (oracle/_ref, libtorch on all host cores; the C port if
_ref is absent) on a bounded sample of the same workload and prints the same JSON line (same `config`).
--config 2/3/4: the other BASELINE.json configurations (parity / scaling / stress cases; not the driver's bench line).
--dump-outputs DIR: after the timed steps, write what the last timed scan returned as DIR/<name>.npy (float32/float64, at
most 64 MB); inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
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

WORKLOAD = dict(sensor="64", particles=1000, iterations=30, K=100, max_dist=3.0, lr=1.0, svn_full_grad=True,
                scan_index=8, n_map_scans=8)
METRIC = "scans/sec at 1000 particles (64-beam ~120k-pt synthetic scan, K=100, 30 SVN iterations)"
WORKLOAD_NAME = "configs[1]: 64-beam synthetic scan, 1000 particles, particle-sharded when N>1"
# N-GPU vs 1-GPU at the full size after 30 iterations: identical algorithm, but the grouping of the fp32 Gauss-Newton partial sums
# depends on the slice, and a near-tie correspondence that flips because of it moves single particles by ~1e-6..1e-5 through the
# repulsive dynamics (the same effect bounds ours-vs-reference at 7.6e-6).  Short scans agree to ~2e-9 (tests/mgpu_worker.py, 1e-7).
SHARD_TOL = 5e-5       # single particles
SHARD_TOL_MEAN = 1e-6  # particle mean


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def bench_config(n_s: int, n_t: int, world: int) -> dict:
    """The `config` object of the JSON line: built by this one function for BOTH arms, so they are identical."""
    P = WORKLOAD["particles"]
    return dict(workload=WORKLOAD_NAME, n_s=int(n_s), n_t=int(n_t),
                l2="candidate table 16*N_s*K bytes > 126 MB L2 is re-streamed every iteration; inputs are not L2 resident",
                particles_per_gpu=-(-P // max(world, 1)), **WORKLOAD)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                    samples=len(sm))


def make_problem(P, seed=0xC0FFEE, scan_index=None):
    from svn_icp_b200 import synth
    t = time.time()
    pb = synth.make_problem_saturated(P, sensor=WORKLOAD["sensor"], scan_index=WORKLOAD["scan_index"] if scan_index is None else scan_index,
                                      seed=seed)
    return pb, time.time() - t


def _subsample(pb, ns, seed=1):
    sel = np.sort(np.random.default_rng(seed).choice(len(pb.source), ns, replace=False))
    return pb.source[sel]


def _oracle_params(iters):
    import oracle as orc
    return orc.make_params(iterations=iters, knn_count=WORKLOAD["K"], max_dist=WORKLOAD["max_dist"], lr=WORKLOAD["lr"],
                           svn_full_grad=WORKLOAD["svn_full_grad"])


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, out, history, P):
    """--dump-outputs: the getters of the last timed scan (mean, distribution, covariance, particles [6][P], history [I][6][P]).
    Beyond DUMP_BYTES the particles and their history are a fixed, seeded sample of the particle columns, whose indices are
    written as particle_index.npy."""
    mean, dist, cov, particles = out
    particles = particles.reshape(6, P)
    history = history.reshape(len(history), 6, P)
    per_particle = particles.dtype.itemsize * 6 + history.dtype.itemsize * history.shape[0] * 6
    arrays = dict(transformation=mean, distribution=dist, cov_matrix=cov.reshape(6, 6))
    keep = min(P, (DUMP_BYTES - 4096) // (per_particle + 8))
    if keep < P:
        sel = np.sort(np.random.default_rng(0).choice(P, keep, replace=False))
        particles, history = particles[:, sel], history[:, :, sel]
        arrays["particle_index"] = sel.astype(np.float64)
    arrays.update(particles=particles, particle_history=history)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------------------------------------
# CPU legs (test infrastructure: the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------------------------
def cpu_baseline_port(pb, cand_idx):
    """The C restatement (OpenMP, all host cores).  MEASURED: one full-size Gauss-Newton iteration (all particles x all
    source points, the reference's 1-NN among K candidates + robust H, b) and one full-size Stein step.  The per-scan
    brute-force K-NN is timed on a row subset and scaled by the row count (every query row is an independent identical
    sweep over the whole map, so this leg is exactly linear).  scan = knn + iterations * (gn + stein)."""
    import oracle as orc
    O = orc.Oracle()
    cores = host_cores()
    O.set_num_threads(cores)  # torchrun exports OMP_NUM_THREADS=1: set the thread count explicitly
    P, I, K = pb.init_pose.shape[1], WORKLOAD["iterations"], WORKLOAD["K"]
    n_s = len(pb.source)
    R = np.stack([O.so3_exp(pb.init_pose[3:, p])[0] for p in range(P)])
    t = np.ascontiguousarray(pb.init_pose[:3].T)
    sub = 4096
    q0 = O.transform_q0(pb.source[:sub], pb.R0, pb.t0)
    O.knn_mink(q0[:256], pb.target, K)  # warm-up: thread pool, page-in of the map
    t0 = time.time()
    O.knn_mink(q0, pb.target, K)
    t_knn_sub = time.time() - t0
    t0 = time.time()
    H, b = O.gn(R, t, pb.R0, pb.t0, pb.source, pb.target, cand_idx, WORKLOAD["max_dist"])[:2]
    t_gn = time.time() - t0
    x = np.concatenate([t, np.zeros((P, 3))], axis=1)
    t0 = time.time()
    O.stein_step(x, H, b, full=WORKLOAD["svn_full_grad"], lr=WORKLOAD["lr"])
    t_stein = time.time() - t0
    t_knn = t_knn_sub * n_s / sub
    t_scan = t_knn + I * (t_gn + t_stein)
    return dict(value=1.0 / t_scan, unit="scans/sec", cores=O.num_threads(), kind="port", sampled=True,
                measured_s=dict(gn_one_full_iteration=t_gn, stein_one_step=t_stein, knn_rows=sub, knn_subset=t_knn_sub),
                extrapolated=dict(knn_full_s=t_knn, scan_s=t_scan, rule="knn * N_s/rows + iterations * (gn + stein)"),
                sample=f"C port (OpenMP, {O.num_threads()} threads): ONE full-size iteration measured (all {P} particles x all {n_s} "
                       f"points x K={K}: {t_gn:.1f}s) + one Stein step ({t_stein:.2f}s); brute-force K-NN timed on {sub} of {n_s} rows "
                       f"against the full {len(pb.target)}-point map ({t_knn_sub:.1f}s) and scaled by rows; scan = knn + {I} x (gn + stein)")


def cpu_config0(kind="port"):
    """BASELINE.json configs[0] in FULL on the host cores (no sampling): 100 particles, the voxel-down-sampled scan
    (uniform 0.5 m then 1.5 m, OdometryPipeline.cpp:559-560), full local map, 30 iterations."""
    import oracle as orc
    from svn_icp_b200 import synth
    pb, _ = make_problem(100)
    ds = np.ascontiguousarray(synth.uniform_downsample(synth.uniform_downsample(pb.source, 0.5), 1.5))
    prm = _oracle_params(WORKLOAD["iterations"])
    cores = host_cores()
    if kind == "reference":
        eng = orc.Reference()
        eng.set_num_threads(cores)
        call = lambda: eng.scan(prm, ds, pb.target, pb.init_pose, pb.R0, pb.t0)
    else:
        eng = orc.Oracle()
        eng.set_num_threads(cores)
        call = lambda: eng.align(prm, ds, pb.target, pb.init_pose, pb.R0, pb.t0)
    call()
    t0 = time.time()
    out = call()
    dt = time.time() - t0
    mean = out["mean"] if isinstance(out, dict) and "mean" in out else None
    return dict(workload="configs[0]: 100 particles, voxel-down-sampled 64-beam scan", n_s=int(len(ds)), n_t=int(len(pb.target)),
                particles=100, iterations=WORKLOAD["iterations"], seconds_per_scan=dt, scans_per_sec=1.0 / dt, cores=eng.num_threads(),
                kind=kind, sampled=False, mean=[float(v) for v in mean] if mean is not None else None)


def run_reference(args, rank, world):
    """--impl reference: the reference's own sources on the host cores (oracle/_ref; the C port if absent).  A step is a
    bounded sample of the bench workload (all particles, the full map, two source subsets x 1 and 2 iterations); the
    per-scan time follows from T(n_s, iters) = setup(n_s) + iters * (a + b n_s), fitted on the MEDIANS over the steps."""
    if rank != 0:
        return
    import oracle as orc
    P = WORKLOAD["particles"]
    pb, _ = make_problem(P)
    I = WORKLOAD["iterations"]
    ns_full = len(pb.source)
    cores = host_cores()
    if orc.ref_available():
        eng = orc.Reference()
        kind = "reference"
        call = lambda prm, src: eng.scan(prm, src, pb.target, pb.init_pose, pb.R0, pb.t0)
    else:
        eng = orc.Oracle()
        kind = "port"
        call = lambda prm, src: eng.align(prm, src, pb.target, pb.init_pose, pb.R0, pb.t0)
    eng.set_num_threads(cores)  # explicit: torchrun exports OMP_NUM_THREADS=1

    def run(ns, iters):
        src = _subsample(pb, ns)
        t0 = time.time()
        call(_oracle_params(iters), src)
        return time.time() - t0

    ns1, ns2 = 256, 1024  # ~5 s per step on a 16-core host
    for _ in range(max(args.warmup, 1)):
        run(ns1, 1)
    T = dict(a22=[], a21=[], a12=[], a11=[])
    t_begin = time.time()
    steps_done = 0
    for _ in range(args.steps):  # a step = one bounded sample (4 short runs)
        T["a22"].append(run(ns2, 2)); T["a21"].append(run(ns2, 1)); T["a12"].append(run(ns1, 2)); T["a11"].append(run(ns1, 1))
        steps_done += 1
        if time.time() - t_begin > 240.0:  # time box: the whole arm must end within a few minutes on any host
            break
    wall = time.time() - t_begin
    T22, T21, T12, T11 = (float(np.median(T[k])) for k in ("a22", "a21", "a12", "a11"))
    it2, it1 = max(T22 - T21, 1e-9), max(T12 - T11, 1e-9)
    b = max((it2 - it1) / (ns2 - ns1), 0.0)
    a = max(it2 - b * ns2, 0.0)
    setup2 = max(T21 - it2, 0.0)
    t_scan = setup2 * ns_full / ns2 + I * (a + b * ns_full)
    spread = float(np.std([x - y for x, y in zip(T["a22"], T["a21"])]) / it2) if steps_done > 1 else 0.0
    val = 1.0 / t_scan
    sample = (f"{kind} ({'libtorch CPU, device-swapped reference sources' if kind == 'reference' else 'C port'}, {eng.num_threads()} threads): "
              f"all {P} particles, full {len(pb.target)}-point map; per step 4 runs at N_s={ns1},{ns2} x iterations=1,2 (medians over "
              f"{steps_done} steps): setup {setup2:.2f}s@{ns2} pts, per iteration {a:.3f}s (Stein, N_s-independent) + {b * 1e3:.3f} ms/point; "
              f"extrapolated to N_s={ns_full}, {I} iterations")
    line = dict(metric=METRIC, value=val, unit="scans/sec", n_gpus=args.gpus, steps=steps_done, warmup=args.warmup,
                ms_per_step=wall / max(steps_done, 1) * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                impl="reference", sampled=True, config=bench_config(ns_full, len(pb.target), args.gpus),
                extrapolated=dict(scan_s=t_scan, ms_per_scan=t_scan * 1e3, rel_spread_of_iteration_time=spread,
                                  note="ms_per_step is the wall time of one bounded sample (what was timed); value = 1 / extrapolated full-scan time"),
                cpu_baseline=dict(value=val, unit="scans/sec", cores=eng.num_threads(), kind=kind, sample=sample, sampled=True),
                e2e=dict(value=val, unit="scans/sec", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    # configs[0] is small enough to be MEASURED in full on the host (separate process: the reference freezes the particle
    # count in function-static tensors, SVNICP.cpp:42,167)
    if not args.no_variants:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-config0", kind], cwd=ROOT, capture_output=True, text=True, timeout=600)
            line["config0_full_measurement"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as exc:  # noqa: BLE001
            line["config0_full_measurement"] = dict(error=f"{type(exc).__name__}: {str(exc)[:200]}")
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--particles", type=int, default=WORKLOAD["particles"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--cpu-config0", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--config", type=int, default=1, choices=(1, 2, 3, 4),
                    help="BASELINE.json configs index: 1 = the contract workload (default); 2 = 128-beam ~260k-point scan, 4096 particles; "
                         "3 = throughput mode, 8 independent streams x 256 particles per GPU; 4 = 10M-point map, 16384 particles")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed scan returned (mean, distribution, covariance, particles, particle history) "
                         "as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config in (3, 4)):
        ap.error("--dump-outputs covers the timed scan of --config 1 and 2 with --impl b200")
    if args.cpu_config0:
        print(json.dumps(cpu_config0(args.cpu_config0)))
        return
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    WORKLOAD["particles"] = args.particles
    global METRIC, WORKLOAD_NAME
    if args.config == 2:
        WORKLOAD.update(sensor="128", particles=4096 if args.particles == 1000 else args.particles)
        METRIC = "scans/sec at 4096 particles (128-beam ~260k-pt synthetic scan, K=100, 30 SVN iterations)"
        WORKLOAD_NAME = "configs[2]: 128-beam synthetic scan, 4096 particles, particle-sharded when N>1"
        args.no_variants = True
        args.no_cpu_baseline = True
    if args.config in (3, 4):
        import bench_extra
        return bench_extra.run(args, rank, world, local_rank)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import svn_icp_b200 as sv

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    P, I, K = WORKLOAD["particles"], WORKLOAD["iterations"], WORKLOAD["K"]
    pb, gen_s = make_problem(P)
    n_s, n_t = len(pb.source), len(pb.target)
    rng = np.random.default_rng(123)
    from svn_icp_b200 import synth
    particles = [synth.init_particles(P, rng) for _ in range(W + args.steps + 2)]

    def new_handle(flags=0, sharded=True, **kw):
        prm = sv.SteinICPParam(iterations=I, KNN_count=K, max_dist=WORKLOAD["max_dist"], lr=WORKLOAD["lr"], SVN_full_grad=WORKLOAD["svn_full_grad"],
                               check_early_stop=False, flags=flags, **kw)
        h = sv.SVNICP(prm, particles[0], device=local_rank)
        if world > 1 and sharded:
            uid = [sv.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            h.init_sharding(uid[0], rank, world)
        h.set_stream(stream.cuda_stream)
        return h

    stream = torch.cuda.current_stream()
    icp = new_handle()

    src_dev = torch.from_numpy(pb.source).to(dev)
    tgt_dev = torch.from_numpy(pb.target).to(dev)
    src_pin = torch.from_numpy(pb.source).pin_memory()
    tgt_pin = torch.from_numpy(pb.target).pin_memory()

    def scan_device(i, h=None):
        h = h or icp
        h.add_cloud_device(src_dev.data_ptr(), n_s, tgt_dev.data_ptr(), n_t, particles[i])
        h.set_initial_mean(pb.R0, pb.t0)
        assert h.stein_align() == sv.ALIGN_SUCCESS
        return h.get_transformation(), h.get_distribution(), h.get_cov_matrix(), h.get_particles()

    def scan_host(i):
        icp.add_cloud_pinned(src_pin.data_ptr(), n_s, tgt_pin.data_ptr(), n_t, particles[i])
        icp.set_initial_mean(pb.R0, pb.t0)
        assert icp.stein_align() == sv.ALIGN_SUCCESS
        return icp.get_transformation(), icp.get_distribution(), icp.get_cov_matrix(), icp.get_particles()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, first, count):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(count):
            out = fn(first + i)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    for i in range(W):
        scan_device(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, out = timed(scan_device, W, args.steps)
    launches = icp.launch_count() * args.steps
    clocks = sampler.stop() if rank == 0 else None
    last_hist, last_iters = icp.get_particle_history(), icp.iterations_done()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, last_hist, P)
    scan_host(0)
    ms_e2e, out_h = timed(scan_host, W, args.steps)

    # N > 1: the same scan (the last timed one) on an UNSHARDED handle on rank 0 -- the driver-visible multi-GPU parity figure
    check = dict(mean=[float(v) for v in out[0]], gt=[float(v) for v in pb.gt_rel])
    if world > 1:
        if rank == 0:
            single = new_handle(sharded=False)
            o1 = scan_device(W + args.steps - 1, single)
            d_part = float(np.nanmax(np.abs(o1[3] - out[3])))
            d_hist = float(np.nanmax(np.abs(single.get_particle_history() - last_hist)))
            d_mean = float(np.max(np.abs(o1[0] - out[0])))
            check["sharded_vs_single_max_abs"] = dict(particles=d_part, history_f32=d_hist, mean=d_mean,
                                                      cov=float(np.max(np.abs(o1[2] - out[2]))), iterations=[int(last_iters), int(single.iterations_done())],
                                                      tolerance=dict(particles=SHARD_TOL, mean=SHARD_TOL_MEAN),
                                                      ok=bool(d_part <= SHARD_TOL and d_mean <= SHARD_TOL_MEAN and last_iters == single.iterations_done()))
            single.close()
        barrier()

    # per-phase device times of one profiled scan (events around each launch group): the roofline numerators
    icp.set_profiling(True)
    scan_device(W)
    ph = icp.get_phase_times()
    info = icp.get_scan_info()
    prune = icp.get_prune_stats()
    icp.set_profiling(False)
    lo, hi = icp.slice()
    P_g = hi - lo
    hbm_peak, peak_src, sm_max = peaks()
    iters = max(ph["iterations"], 1)
    # algorithmic bytes per iteration per GPU (SURVEY.md 8(d), restated in DESIGN.md)
    b_alg = 16.0 * n_s * (1 + K) + 156.0 * P_g
    t_pass = (ph["filter_ms"] + ph["gn_ms"]) / iters * 1e-3
    # the HBM-streaming kernel alone: once the lists are short the default path prunes the previous iteration's lists
    # instead of streaming the K-slot table (k_filter_reuse), so its bytes/time is measured on a scan that streams the
    # table every iteration (SVNICP_FLAG_FILTER_FULL)
    icp_ff = new_handle(flags=sv.FLAG_FILTER_FULL)
    icp_ff.set_profiling(True)
    for _ in range(2):
        scan_device(W, icp_ff)
    ph_ff = icp_ff.get_phase_times()
    icp_ff.close()
    t_filter = ph_ff["filter_ms"] / max(ph_ff["iterations"], 1) * 1e-3
    fp32_peak_results = 148 * 128 * sm_max * 1e6  # FP32 results/s: 128 lanes per SM, as FFMA or FFMA2 (scripts/ubench/ffma2.cu)
    roofline = dict(bound="hbm", kernel="k_filter + k_gn (correspondence + Gauss-Newton reduction pass, per iteration)",
                    achieved=b_alg / t_pass / 1e9, peak=hbm_peak, unit="GB/s", frac=b_alg / t_pass / 1e9 / hbm_peak, traffic=None,
                    peak_source=peak_src, algorithmic_bytes_per_launch=b_alg, ms_per_launch=t_pass * 1e3,
                    note="the pass is FP32 bound for P >~ 20 (every loaded byte is reused by all particles: 0.57*P flop/B): k_gn "
                         "carries two particles per thread in packed fp32 (FFMA2), FMA pipe 62-67 % busy (ncu, profiles/); the "
                         "HBM-bound kernel of the path is k_filter alone (filter_only)",
                    filter_only=dict(achieved=16.0 * n_s * (1 + K) / t_filter / 1e9, frac=16.0 * n_s * (1 + K) / t_filter / 1e9 / hbm_peak,
                                     ms_per_launch=t_filter * 1e3,
                                     note="k_filter streaming the K-slot table every iteration (SVNICP_FLAG_FILTER_FULL scan)"),
                    gn_fp32=dict(ms_per_launch=ph["gn_ms"] / iters, pairs_per_launch=float(P_g) * n_s,
                                 fma_lane_cycles_per_pair=ph["gn_ms"] / iters * 1e-3 * fp32_peak_results / (float(P_g) * n_s),
                                 note="k_gn time expressed as FMA-pipe lane-cycles (128 per SM and clock at sm_max) per (particle, point) "
                                      "pair, averaged over the scan; the executed packed-instruction counts are in profiles/ (ncu)"))
    # dram__bytes_{read,write}.sum per launch from the committed ncu --set full captures (profiles/), if present
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        # mean over the scan: 10 early iterations (K-slot table streamed, long lists written and re-read) + 20 late ones
        roofline["traffic"] = tr["pass_bytes_per_launch_mean"]
        roofline["traffic_detail"] = tr
    except Exception:  # noqa: BLE001
        pass

    # secondary variants of the same scan (SURVEY.md 8(d)): the reference's own pre-processing (uniform down-sampling
    # 0.5 m then 1.5 m voxels, OdometryPipeline.cpp:559-560) and reference-style early stop (geodeAlpha.yaml:9,17-19)
    variants = {}
    if world == 1 and not args.no_variants:
        ds = synth.uniform_downsample(synth.uniform_downsample(pb.source, 0.5), 1.5)
        ds_dev = torch.from_numpy(np.ascontiguousarray(ds)).to(dev)

        def run_variant(h, src_ptr, ns, parts, steps=args.steps):
            def scan(i):
                h.add_cloud_device(src_ptr, ns, tgt_dev.data_ptr(), n_t, parts[i % len(parts)])
                h.set_initial_mean(pb.R0, pb.t0)
                h.stein_align()
                return h.get_transformation()
            scan(0)
            ms, mean = timed(scan, 1, steps)
            return dict(scans_per_sec=steps / (ms * 1e-3), ms_per_scan=ms / steps, mean=[float(v) for v in mean])

        variants["downsampled_source"] = dict(n_s=int(len(ds)), **run_variant(icp, ds_dev.data_ptr(), len(ds), particles))
        prm_es = sv.SteinICPParam(iterations=100, KNN_count=K, max_dist=WORKLOAD["max_dist"], lr=WORKLOAD["lr"],
                                  SVN_full_grad=WORKLOAD["svn_full_grad"], check_early_stop=True, convergence_threshold=5e-4)
        icp_es = sv.SVNICP(prm_es, particles[0], device=local_rank)
        icp_es.set_stream(stream.cuda_stream)
        variants["early_stop_thr5e-4_max100"] = run_variant(icp_es, src_dev.data_ptr(), n_s, particles)
        variants["early_stop_thr5e-4_max100"]["iterations_executed"] = icp_es.iterations_done()
        icp_es.close()
        # BASELINE.json configs[0]: 100 particles on the voxel-down-sampled scan (the reference's CPU-runnable case)
        p100 = [synth.init_particles(100, rng) for _ in range(4)]
        icp_c0 = sv.SVNICP(sv.SteinICPParam(iterations=I, KNN_count=K, max_dist=WORKLOAD["max_dist"], lr=WORKLOAD["lr"],
                                            SVN_full_grad=WORKLOAD["svn_full_grad"]), p100[0], device=local_rank)
        icp_c0.set_stream(stream.cuda_stream)
        variants["config0_p100_downsampled"] = dict(n_s=int(len(ds)), particles=100, **run_variant(icp_c0, ds_dev.data_ptr(), len(ds), p100))
        variants["config0_p100_raw_scan"] = dict(n_s=n_s, particles=100, **run_variant(icp_c0, src_dev.data_ptr(), n_s, p100))
        icp_c0.close()
        # the shipped regime (geodeAlpha.yaml:9-22): 30 particles, <= 100 iterations, early stop 5e-4, pre-conditioned SVGD step
        # (SVNFullGrad false), down-sampled source
        p30 = [synth.init_particles(30, rng) for _ in range(4)]
        icp_sh = sv.SVNICP(sv.SteinICPParam(iterations=100, KNN_count=K, max_dist=3.0, lr=1.0, SVN_full_grad=False, check_early_stop=True,
                                            convergence_threshold=5e-4), p30[0], device=local_rank)
        icp_sh.set_stream(stream.cuda_stream)
        variants["shipped_p30_es_downsampled"] = dict(n_s=int(len(ds)), particles=30, **run_variant(icp_sh, ds_dev.data_ptr(), len(ds), p30))
        variants["shipped_p30_es_downsampled"]["iterations_executed"] = icp_sh.iterations_done()
        icp_sh.close()
        # the other registration class behind the same interface (class_type = SVGDICP, SURVEY.md 8(f) row 2): same scan,
        # same particle count, the reference's shipped SVGD settings (Adam, lr 0.03; stein_icp params)
        prm_gd = sv.SteinICPParam(iterations=I, KNN_count=K, max_dist=WORKLOAD["max_dist"], lr=0.03, optimizer="Adam", check_early_stop=False)
        icp_gd = sv.SVGDICP(prm_gd, particles[0], device=local_rank)
        icp_gd.set_stream(stream.cuda_stream)
        variants["svgd_icp_class_adam"] = run_variant(icp_gd, src_dev.data_ptr(), n_s, particles, steps=min(args.steps, 5))
        icp_gd.set_profiling(True)
        icp_gd.add_cloud_device(src_dev.data_ptr(), n_s, tgt_dev.data_ptr(), n_t, particles[1])
        icp_gd.set_initial_mean(pb.R0, pb.t0)
        icp_gd.stein_align()
        variants["svgd_icp_class_adam"]["phases_ms_per_scan"] = icp_gd.get_phase_times()
        icp_gd.close()

    # The reference ITSELF on this GPU (SURVEY.md 8(d) item 3): its unmodified SVNICP sources + its vendored knn.cu against
    # libtorch CUDA (oracle/_ref/libsvnicp_ref_cuda.so, built by oracle/build_ref_cuda.sh), same scan, same particles, in a
    # subprocess (its O(P*N_s) fp64 temporaries peak at ~83 GB; a failure there must not take this bench down).  Also the
    # full-size parity figure: our particles against the reference's on the BASELINE-size problem.
    reference_on_gpu = None
    if world == 1 and not args.no_variants:
        ref_so = os.path.join(ROOT, "oracle", "_ref", "libsvnicp_ref_cuda.so")
        if os.path.exists(ref_so):
            tmp = tempfile.TemporaryDirectory(prefix="svnicp_bench_")  # the tree may be read-only
            out_npy = os.path.join(tmp.name, "ref_gpu_particles.npy")
            try:
                r = subprocess.run([sys.executable, "-m", "oracle.ref_gpu_run", str(P), str(I), "0", out_npy], cwd=ROOT, capture_output=True,
                                   text=True, timeout=420)
                reference_on_gpu = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as exc:  # noqa: BLE001
                reference_on_gpu = dict(ok=False, error=f"{type(exc).__name__}: {str(exc)[:200]}")
            if reference_on_gpu.get("ok"):
                icp.add_cloud_device(src_dev.data_ptr(), n_s, tgt_dev.data_ptr(), n_t, pb.init_pose)
                icp.set_initial_mean(pb.R0, pb.t0)
                icp.stein_align()
                ours = icp.get_particles().reshape(6, P)
                theirs = np.load(out_npy)
                reference_on_gpu.update(
                    scans_per_sec=1.0 / reference_on_gpu["seconds_scan"],
                    speedup_device=(args.steps / (ms_dev * 1e-3)) * reference_on_gpu["seconds_scan"],
                    parity_full_size=dict(max_abs_particle_diff=float(np.nanmax(np.abs(ours - theirs))),
                                          max_abs_mean_diff=float(np.max(np.abs(icp.get_transformation() - np.array(reference_on_gpu["mean"])))),
                                          note="our scan vs the reference's own GPU run, same inputs, 30 iterations, all particles"))
            tmp.cleanup()
        else:
            reference_on_gpu = dict(ok=False, error="oracle/_ref/libsvnicp_ref_cuda.so not built (oracle/build_ref_cuda.sh needs the reference's sources)")

    # CPU baseline (rank 0, N = 1 only): needs the candidate table for the full-size iteration -> one tiny parity-tap handle
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        tap = sv.SVNICP(sv.SteinICPParam(iterations=0, KNN_count=K, max_dist=WORKLOAD["max_dist"], debug_corr=True), np.zeros((6, 1)), device=local_rank)
        tap.add_cloud_device(src_dev.data_ptr(), n_s, tgt_dev.data_ptr(), n_t, np.zeros((6, 1)))
        tap.set_initial_mean(pb.R0, pb.t0)
        tap.stein_align()
        cand_idx = tap.get_candidates().astype(np.int64)
        tap.close()
        cpu_baseline = cpu_baseline_port(pb, cand_idx)
        if not args.no_variants:
            cpu_baseline["config0_full_measurement"] = cpu_config0("port")

    if rank == 0:
        h2d = (n_s + n_t) * 24 + 6 * P * 8
        d2h = (48 + 6 * P) * 8
        line = dict(metric=METRIC, value=args.steps / (ms_dev * 1e-3), unit="scans/sec", n_gpus=world, steps=args.steps, warmup=W,
                    ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32 geometry / f64 reduction+Stein",
                    data="synthetic", config=bench_config(n_s, n_t, world),
                    e2e=dict(value=args.steps / (ms_e2e * 1e-3), unit="scans/sec", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
                    gpu_launches=int(launches), roofline=roofline, clocks=clocks,
                    phases_ms_per_scan=ph, scan_info=info, prune_mean_kept=[round(float(x), 2) for x in prune], variants=variants,
                    check=check, datagen_s=gen_s)
        if reference_on_gpu is not None:
            line["reference_on_gpu"] = reference_on_gpu
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    icp.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
        if rank == 0 and not check["sharded_vs_single_max_abs"]["ok"]:
            raise SystemExit(f"sharded run differs from the single-GPU run: {check['sharded_vs_single_max_abs']}")


if __name__ == "__main__":
    main()
