"""Golden vectors for the scans on the bench problem (bench.make_problem, BASELINE.json configs[1]) that tests/test_gpu_fullsize.py
and tests/test_gpu_parity.py compare against:

  bench_full_p1000.npz   P = 1000, the whole 64-beam scan (143k points), 30 iterations
  bench_sub6000_p64.npz  P = 64, a 6000-point subsample of that scan (bench._subsample), 12 iterations

Each file holds the fp64 outputs of the C restatement (oracle/, pinned to the reference's own outputs by
tests/test_oracle_golden*.py) and fingerprints of the seeded inputs, so a change of the problem generator fails loudly instead of
comparing different scans.  bench_full_p1000.npz also holds the particle mean of the reference's own sources (SVNICP.cpp with its
vendored knn.cu against libtorch CUDA) on the same scan, as recorded on a B200 by bench.py's `reference_on_gpu` leg
(profiles/r02_bench_n1.json); the oracle's mean agrees with it to 4e-12.

    python tests/golden/make_golden_bench.py      # CPU only; the full-size case takes about 13 minutes on 8 cores
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

# name -> (P, iterations, n_s cap (0 = whole scan))
CASES = {"bench_full_p1000": (1000, 30, 0), "bench_sub6000_p64": (64, 12, 6000)}


def fingerprint(pb, src):
    return dict(in_gt_rel=pb.gt_rel, in_R0=pb.R0, in_t0=pb.t0, in_init_pose=pb.init_pose, in_n=np.array([len(src), len(pb.target)]),
                in_source_sum=src.sum(0), in_target_sum=pb.target.sum(0))


def run_case(name: str) -> None:
    sys.path.insert(0, ROOT)
    import bench
    import oracle as orc

    P, I, cap = CASES[name]
    pb, _ = bench.make_problem(P)
    src = pb.source if not cap else bench._subsample(pb, cap)
    O = orc.Oracle()
    O.set_num_threads(os.cpu_count() or 1)
    o = O.align(bench._oracle_params(I), src, pb.target, pb.init_pose, pb.R0, pb.t0)
    out = dict(params=np.array([P, I, cap], dtype=np.float64), oracle_particles=o["particles"], oracle_mean=o["mean"],
               oracle_cov=o["cov"], oracle_state=np.array([o["state"]]), **fingerprint(pb, src))
    if name == "bench_full_p1000":
        rec = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_n1.json")))["reference_on_gpu"]
        assert (rec["particles"], rec["iterations"], rec["n_s"], rec["n_t"]) == (P, I, len(src), len(pb.target)), rec
        np.testing.assert_array_equal(np.array(rec["gt"]), pb.gt_rel)  # the recorded run saw the same problem
        out["reference_mean"] = np.array(rec["mean"])
        print(name, "|oracle mean - reference mean| =", np.abs(o["mean"] - out["reference_mean"]).max())
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "ok; mean", o["mean"])


if __name__ == "__main__":
    for n in sys.argv[1:] or CASES:
        run_case(n)
