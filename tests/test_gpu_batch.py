"""Throughput mode (BASELINE.json configs[3]): svnicp_batch_* runs several independent streams on one GPU with their scans
interleaved.  Each stream's result must be BIT-IDENTICAL to the same scan on an ordinary single handle."""
import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth

pytestmark = pytest.mark.gpu


# 20 iterations without early stop: every stream captures and replays its CUDA graphs while the scans are interleaved
@pytest.mark.parametrize("full,es,I", [(True, False, 9), (False, True, 9), (True, False, 20)],
                         ids=["True-False", "False-True", "True-False-20"])
def test_batched_streams_equal_single_handles(full, es, I):
    S, P = 5, 96
    rng = np.random.default_rng(11)
    pbs = [synth.make_problem(P, sensor="32", scan_index=5 + (s % 2), n_map_scans=5, seed=0xC0FFEE + (s % 2)) for s in range(2)]
    inits = np.stack([synth.init_particles(P, rng) for _ in range(S)])
    prm = sv.SteinICPParam(iterations=I, KNN_count=40, max_dist=3.0, lr=1.0, SVN_full_grad=full, check_early_stop=es, convergence_threshold=5e-3)
    batch = sv.SVNICPBatch(prm, inits)
    assert len(batch.streams) == S
    srcs = []
    for s, h in enumerate(batch.streams):
        pb = pbs[s % 2]
        src = pb.source[s::3]  # ragged: every stream has its own source size
        srcs.append(src)
        h.add_cloud(src, pb.target, inits[s])
        h.set_initial_mean(pb.R0, pb.t0)
    states = batch.stein_align()
    assert states == [sv.ALIGN_SUCCESS] * S
    # a second batched scan on the same handles (buffers reused) must reproduce itself
    first = [(h.get_particles().copy(), h.get_particle_history().copy(), h.iterations_done()) for h in batch.streams]
    for s, h in enumerate(batch.streams):
        pb = pbs[s % 2]
        h.add_cloud(srcs[s], pb.target, inits[s])
        h.set_initial_mean(pb.R0, pb.t0)
    assert batch.stein_align() == [sv.ALIGN_SUCCESS] * S
    for s, h in enumerate(batch.streams):
        np.testing.assert_array_equal(h.get_particles(), first[s][0])
    for s in range(S):
        pb = pbs[s % 2]
        one = sv.SVNICP(prm, inits[s])
        one.add_cloud(srcs[s], pb.target, inits[s])
        one.set_initial_mean(pb.R0, pb.t0)
        assert one.stein_align() == sv.ALIGN_SUCCESS
        np.testing.assert_array_equal(one.get_particles(), first[s][0])
        np.testing.assert_array_equal(one.get_particle_history(), first[s][1])
        assert one.iterations_done() == first[s][2]
        np.testing.assert_array_equal(one.get_cov_matrix(), batch.streams[s].get_cov_matrix())
        one.close()
    batch.close()
