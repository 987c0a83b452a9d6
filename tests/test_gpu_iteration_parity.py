"""Correspondences and the Gauss-Newton system checked at iterations after the first.

From iteration 1 on, the exact-pruning ball comes from the last CTA of k_tail (not k_prep), the pruning kernel can be
k_filter_reuse, and the rows are mostly one-to-four-candidate lists that k_gn walks with its short-list bodies.  The taps
(svnicp_get_correspondences, svnicp_get_gn_system) record the last executed iteration, so iteration e is tapped by a fresh
scan of e + 1 iterations; its particle history must first equal the first e rows of one long production scan (which
replays CUDA graphs at I >= 16, the debug_corr handle never does), which proves the tapped state is iteration e of that scan.
At every tap:
  (1) indices and mask bit-exact against oracle_corr_f32 (slot-by-slot strict '<' over the whole K-slot row) on the
      tap's own transforms, every particle and every row;
  (2) H and b of the production k_gn instantiation bit-equal to those of the debug_corr instantiation;
  (3) H and b against the fp64 oracle on the tap's correspondences (bars of test_gpu_evaluate.check_system);
  (4) the path under test ran: mean kept candidates per row, the reuse fraction, k_filter under the k_tail ball.
"""
import types

import numpy as np
import pytest

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_gpu_evaluate import check_system

pytestmark = pytest.mark.gpu

MAX_DIST = 3.0
FR_SWITCH = 12  # iter_kernels.cu: k_filter_reuse takes over once the previous iteration kept <= 12 candidates per row
GN_CONSUMERS, GN_FLUSH_ROWS, GN_FLUSH2 = 512, 32, 64  # kernels.h / iter_kernels.cu: k_gn's threads and accumulation levels


@pytest.fixture(scope="module")
def lidar():
    # 32-beam x 900 column synthetic scan (28.7k points) against a 6-scan voxel map
    return synth.make_problem(64, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)


@pytest.fixture(scope="module")
def c2():
    return synth.make_problem_saturated(4096, sensor="128")


def particles(pb, P):
    return pb.init_pose if P == pb.init_pose.shape[1] else synth.init_particles(P, np.random.default_rng(P))


def scan(cls, pb, src, init, I, K=100, max_dist=MAX_DIST, debug=False, flags=0, full=True):
    if cls == "svn":
        prm = sv.SteinICPParam(iterations=I, KNN_count=K, max_dist=max_dist, lr=1.0, SVN_full_grad=full, flags=flags, debug_corr=debug)
        icp = sv.SVNICP(prm, init)
    else:
        prm = sv.SteinICPParam(iterations=I, KNN_count=K, max_dist=max_dist, lr=0.03, optimizer="Adam", flags=flags, debug_corr=debug)
        icp = sv.SVGDICP(prm, init)
    icp.add_cloud(src, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    return icp


def check_indices(oracle, icp, max_dist, what, sel=None):
    """(1): the tap's idx / mask against oracle_corr_f32 on the tap's own transforms; a failure names the particle, the row and
    the slots (in the K-slot candidate row) that the kernel and the oracle picked."""
    xf, idx, mask = icp.get_correspondences()
    if sel is not None:
        xf, idx, mask = xf[sel], idx[sel], mask[sel]
    cidx, rel = icp.get_candidates(want_rel=True)
    oidx, omask = oracle.corr_f32(xf, icp.get_source_f32(), rel, cidx, max_dist)
    bad = np.argwhere((idx != oidx) | (mask != omask))
    if len(bad):
        p, r = bad[0]
        slot = lambda i: np.flatnonzero(cidx[r] == i).tolist()  # noqa: E731
        pytest.fail(f"{what}: {len(bad)} of {idx.size} (particle, row) pairs differ; first: particle "
                    f"{p if sel is None else sel[p]}, row {r}: kernel slot {slot(idx[p, r])} mask {mask[p, r]}, oracle slot "
                    f"{slot(oidx[p, r])} mask {omask[p, r]}")
    return xf, idx, mask


def check_svn_system(oracle, pb, src, icp, idx, mask, max_dist, sel=None, what=""):
    """(3): H, b against the fp64 oracle on the tap's correspondences, R and t from the record's x"""
    H, b, x = icp.get_gn_system()
    if sel is not None:
        H, b, x = H[sel], b[sel], x[sel]
    R = np.stack([oracle.so3_exp(v[3:])[0] for v in x])
    cH, cb = oracle.gn_given_corr(R, np.ascontiguousarray(x[:, :3]), pb.R0, pb.t0, src, pb.target, idx, mask, max_dist)
    try:
        check_system(H, b, cH, cb, types.SimpleNamespace(source=src))
    except AssertionError as err:
        raise AssertionError(f"{what}: H, b against the fp64 oracle") from err


SVN_TAPS = (0, 1, 2, 4, 8, 13, 19, 29, 39, 49)


# (P, SVN_full_grad, K, flags, source stride): non-UNI k_gn (P <= 32: 9, 30) and UNI (64, 65), an odd last pair (9, 65),
# k_filter with the k_tail ball at every iteration (FILTER_FULL), padded rows Kp > K (7, 33), the chunked envelope of k_tail
# (P_l = 1100 > TL_ENV_CHUNK = 1024) on a 4.8k-point subsample.  50 iterations: the lidar scan's lists shrink more slowly
# than those of the 64-beam bench scan.
SVN_CASES = [(P, full, 100, 0, 1) for P in (9, 30, 64, 65) for full in (True, False)] + [
    (30, True, 100, sv.FLAG_FILTER_FULL, 1), (30, True, 7, 0, 1), (64, False, 33, 0, 1), (1100, True, 100, 0, 6)]


def case_id(c):
    P, full, K, flags, step = c
    return f"P{P}-{'full' if full else 'precond'}-K{K}" + ("-filterfull" if flags else "") + (f"-every{step}" if step > 1 else "")


@pytest.mark.parametrize("case", SVN_CASES, ids=[case_id(c) for c in SVN_CASES])
def test_svn_taps_every_iteration(oracle, lidar, case):
    P, full, K, flags, step = case
    pb, src = lidar, np.ascontiguousarray(lidar.source[::step])
    init = particles(pb, P)
    I = SVN_TAPS[-1] + 1
    long = scan("svn", pb, src, init, I, K, flags=flags, full=full)
    hist = long.get_particle_history()
    kept = long.get_prune_stats()
    long.close()
    stats = scan("svn", pb, src, init, I, K, flags=flags | sv.FLAG_REUSE_STATS, full=full)
    np.testing.assert_array_equal(stats.get_particle_history(), hist)
    reuse = stats.get_prune_stats()
    stats.close()
    print(f"\n{case_id(case)}: mean kept per row at the taps", {e: round(float(kept[e]), 3) for e in SVN_TAPS},
          "reuse fraction", {e: round(float(reuse[e]), 4) for e in SVN_TAPS})
    for e in SVN_TAPS:
        dbg = scan("svn", pb, src, init, e + 1, K, debug=True, flags=flags, full=full)
        np.testing.assert_array_equal(dbg.get_particle_history()[:e], hist[:e], err_msg=f"iteration {e}: not the state of the long scan")
        _, idx, mask = check_indices(oracle, dbg, MAX_DIST, f"iteration {e}")
        H, b, x = dbg.get_gn_system()
        prod = scan("svn", pb, src, init, e + 1, K, flags=flags, full=full)
        Hp, bp, xp = prod.get_gn_system()
        np.testing.assert_array_equal(xp, x)
        np.testing.assert_array_equal(Hp, H, err_msg=f"iteration {e}: production k_gn differs from the debug_corr instantiation")
        np.testing.assert_array_equal(bp, b, err_msg=f"iteration {e}: production k_gn differs from the debug_corr instantiation")
        prod.close()
        check_svn_system(oracle, pb, src, dbg, idx, mask, MAX_DIST, what=f"iteration {e}")
        dbg.close()
    # (4) the paths ran (checked after the taps, so that a wrong pick is reported as such): long lists at iteration 0, k_filter
    # under the k_tail ball, k_filter_reuse taking whole iterations, short lists late.  On this scan the mean list plateaus at
    # 3.2 .. 5.8 candidates per row with the full gradient (measured on a B200), and the containment test of k_filter_reuse
    # fails for part of the rows at some late iterations (reuse fraction 0.3 .. 1.0), so these are coverage floors, not bars.
    if K > FR_SWITCH:
        assert kept[0] > 4
        assert any(kept[e - 1] > FR_SWITCH for e in SVN_TAPS if e >= 1), "no tap runs k_filter with the k_tail ball"
    if full and K == 100 and P <= 65:
        assert kept[SVN_TAPS[-1]] < 6
    if flags & sv.FLAG_FILTER_FULL:
        assert reuse.max() == 0.0
    elif P <= 65:
        assert sum(reuse[e] > 0.99 for e in SVN_TAPS) >= 2, "k_filter_reuse took fewer than two taps"


@pytest.mark.parametrize("P", [7, 64])
def test_svgd_first_order_taps(oracle, lidar, P):
    """SVGD-ICP class: k_gn<FIRST> at late iterations; the gradient against the fp64 oracle on the tap's correspondences at the
    tap's x (bars of test_gpu_svgd.py::test_first_order_gradient (1))."""
    pb = lidar
    init = particles(pb, P)
    taps = (0, 3, 7)
    hist = scan("svgd", pb, pb.source, init, taps[-1] + 1).get_particle_history()
    for e in taps:
        dbg = scan("svgd", pb, pb.source, init, e + 1, debug=True)
        np.testing.assert_array_equal(dbg.get_particle_history()[:e], hist[:e], err_msg=f"iteration {e}: not the state of the long scan")
        _, idx, mask = check_indices(oracle, dbg, MAX_DIST, f"iteration {e}")
        _, g, x = dbg.get_gn_system()
        _, gp, xp = scan("svgd", pb, pb.source, init, e + 1).get_gn_system()
        np.testing.assert_array_equal(xp, x)
        np.testing.assert_array_equal(gp, g, err_msg=f"iteration {e}: production k_gn<FIRST> differs from the debug_corr instantiation")
        og = oracle.svgd_grad_given_corr(x, pb.R0, pb.t0, pb.source, pb.target, idx, mask, MAX_DIST)
        np.testing.assert_allclose(g, og, atol=2e-6 * np.abs(og).max(), rtol=1e-5, err_msg=f"iteration {e}")


# ---- exact ties -----------------------------------------------------------------------------------------------------------
# Pythagorean ring of radius 5: 12 integer points at exactly distance 5 from the centre, in the centre's z-plane
RING = np.array([(5, 0), (-5, 0), (0, 5), (0, -5), (3, 4), (3, -4), (-3, 4), (-3, -4), (4, 3), (4, -3), (-4, 3), (-4, -3)], dtype=np.float64)
RING_SIZES = (1, 2, 3, 4, 5, 8, 12)
TIE_K = 32


def tie_problem(P, spread, n_rows=256, seed=7):
    """Every source point s (integer coordinates 100 m apart, R0 = I, t0 = 0) has its own cluster of map points: a subset of
    the ring around s (1 .. 12 points), then decoys.  Particles: zero rotation, translation (0, 0, z_p), z_p dyadic and
    distinct, so each query is s + (0, 0, z_p) and every ring point lies at exactly sqrt(25 + z_p^2) from it, in fp32 too.

    narrow: |z_p| < 1/4.  The pruned list is the ring subset alone (decoys at in-plane radius 6 and beyond), so the list class
            of k_gn follows the tie count: 1-2 -> two-candidate body, 3-4 -> 4-way tournament, 5+ -> long list.
    wide:   z_p in [2, 3).  Five decoys below the plane (|c| < 5, farther from every query than the ring) take slots 0..4, so
            the ties start inside chunk 1 of the long list and run across chunk boundaries; two in-plane decoys at radius 6 and
            four above the plane (|c| = 9.01, inside the pruning ball) end every list: past them the exact early exit fires."""
    rng = np.random.default_rng(seed)
    g = np.arange(n_rows)
    src = 100.0 * np.stack([g % 8, (g // 8) % 8, g // 64], axis=1).astype(np.float64)
    sizes = rng.choice(RING_SIZES, n_rows)
    below = np.array([(1, 0, -3.5), (-1, 0, -3.5), (0, 1, -3.5), (0, -1, -3.5), (0, 0, -3.75)])
    side = np.array([(6, 0, 0), (0, 6, 0)], dtype=np.float64)
    above = np.array([(0.5, 0, 9), (-0.5, 0, 9), (0, 0.5, 9), (0, -0.5, 9)])
    far6 = np.array([(6, 0, 0), (-6, 0, 0), (0, 6, 0), (0, -6, 0)], dtype=np.float64)
    tgt = []
    for s, n in zip(src, sizes):
        ring = np.c_[RING[rng.permutation(12)[:n]], np.zeros(n)]
        near = np.concatenate([below, ring, side, above]) if spread == "wide" else np.concatenate([ring, far6])
        a = 0.37 * np.arange(TIE_K + 4 - len(near))
        r = 20.0 + 0.25 * np.arange(len(a))
        fill = np.stack([r * np.cos(a), r * np.sin(a), np.zeros_like(a)], axis=1)  # fills the K nearest with the cluster's own points
        tgt.append(s + np.concatenate([near, fill]))
    tgt = np.concatenate(tgt)
    tgt = tgt[rng.permutation(len(tgt))]
    if spread == "narrow":
        z = (2.0 * np.arange(P) - (P - 1)) / 256.0
    else:
        z = 2.0 + np.round(np.arange(P) * 63.0 / max(P - 1, 1)) / 64.0
    assert len(np.unique(z)) == P
    init = np.zeros((6, P))
    init[2] = z
    return types.SimpleNamespace(source=src, target=tgt, R0=np.eye(3), t0=np.zeros(3), init_pose=init, sizes=sizes, z=z)


@pytest.mark.parametrize("spread", ["narrow", "wide"])
@pytest.mark.parametrize("P", [9, 64])
def test_exact_ties_lowest_slot_wins(oracle, P, spread):
    """Iteration 0 on a problem where every query has exact ties: the lowest slot must win in the two-candidate body, in the
    4-way tournament, and across the chunks of the long-list scan (chunk minimum + gn_recover); max_dist equals one
    particle's winning squared distance exactly (strict '<' of the mask, squared distance against the unsquared max_dist)."""
    pb = tie_problem(P, spread)
    z_eq = pb.z[3 * P // 4]
    max_dist = 25.0 + z_eq * z_eq
    assert np.float32(max_dist) == max_dist
    icp = scan("svn", pb, pb.source, pb.init_pose, 1, TIE_K, max_dist=max_dist, debug=True)
    xf, idx, mask = check_indices(oracle, icp, max_dist, f"ties ({spread})")
    # preconditions: zero rotation block, and the oracle really sees equal minima (as many as ring points)
    assert not xf[:, :9].any()
    cidx, rel = icp.get_candidates(want_rel=True)
    q = xf[:, None, None, 9:]  # [P, 1, 1, 3]: a = 0, so the query relative to q0 is tau
    d2 = (((q - rel[None]).astype(np.float64)) ** 2).sum(-1)  # exact: every operand is a small dyadic number
    ties = (d2 == d2.min(axis=2, keepdims=True)).sum(axis=2)
    np.testing.assert_array_equal(ties, np.broadcast_to(pb.sizes, ties.shape))
    np.testing.assert_array_equal(d2.min(axis=2), np.broadcast_to((25.0 + pb.z ** 2)[:, None], ties.shape))
    assert 0 < mask.sum() < mask.size and not mask[3 * P // 4].any()  # the particle at max_dist is masked on every row
    # the pruned lists are what the docstring of tie_problem says (kept candidates per row, summed over the rows)
    n_list = pb.sizes + (11 if spread == "wide" else 0)
    assert icp.get_prune_stats()[0] * len(pb.source) == pytest.approx(float(n_list.sum()), abs=1e-6)
    check_svn_system(oracle, pb, pb.source, icp, idx, mask, max_dist)


# ---- third accumulation level -----------------------------------------------------------------------------------------
def busiest_rows(P, n_s, TB, n_slices, n_pgroups):
    """Rows the thread of slice 0, row group 0 accumulates in k_gn (choose_shape / prepare_scan in capi.cu)."""
    pairs = (P + 1) // 2
    PG = 1
    while PG < pairs and PG < GN_CONSUMERS:
        PG <<= 1
    RG = GN_CONSUMERS // PG
    assert n_pgroups == (pairs + PG - 1) // PG
    n_tiles = (n_s + TB - 1) // TB
    rows = 0
    for tile in range(0, n_tiles, n_slices):
        rows += sum(1 for r in range(0, TB, RG) if tile * TB + r < n_s)
    return rows


def test_third_accumulation_level(oracle, c2):
    """P = 4096 (4 particle groups) on a 110k-point subsample of the configs[2] scan: the busiest k_gn thread accumulates more
    than GN_FLUSH2 x GN_FLUSH_ROWS rows, so its fp32 shared-memory sums are folded into the fp64 partial slot once and a
    remainder is added on top.  Iteration 0 and a late iteration (whose partial slots hold the previous iteration's sums)."""
    P, n_s = 4096, 110_000
    rng = np.random.default_rng(11)
    src = np.ascontiguousarray(c2.source[np.sort(rng.choice(len(c2.source), n_s, replace=False))])
    sel = np.unique(np.r_[0, 1, P - 2, P - 1, 1023, 1024, 2047, 2048, 3071, 3072, rng.choice(P, 54, replace=False)])
    hist = scan("svn", c2, src, c2.init_pose, 6).get_particle_history()
    for e in (0, 5):
        dbg = scan("svn", c2, src, c2.init_pose, e + 1, debug=True)
        info = dbg.get_scan_info()
        rows = busiest_rows(P, n_s, info["TB"], info["n_slices"], info["n_pgroups"])
        print(f"\niteration {e}: TB {info['TB']}, {info['n_slices']} slices x {info['n_pgroups']} particle groups, "
              f"{rows} rows for the busiest thread (fold at {GN_FLUSH2 * GN_FLUSH_ROWS})")
        assert rows >= 1.25 * GN_FLUSH2 * GN_FLUSH_ROWS
        np.testing.assert_array_equal(dbg.get_particle_history()[:e], hist[:e])
        _, idx, mask = check_indices(oracle, dbg, MAX_DIST, f"iteration {e}", sel=sel)
        H, b, x = dbg.get_gn_system()
        Hp, bp, _ = scan("svn", c2, src, c2.init_pose, e + 1).get_gn_system()
        np.testing.assert_array_equal(Hp, H)
        np.testing.assert_array_equal(bp, b)
        check_svn_system(oracle, c2, src, dbg, idx, mask, MAX_DIST, sel=sel, what=f"iteration {e}")
        dbg.close()


def test_whole_scan_debug_equals_production(lidar):
    """Every iteration, including those between the taps: the debug_corr handle (direct launches, DBG k_gn) and the production
    handle (CUDA-graph replay, production k_gn) give the same bits."""
    a = scan("svn", lidar, lidar.source, lidar.init_pose, 30, debug=True)
    b = scan("svn", lidar, lidar.source, lidar.init_pose, 30)
    np.testing.assert_array_equal(a.get_particles(), b.get_particles())
    np.testing.assert_array_equal(a.get_cov_matrix(), b.get_cov_matrix())
    np.testing.assert_array_equal(a.get_particle_history(), b.get_particle_history())
