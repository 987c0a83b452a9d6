"""The Stein phase (tail2.cu) checked at iterations after the first, on every path of the bandwidth median and every k_tail shape.

The bandwidth is h = (exact lower median of the P^2 pairwise squared distances) / log(P + 1).  k_head_* find the median by one of
three paths, reported per iteration by svnicp_get_median_paths: 0 sort of all pairs (P <= 64), 1 linear histogram over
[0.5, 1.5) x the previous median and a pick from the bin's values (iterations >= 1), 2 radix select (iteration 0, a window miss),
3 radix select after the bin held more than HD_COLLECT_CAP values.  k_tail runs as NI particles x JQ warps per CTA with a
TMA ring of record tiles; iteration e reads the record buffer of parity e & 1.

A tap at iteration e is a fresh scan of e + 1 iterations (svnicp_get_gn_system / _get_stein record the last executed
iteration); its particle history must equal the first e rows of one long scan, which proves the tap is that scan's state
(test_gpu_iteration_parity.py).  At every tap, on the tap's own x, H, b:
  - h is exactly m / L for the kernel-order median m (oracle_pair_median_kernel_order) and L one of log(P + 1) and its two
    neighbouring doubles (the device log may be one ulp off glibc's), and no such L maps the nearest distinct entries below
    and above m onto h: a median off by one rank fails even where a relative bar would pass;
  - delta against oracle.stein_step at the bars of test_gpu_parity.py::test_stein_step;
  - the particles after the tap against oracle.pose_update of the tap's x by the oracle's delta.
"""
import numpy as np
import pytest
import torch

import svn_icp_b200 as sv
from svn_icp_b200 import synth
from test_gpu_iteration_parity import particles, scan

pytestmark = pytest.mark.gpu

SM_COUNT = 148  # the case table below is laid out for a B200's SM count
REC = 41  # common.cuh: doubles per particle record
TL_WARPS, TL_ENV_CHUNK = 8, 1024  # tail2.cu: consumer warps of k_tail, particles per envelope pass
HD_SMALL_P, HD_COLLECT_CAP = 64, 4096  # tail2.cu
RTOL, ATOL = 1e-8, 1e-12  # test_gpu_parity.py::test_stein_step
SORT, FAST, RADIX, OVERFLOW = sv.MEDIAN_SORT, sv.MEDIAN_FAST, sv.MEDIAN_RADIX, sv.MEDIAN_OVERFLOW


@pytest.fixture(scope="module")
def lidar():
    return synth.make_problem(64, sensor="32", scan_index=6, n_map_scans=6, seed=0xC0FFEE)


@pytest.fixture(scope="module")
def c2():
    return synth.make_problem_saturated(4096, sensor="128")


@pytest.fixture(scope="module")
def sm_count():
    n = torch.cuda.get_device_properties(0).multi_processor_count
    assert n == SM_COUNT, f"the k_tail / k_head shapes of this file are laid out for {SM_COUNT} SMs, this device has {n}"
    return n


def tail_shape(P_l, sm):
    """tail2.cu tail_shape: (NI, JQ, stages, tiles, CTAs)"""
    ni = 8
    while ni > 1 and (P_l + ni - 1) // ni < (sm * 4) // 5:
        ni >>= 1
    jq = TL_WARPS // ni
    stages = min(12, max(1, (150 * 1024) // (32 * jq * REC * 8)))
    return ni, jq, stages, -(-P_l // (32 * jq)), -(-P_l // ni)


def head_grid(P, sm):
    """tail2.cu head_grid: CTAs of the multi-CTA median chain"""
    return 1 if P < 2 else min(max(-(-(P * P // 2) // 4096), 4), sm)


# ---- the checks at a tap ------------------------------------------------------------------------------------------------
def log_candidates(P):
    L = np.log(np.float64(P + 1))
    return (np.nextafter(L, 0.0), L, np.nextafter(L, np.inf))


def bandwidth_errors(oracle, x, h, what):
    m, below, above = oracle.pair_median_kernel_order(x)
    Ls = log_candidates(len(x))
    errs = []
    if not any(np.float64(h) == np.float64(m) / L for L in Ls):
        errs.append(f"{what}: h = {h!r}, kernel-order median {m!r} / log(P+1) = {m / Ls[1]!r}")
    for v in (below, above):
        if np.isfinite(v) and any(np.float64(v) / L == np.float64(h) for L in Ls):
            errs.append(f"{what}: h = {h!r} is also reached from the neighbouring distinct entry {v!r} (median {m!r})")
    return errs


def close_errors(got, want, what, rtol=RTOL, atol=ATOL):
    try:
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol)
    except AssertionError as err:
        return [f"{what}: {str(err).strip().splitlines()[:6]}"]
    return []


def svn_tap_errors(oracle, icp, full, lr, what, P):
    """all checks of one SVN-ICP tap; a list of failures (empty = pass)"""
    H, b, x = icp.get_gn_system()
    delta, h = icp.get_stein()
    errs = [] if P == 1 else bandwidth_errors(oracle, x, h, what)
    od, _ = oracle.stein_step(x, H, b, full=full, lr=lr)
    if np.isnan(od).any():
        if not (np.isnan(od).all() and np.isnan(delta).all()):
            errs.append(f"{what}: NaN deltas: kernel {np.isnan(delta).sum()}, oracle {np.isnan(od).sum()} of {od.size}")
        return errs, delta, h
    errs += close_errors(delta, od, f"{what}: delta")
    R = np.stack([oracle.so3_exp(v[3:])[0] for v in x])
    R2, t2 = oracle.pose_update(R, np.ascontiguousarray(x[:, :3]), od)
    want = np.concatenate([t2, np.stack([oracle.so3_log(r) for r in R2])], axis=1)
    errs += close_errors(icp.get_particles().reshape(6, P).T, want, f"{what}: particles after the update", rtol=0, atol=1e-10)
    return errs, delta, h


def first_of_each_code(paths):
    return {int(c): int(np.flatnonzero(paths == c)[0]) for c in np.unique(paths) if c >= 0}


# ---- (a) SVN taps ---------------------------------------------------------------------------------------------------------
I_LONG = 30
TAPS = (0, 1, 2, 3, 8, 17, 29)

# (name, P, SVN_full_grad, source stride, initial spread in units of synth.PARTICLE_UB)
SVN_CASES = [
    ("P1-gn", 1, True, 1, 1),                # MODE 0, no median
    ("P3-full", 3, True, 1, 1),              # k_head_small
    ("P46-precond", 46, False, 1, 1),        # k_head_small, 1035 pairs padded to 2048
    ("P64-full", 64, True, 1, 1),            # k_head_small at its limit
    ("P65-full", 65, True, 1, 1),            # multi-CTA chain; k_tail NI 1, JQ 8, one stage, one tile
    ("P65-precond", 65, False, 1, 1),
    ("P300-precond", 300, False, 1, 1),      # NI 2, 3 stages, 3 tiles
    ("P513-full", 513, True, 1, 1),          # NI 4, 7 stages, 9 tiles: the ring wraps; last CTA partial
    ("P1000-full", 1000, True, 1, 1),        # bench shape: NI 8, 12 stages, 32 tiles
    ("P1100-precond-every6", 1100, False, 6, 1),  # NI 8, last CTA partial, envelope in two chunks
    ("P300-full-wide", 300, True, 1, 4),     # four times the spread: the first update shrinks the median out of the window
]


def test_case_table_covers_the_shapes(sm_count):
    """The cases reach every NI, a wrapping ring, a partial last CTA, the chunked envelope, and head grids from the floor of 4
    CTAs to the SM count (P = 4096 of test_svn_taps_c2)."""
    shapes = {name: tail_shape(P, sm_count) for name, P, *_ in SVN_CASES}
    for name, (ni, jq, st, tiles, ctas) in shapes.items():
        print(f"{name}: NI {ni} JQ {jq} stages {st} tiles {tiles} CTAs {ctas}")
    assert {s[0] for s in shapes.values()} == {1, 2, 4, 8}
    assert shapes["P513-full"][:4] == (4, 2, 7, 9) and 513 % 4
    assert shapes["P1000-full"][:4] == (8, 1, 12, 32)
    assert shapes["P300-precond"][:4] == (2, 4, 3, 3)
    assert shapes["P65-full"][:4] == (1, 8, 1, 1)
    assert shapes["P1100-precond-every6"][0] == 8 and 1100 % 8 and 1100 > TL_ENV_CHUNK
    assert any(tiles > st for _, _, st, tiles, _ in shapes.values()), "no case wraps the tile ring"
    assert {P for _, P, *_ in SVN_CASES if P > HD_SMALL_P} and head_grid(65, sm_count) == 4
    assert head_grid(4096, sm_count) == sm_count
    assert {e & 1 for e in TAPS} == {0, 1}


@pytest.mark.parametrize("case", SVN_CASES, ids=[c[0] for c in SVN_CASES])
def test_svn_taps(oracle, lidar, sm_count, case):
    name, P, full, step, spread = case
    pb, src = lidar, np.ascontiguousarray(lidar.source[::step])
    init = particles(pb, P) if spread == 1 else synth.init_particles(P, np.random.default_rng(P), ub=spread * synth.PARTICLE_UB)
    long = scan("svn", pb, src, init, I_LONG, full=full)
    hist, paths = long.get_particle_history(), long.get_median_paths()
    long.close()
    print(f"\n{name}: median paths {paths.tolist()}")
    taps = sorted(set(TAPS) | set(first_of_each_code(paths).values()))
    errs = []
    for e in taps:
        tap = scan("svn", pb, src, init, e + 1, full=full)
        np.testing.assert_array_equal(tap.get_particle_history()[:e], hist[:e], err_msg=f"iteration {e}: not the state of the long scan")
        np.testing.assert_array_equal(tap.get_median_paths(), paths[:e + 1])
        errs += svn_tap_errors(oracle, tap, full, 1.0, f"{name} iteration {e} (path {paths[e]})", P)[0]
        tap.close()
    assert not errs, "\n".join(errs)
    # the paths that ran
    if P == 1:
        assert (paths == -1).all()
    elif P <= HD_SMALL_P:
        assert (paths == SORT).all()
    else:
        assert paths[0] == RADIX and (paths[1:] >= FAST).all()
        assert FAST in paths[1:], "the fast path never ran"
        if spread > 1:
            assert paths[1] == RADIX, "the wide case was meant to miss the window at iteration 1"


def test_svn_taps_c2(oracle, c2, sm_count):
    """P = 4096 on a 110k-point subsample of the configs[2] scan: the head grid is capped at the SM count."""
    P, n_s = 4096, 110_000
    rng = np.random.default_rng(11)
    src = np.ascontiguousarray(c2.source[np.sort(rng.choice(len(c2.source), n_s, replace=False))])
    assert tail_shape(P, sm_count)[0] == 8 and head_grid(P, sm_count) == sm_count
    long = scan("svn", c2, src, c2.init_pose, 6)
    hist, paths = long.get_particle_history(), long.get_median_paths()
    long.close()
    print(f"\nP4096: median paths {paths.tolist()}")
    errs = []
    for e in (0, 1, 5):
        tap = scan("svn", c2, src, c2.init_pose, e + 1)
        np.testing.assert_array_equal(tap.get_particle_history()[:e], hist[:e])
        errs += svn_tap_errors(oracle, tap, True, 1.0, f"P4096 iteration {e} (path {paths[e]})", P)[0]
        tap.close()
    assert not errs, "\n".join(errs)
    assert paths[0] == RADIX and FAST in paths[1:]


# ---- (b) frozen particles: any x in front of the fast path -------------------------------------------------------------
# lr = 1e-20 with zero rotations: the rotation step is far below so3_exp's 1e-12 threshold (dR = I exactly) and the translation
# step far below half an ulp of coordinates >= 0.5 m, so x never changes and Exp(0) = I, Log(I) = 0 make x at iteration 0 equal
# to x at every later one.  (lr = 0 would not do: a zero rotation step makes Jl NaN, 1/a at a = 0, quirk Q7.)
FROZEN_LR = 1e-20


def lattice(nx, ny=None, nz=None, step=0.125):
    g = [1.0 + step * np.arange(n) for n in (nx, ny or nx, nz or nx)]
    t = np.stack(np.meshgrid(*g, indexing="ij"), axis=0).reshape(3, -1)
    return np.concatenate([t, np.zeros_like(t)], axis=0)


def frozen_random(P, seed=5):
    rng = np.random.default_rng(seed)
    t = rng.uniform(0.5, 1.5, (3, P)) * rng.choice([-1.0, 1.0], (3, P))
    return np.concatenate([t, np.zeros((3, P))], axis=0)


# (name, init [6, P], path at iterations 1..4, unordered pairs at the median (the lattices only))
FROZEN_CASES = [
    ("lattice5", lattice(5), FAST, 480),       # every collected value equal
    ("lattice10", lattice(10), FAST, 2940),    # near the cap of HD_COLLECT_CAP collected values
    ("lattice12", lattice(12), OVERFLOW, 21888),  # past the cap: radix takes over
    # past the cap too, but the median is copy 1415 of the run: a pick from the first HD_COLLECT_CAP values would find it
    ("lattice7x14x15", lattice(7, 14, 15), OVERFLOW, 14070),
    ("random300", frozen_random(300), FAST, None),
]


def frozen_scan(pb, src, init, I):
    prm = sv.SteinICPParam(iterations=I, KNN_count=100, max_dist=3.0, lr=FROZEN_LR, SVN_full_grad=True)
    icp = sv.SVNICP(prm, init)
    icp.add_cloud(src, pb.target, init)
    icp.set_initial_mean(pb.R0, pb.t0)
    assert icp.stein_align() == sv.ALIGN_SUCCESS
    return icp


@pytest.mark.parametrize("case", FROZEN_CASES, ids=[c[0] for c in FROZEN_CASES])
def test_frozen_particles(oracle, lidar, case):
    name, init, later, at_median = case
    P = init.shape[1]
    if at_median is not None:  # the premise of the case: how many of the P^2 entries equal the median
        d = init[:3, :, None] - init[:3, None, :]
        D = (d * d).sum(0)
        m = np.sort(D.ravel())[(P * P - 1) // 2]
        assert np.triu(D == m, 1).sum() == at_median
        assert (at_median > HD_COLLECT_CAP) == (later == OVERFLOW)
        first = ((P * P - 1) // 2 - int((D < m).sum())) // 2  # the median's place in the run of equal values
        print(f"\n{name}: the median is copy {first} of {at_median}")
    src = np.ascontiguousarray(lidar.source[::6])
    xs, hs, errs = [], [], []
    paths = None
    for e in range(5):
        tap = frozen_scan(lidar, src, init, e + 1)
        H, b, x = tap.get_gn_system()
        _, h = tap.get_stein()
        xs.append(x)
        hs.append(h)
        paths = tap.get_median_paths()
        errs += bandwidth_errors(oracle, x, h, f"{name} iteration {e}")
        tap.close()
    print(f"\n{name}: median paths {paths.tolist()}, h {hs[0]!r}")
    for e in range(1, 5):
        np.testing.assert_array_equal(xs[e], xs[0], err_msg=f"iteration {e}: the particles moved")
    np.testing.assert_array_equal(xs[0][:, 3:], 0.0)
    assert not errs, "\n".join(errs)
    assert paths[0] == RADIX and (paths[1:] == later).all(), paths
    assert all(h == hs[0] for h in hs[1:]), f"h differs between the paths: {hs}"


# ---- (c) exact zeros at iteration 0 ---------------------------------------------------------------------------------------
# g identical particles add g (g - 1) zero entries to the P diagonal zeros; against rank (P^2 - 1) / 2
ZERO_CASES = [
    ("P100-median0", 100, (70, 8, 4, 2), True, RADIX),    # 5000 zeros, rank 4999
    ("P100-above0", 100, (70, 8, 4), False, RADIX),       # 4998 zeros: the smallest positive distance
    ("P64-median0", 64, (45, 2, 2), True, SORT),          # 2048 zeros, rank 2047
    ("P64-above0", 64, (45, 2), False, SORT),             # 2046 zeros
]


@pytest.mark.parametrize("case", ZERO_CASES, ids=[c[0] for c in ZERO_CASES])
def test_zero_distances_iteration0(oracle, lidar, case):
    name, P, sizes, median0, path = case
    init = synth.init_particles(P, np.random.default_rng(P + 1))
    k = 0
    for g in sizes:
        init[:, k:k + g] = init[:, k:k + 1]
        k += g
    assert (P + sum(g * (g - 1) for g in sizes) > (P * P - 1) // 2) == median0
    icp = scan("svn", lidar, np.ascontiguousarray(lidar.source[::6]), init, 1)
    errs, delta, h = svn_tap_errors(oracle, icp, True, 1.0, name, P)
    assert not errs, "\n".join(errs)
    assert icp.get_median_paths().tolist() == [path]
    if median0:
        assert h == 0.0 and np.isnan(delta).all()  # 0 / 0 in the kernel matrix: NaN, as the reference (and P == 2)
    else:
        assert h > 0.0 and np.isfinite(delta).all()


# ---- (d) SVGD-ICP class ---------------------------------------------------------------------------------------------------
SVGD_TAPS = (0, 1, 3, 7)


@pytest.mark.parametrize("P", [64, 300])
def test_svgd_taps(oracle, lidar, P):
    """Same k_head_* chain on the SVGD-ICP class's single record buffer: h exact, the RBF Stein direction of get_stein against
    oracle.svgd_step on the tap's own x and gradient (bars of test_stein_step), the path codes recorded."""
    pb = lidar
    init = particles(pb, P)
    long = scan("svgd", pb, pb.source, init, SVGD_TAPS[-1] + 1)
    hist, paths = long.get_particle_history(), long.get_median_paths()
    long.close()
    print(f"\nSVGD P{P}: median paths {paths.tolist()}")
    errs = []
    for e in SVGD_TAPS:
        tap = scan("svgd", pb, pb.source, init, e + 1)
        np.testing.assert_array_equal(tap.get_particle_history()[:e], hist[:e], err_msg=f"iteration {e}: not the state of the long scan")
        np.testing.assert_array_equal(tap.get_median_paths(), paths[:e + 1])
        _, g, x = tap.get_gn_system()
        d, h = tap.get_stein()
        errs += bandwidth_errors(oracle, x, h, f"SVGD P{P} iteration {e}")
        od, _ = oracle.svgd_step(x, -g)
        errs += close_errors(d, od, f"SVGD P{P} iteration {e}: Stein direction")
        tap.close()
    assert not errs, "\n".join(errs)
    if P <= HD_SMALL_P:
        assert (paths == SORT).all()
    else:
        assert paths[0] == RADIX and (paths[1:] >= FAST).all() and FAST in paths[1:]
