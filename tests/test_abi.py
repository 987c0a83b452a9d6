"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads and exports every symbol that
include/svnicp_b200.h declares.  No compute calls (there is no GPU here and no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import svn_icp_b200 as sv
from conftest import ROOT


@pytest.fixture(scope="module")
def lib():
    from svn_icp_b200 import build
    build.build()
    return sv.load_library()


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "svnicp_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(svnicp_[a-z0-9_]+)\s*\(", hdr)))


def test_header_symbols_exported(lib):
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/svnicp_b200.h but not exported"
    assert sorted(sv.EXPORTS) == names


def test_abi_version_and_defaults(lib):
    assert lib.svnicp_abi_version() == 2
    p = sv._CParams()
    lib.svnicp_default_params(C.byref(p))
    # SteinICPParam defaults, reference SVGDICP.h:41-57
    assert (p.iterations, p.batch_size, p.KNN_count, p.convergence_steps) == (50, 50, 100, 5)
    assert (p.lr, p.max_dist, p.convergence_threshold) == (0.02, 1.0, 1e-5)
    assert (p.use_minibatch, p.normalize_cloud, p.check_early_stop, p.SVN_full_grad) == (0, 1, 0, 1)
    assert p.optimizer == b"Adam"
    assert (p.flags, p.gn_stages, p.gn_smem_kb, p.debug_corr) == (0, 0, 0, 0)  # extensions default off
    d = sv.SteinICPParam()
    assert (d.iterations, d.lr, d.max_dist, d.KNN_count, d.SVN_full_grad) == (50, 0.02, 1.0, 100, True)


def test_every_export_has_argtypes(lib):
    """ctypes must know every signature (a missing argtypes entry lets a Python int be truncated to 32 bits)."""
    for n in declared_symbols():
        assert getattr(lib, n).argtypes is not None, n


def test_no_cpu_fallback(lib):
    """Without a CUDA device creation must fail loudly (SVNICP_ERR_NO_DEVICE), never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(sv.SvnIcpError, match="no CUDA device|no CPU fallback"):
        sv.SVNICP(sv.SteinICPParam(), np.zeros((6, 4)))


def test_particle_count_limit(lib):
    """P > 65535 is refused before any device work: the bandwidth median counts the P^2 pair distances in 32-bit histogram
    bins, and 65536^2 = 2^32 wraps them.  65535 passes that check (it then fails only where there is no device)."""
    hdr = open(os.path.join(ROOT, "include", "svnicp_b200.h")).read()
    assert int(re.search(r"#define\s+SVNICP_MAX_PARTICLES\s+(\d+)", hdr).group(1)) == sv.MAX_PARTICLES == 65535
    assert sv.MAX_PARTICLES ** 2 < 2 ** 32 <= (sv.MAX_PARTICLES + 1) ** 2
    for cls in (sv.SVNICP, sv.SVGDICP):
        with pytest.raises(sv.SvnIcpError, match="65536 exceeds 65535: the bandwidth median counts .* 32-bit histograms"):
            cls(sv.SteinICPParam(iterations=1), np.zeros((6, 65536)))
    with pytest.raises(sv.SvnIcpError, match="exceeds 65535"):
        sv.SVNICPBatch(sv.SteinICPParam(iterations=1), np.zeros((1, 6, 70000)))
    try:
        sv.SVNICP(sv.SteinICPParam(iterations=1), np.zeros((6, 65535))).close()
    except sv.SvnIcpError as err:
        assert "exceeds" not in str(err) and "no CUDA device" in str(err)


def test_particle_initialisers(lib):
    """initialize_particles / _gaussian (ICPUtils.cpp:45-75): bounds, clamping, P == 1 -> zeros, determinism."""
    ub = np.array([0.3, 0.2, 0.1, 0.004, 0.004, 0.012])
    a = sv.initialize_particles(1000, ub, -ub, seed=7)
    assert a.shape == (6, 1000)
    assert np.all(a <= ub[:, None]) and np.all(a >= -ub[:, None])
    assert np.all(np.abs(a.mean(axis=1)) < 0.1 * ub)
    np.testing.assert_array_equal(a, sv.initialize_particles(1000, ub, -ub, seed=7))
    assert np.abs(a - sv.initialize_particles(1000, ub, -ub, seed=8)).max() > 0
    np.testing.assert_array_equal(sv.initialize_particles(1, ub, -ub), np.zeros((6, 1)))
    cov = np.array([0.01, 0.01, 0.0025, 1e-6, 1e-6, 4e-6])
    g = sv.initialize_particles_gaussian(4000, cov, seed=3)
    sd = np.sqrt(cov)
    assert np.all(np.abs(g) <= 3 * sd[:, None] + 1e-15)
    np.testing.assert_allclose(g.std(axis=1), sd, rtol=0.08)
    np.testing.assert_array_equal(sv.initialize_particles_gaussian(1, cov), np.zeros((6, 1)))


def test_flag_constants_mirror_the_header():
    """Every SVNICP_FLAG_* of include/svnicp_b200.h has a Python twin FLAG_* with the same value, the values are distinct bits,
    and the debug-build switch of the loader is an explicit path (never a silent fallback)."""
    import re
    hdr = open(os.path.join(ROOT, "include", "svnicp_b200.h")).read()
    flags = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+SVNICP_FLAG_(\w+)\s+(\d+)", hdr)}
    assert len(flags) >= 8
    for name, value in flags.items():
        assert getattr(sv, "FLAG_" + name) == value, name
        assert value & (value - 1) == 0, f"{name} is not a single bit"
    assert len(set(flags.values())) == len(flags)
    assert sv.LIB_PATH.endswith(".so")
