"""CPU check of oracle_pair_median_kernel_order, the reference the GPU tests hold the bandwidth median of k_head_* against.

Distances: every unordered pair rounded as hd_sweep does (tail2.cu), s = fma(df0, df0, df1 * df1), then s = fma(df, df, s) for
d = 2..5, emulated exactly with fractions (each fma is one correctly rounded operation).  Order statistic: np.sort of the full
P x P matrix (diagonal zeros, every pair twice).  Inputs: random poses, lattices (exact ties at the median) and repeated
particles (runs of exact zeros that reach or pass the median rank)."""
from fractions import Fraction

import numpy as np
import pytest


def fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))  # one rounding: Fraction -> float rounds to nearest even


def fma_sq_sum(xi, xj):
    """sum_d (xi_d - xj_d)^2 rounded as the kernel rounds it"""
    df = [float(np.float64(xi[d]) - np.float64(xj[d])) for d in range(6)]  # IEEE subtraction, as on the device
    s = fma(df[0], df[0], df[1] * df[1])
    for d in range(2, 6):
        s = fma(df[d], df[d], s)
    return s


def reference(x):
    P = len(x)
    D = np.zeros((P, P))
    for i in range(P):
        for j in range(i + 1, P):
            D[i, j] = D[j, i] = fma_sq_sum(x[i], x[j])
    e = np.sort(D.ravel())
    m = e[(P * P - 1) // 2]
    below, above = e[e < m], e[e > m]
    return m, (below[-1] if len(below) else -np.inf), (above[0] if len(above) else np.inf), D


def random_poses(P, seed):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(-0.5, 0.5, (P, 3)), rng.uniform(-0.02, 0.02, (P, 3))], axis=1)


def lattice(n, step=0.125):
    g = np.arange(n) * step + 1.0
    t = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    return np.concatenate([t, np.zeros_like(t)], axis=1)


def groups(sizes, P, seed):
    """P particles: len(sizes) groups of identical ones, the rest distinct"""
    x = random_poses(P, seed)
    k = 0
    for g in sizes:
        x[k:k + g] = x[k]
        k += g
    return x


CASES = {
    "random-P25": random_poses(25, 1),      # 300 pairs
    "random-P64": random_poses(64, 2),      # 2016 pairs
    "random-P2": random_poses(2, 3),        # median is the diagonal zero
    "lattice-3cubed": lattice(3),           # 27 particles, ties at the median
    "lattice-4cubed": lattice(4),
    "zeros-at-median-P64": groups((45, 2, 2), 64, 4),   # 2048 zeros, rank 2047: median 0
    "zeros-below-median-P64": groups((45, 2), 64, 5),   # 2046 zeros: median is the smallest positive distance
    "zeros-all-P10": groups((10,), 10, 6),
}


@pytest.mark.parametrize("name", list(CASES))
def test_kernel_order_median_exact(oracle, name):
    x = CASES[name]
    m, lo, hi, D = reference(x)
    got = oracle.pair_median_kernel_order(x)
    assert got == (m, lo, hi)
    # the rounding order matters: neither a plain sum of squares nor fma from s = 0 in index order gives these values
    if name.startswith("random-P6"):
        d = x[:, None, :] - x[None, :, :]
        assert (((d ** 2).sum(-1)) != D).any()
        assert any(fma(d[i, j, 1], d[i, j, 1], d[i, j, 0] * d[i, j, 0]) != fma(d[i, j, 0], d[i, j, 0], d[i, j, 1] * d[i, j, 1])
                   for i in range(20) for j in range(i + 1, 20))


def test_zero_runs_against_the_rank():
    """The zero-count cases of the GPU tests: g identical particles add g (g - 1) zeros to the P diagonal ones."""
    for sizes, P, want_zero in (((70, 8, 4, 2), 100, True), ((70, 8, 4), 100, False), ((45, 2, 2), 64, True), ((45, 2), 64, False)):
        zeros = P + sum(g * (g - 1) for g in sizes)
        rank = (P * P - 1) // 2
        assert (zeros > rank) == want_zero, (sizes, zeros, rank)


@pytest.mark.parametrize("n", [5, 10])
def test_lattice_median_plain_sum(oracle, n):
    """Larger lattices: every coordinate is a multiple of 1/8 m, so each difference, square and sum is exact and the plain
    numpy sum is the kernel's value; the median against np.sort of the full matrix."""
    x = lattice(n)
    d = x[:, None, :3] - x[None, :, :3]
    e = np.sort((d * d).sum(-1).ravel())
    m = e[(len(x) ** 2 - 1) // 2]
    assert oracle.pair_median_kernel_order(x) == (m, e[e < m][-1], e[e > m][0])
