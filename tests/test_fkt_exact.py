"""CPU side of the exact F(k,t) tests (tests/fkt_inputs.py): the FMA emulation, the exact reference, the restated
launch geometry, the summation model and its bound, and F*."""
from fractions import Fraction

import numpy as np
import pytest

import fkt_inputs as fi
from oracle import oracle as O


def _hard_fma_inputs(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.uniform(1, 2, n) * 2.0 ** rng.integers(-30, 31, n) * rng.choice([-1, 1], n)
    b = rng.uniform(1, 2, n) * 2.0 ** rng.integers(-30, 31, n) * rng.choice([-1, 1], n)
    c = rng.uniform(1, 2, n) * 2.0 ** rng.integers(-30, 31, n) * rng.choice([-1, 1], n)
    q = n // 4
    # cancellation: c = -fl(a b), the result is the product's rounding error (or exactly 0)
    c[:q] = -(a[:q] * b[:q])
    # exact zero: dyadic a, b with c = -a b exactly
    a[q:q + 100] = rng.integers(1, 2 ** 20, 100).astype(float)
    b[q:q + 100] = rng.integers(1, 2 ** 20, 100).astype(float)
    c[q:q + 100] = -a[q:q + 100] * b[q:q + 100]
    # ties: a b + c exactly halfway between two doubles (c = 1, a b = 2^-53 (1 + 2k) ... built from integers)
    m = rng.integers(1, 2 ** 26, q)
    a[2 * q:3 * q] = (2 * m + 1).astype(float) * 2.0 ** -27
    b[2 * q:3 * q] = 2.0 ** -27
    c[2 * q:3 * q] = rng.choice([1.0, -1.0, 2.0 ** 20, 3.0], q)
    return a, b, c


def test_fma_emulation_matches_fractions():
    a, b, c = _hard_fma_inputs(100_000, 1)
    got = fi.fma(a, b, c)
    want = np.array([fi.fraction_fma(x, y, z) for x, y, z in zip(a.tolist(), b.tolist(), c.tolist())])
    assert np.array_equal(got, want)
    # the cases were hard: many differ from the unfused a b + c, some cancel to exactly 0
    assert np.count_nonzero(got != a * b + c) > 10_000
    assert np.count_nonzero(got == 0.0) >= 100


def test_kernel_argument_on_dyadic_grid_is_plain_arithmetic():
    """Positions m / 2^10 and k components n / 2^10: every product and sum of k.r is exact, so the emulated FMAs
    and plain double arithmetic must give the same arguments -- an independent check of the emulation."""
    f = fi.dyadic_frames(3000, 1, seed=4)[0]
    k = fi.dyadic_kvec(64, seed=4)
    plain = (f[:, 0][None, :] * k[:, 0][:, None] + f[:, 1][None, :] * k[:, 1][:, None]) + f[:, 2][None, :] * k[:, 2][:, None]
    assert np.array_equal(fi.kernel_argument(f, k), plain)
    assert np.abs(plain).max() > 1e4  # arguments over several thousand turns


def test_geometry_restates_the_design_values():
    g = fi.geometry(1_000_000, 32, 64, 148)
    assert (g["chunks"][0]["P"], g["chunks"][0]["tiles_per"], g["launches"]) == (37, 53, 2)
    g = fi.geometry(1_000_001, 1, 64, 148)
    assert (g["chunks"][0]["P"], g["chunks"][0]["tiles_per"]) == (280, 7)
    g = fi.geometry(20001, 2, 1025, 148)
    assert [s["groups"] for s in g["slabs"]] == [1, 256] and g["launches"] == 3
    g = fi.geometry(8, 70000, 3, 148)
    assert [c["T"] for c in g["chunks"]] == [65535, 4465] and g["launches"] == 2
    assert fi.geometry(0, 5, 5, 148)["launches"] == 0
    assert fi.geometry(100, 5, 5, 148, threads=0)["threads"] == 256  # any other value than 128 or 256 means 256


def test_reference_against_fractions_of_long_double_terms():
    f = fi.walk_frames(300, 1, seed=2)[0]
    k = fi.kvectors(5)
    kr, c, s = fi.exact_terms(f, k)
    for terms in (c, s):
        R = fi._fsum_rows(terms)
        for i in range(len(k)):
            exact = sum((Fraction(float(x)) + Fraction(float(x - np.longdouble(float(x)))) for x in terms[i]), Fraction(0))
            assert R[i] == float(exact)


@pytest.mark.parametrize("N,T,K,threads", [(200, 1, 7, 256), (1537, 1, 65, 256), (3000, 1, 1025, 128), (5000, 3, 64, 256)])
def test_model_meets_its_bound_and_a_perturbed_term_misses_it(N, T, K, threads):
    frames = fi.decorrelated_frames(N, T, seed=N)
    kvec = fi.kvectors(K)
    geo = fi.geometry(N, T, K, 148, threads)
    ref = fi.reference(frames, kvec, geo, check_frames=[T - 1])
    R, tol_re, _, _ = ref[T - 1]
    ch = fi.chunk_of(geo, T - 1)
    _, c, _ = fi.exact_terms(frames[T - 1], kvec)
    c64 = c.astype(np.float64)
    for k in range(K):
        m, _, _ = fi.model_sum(c64[k], ch["P"], ch["tiles_per"], fi.groups_of(geo, k))
        assert abs(m - R[k].real) <= tol_re[k]
    if N <= 300:  # the bound is below 1e-12 only for small frames
        k = K - 1
        bad = c64[k].copy()
        bad[N // 2] += 1e-12
        m, _, _ = fi.model_sum(bad, ch["P"], ch["tiles_per"], fi.groups_of(geo, k))
        assert tol_re[k] < 1e-12 and abs(m - R[k].real) > tol_re[k]


def test_bound_is_much_tighter_than_the_old_tolerance():
    N = 100001
    frames = fi.walk_frames(N, 1, seed=9)
    kvec = fi.kvectors(8)
    geo = fi.geometry(N, 1, 8, 148)
    _, tr, ti, _ = fi.reference(frames, kvec, geo)[0]
    assert max(tr.max(), ti.max()) < 1e-13 * N / 20


def test_reference_small_agrees_with_the_general_model():
    frames = fi.walk_frames(8, 50, seed=1, sigma=0.5)
    kvec = fi.kvectors(3)
    geo = fi.geometry(8, 50, 3, 148)
    R, tr, ti = fi.reference_small(frames, kvec, geo)
    ref = fi.reference(frames, kvec, geo, check_frames=[0, 49])
    for t in (0, 49):
        assert np.array_equal(ref[t][0], R[t]) and np.allclose(ref[t][1], tr[t], rtol=1e-12)
        assert np.allclose(ref[t][2], ti[t], rtol=1e-12)


@pytest.mark.parametrize("K", [1, 7, 64])
def test_fkt_reference_against_fractions(K):
    rng = np.random.default_rng(K)
    rho = (rng.standard_normal((6, K)) + 1j * rng.standard_normal((6, K))) * 700.0
    rho[5] = 1j * rho[0]
    for o, l in [(0, 0), (0, 3), (2, 3), (1, 4), (0, 5)]:
        F, b = fi.fkt_exact(rho, o, l)
        assert F == fi.fkt_fraction(rho, o, l)
        assert b > 0
    assert fi.fkt_exact(rho, 0, 5)[0] == 0.0


def test_numpy_restatement_within_its_slack_of_the_exact_sum():
    """O.numpy_density_field (the reference's own operation order: np.dot, then libm cos / sin in double, pairwise
    sums) stays within its documented slack of R: 1e-13 N, the argument's rounding |k.r| u per term."""
    N = 100001
    frames = fi.walk_frames(N, 1, seed=3)
    kvec = fi.kvectors(8)
    geo = fi.geometry(N, 1, 8, 148)
    R, tr, ti, _ = fi.reference(frames, kvec, geo)[0]
    ref = O.numpy_density_field(frames[0], kvec)
    assert np.abs(ref - R).max() <= 1e-13 * N
