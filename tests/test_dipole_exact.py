"""The neutral-molecule inputs of tests/dipole_inputs.py, their exact dipole and its tolerance, on the CPU.

Three things are shown here so that tests/test_dipole_exact_gpu.py can rely on them:
  * the builders do what they claim: molecules are intact when unwrapped, the dipole cancels heavily (condition number
    >= 1e7 at 1M particles with images of +-50 or more), the zero case sums to exactly 0;
  * math.fsum and the C oracle's orc_dipole_exact (what tests/test_force_gpu.py measures against) agree to 1 ulp;
  * the inputs are hard enough: a NumPy model of the kernels' reduction order meets the tolerance on every input the GPU
    tests run, and the same model with the low word dropped -- everywhere, or at the cross-thread fold only -- misses it
    by 10x or more on every input of 4096 particles or more.  The table the test prints (pytest -s) gives each error in
    ulp of D.
And one thing is recorded: on the shuffled inputs the reference's own serial sum is more than 1e-10 relative off D, so
the reference cannot judge a kernel's dipole there.
"""
import math

import numpy as np
import pytest

import dipole_inputs as di

GPU_SIZES = [33, 700, 768, 769, 4096, 8192, 150001, 262145, 500000, 1000001]
CPU_SIZES = [33, 4096, 150001, 1000001]
MODEL_THREADS = [295 * 384, 16 * 512]  # the folder step's streaming grid; a 16-CTA cluster of 512 threads


def _inputs(kinds, sizes):
    return [(k, N) for k in kinds for N in sizes]


_CACHE = {}


def system(kind, N):
    if (kind, N) not in _CACHE:
        s = di.build(kind, N)
        ph = di.photon_index(s)
        t = di.dipole_terms(s.pos, s.charge, s.image, s.box, ph)
        D, S = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph)
        _CACHE.clear()  # one large input at a time
        _CACHE[(kind, N)] = (s, ph, t, D, S)
    return _CACHE[(kind, N)]


@pytest.mark.parametrize("kind,N", _inputs(list(di.KINDS) + list(di.MORE_KINDS), CPU_SIZES))
def test_builders(kind, N):
    s, ph, t, D, S = system(kind, N)
    opts = {**di.MORE_KINDS, **di.KINDS}[kind]
    L = np.asarray(s.box)
    assert s.N == N and s.pos.dtype == np.float64 and s.image.dtype == np.int32
    # HOOMD's layouts: float32 positions inside the box, float32-exact charges
    assert np.array_equal(s.pos[:, :3], s.pos[:, :3].astype(np.float32).astype(np.float64))
    assert np.all(s.pos[:, :3] >= -L / 2) and np.all(s.pos[:, :3] < L / 2)
    assert np.array_equal(s.charge, s.charge.astype(np.float32).astype(np.float64))
    # the photon is the first 'L' particle, where it was asked for; the further 'L' particles cancel in +- pairs
    isL = np.nonzero(s.typeid == s.L_typeid)[0]
    assert ph == di.photon_slot(N, opts["photon"]) == isL[0]
    assert len(isL) == 1 + len(di.extra_L_slots(N, ph) if opts.get("extra_L") else [])
    if len(isL) > 1:
        assert math.fsum(s.charge[isL[1:]]) == 0.0 and np.abs(s.image[isL[1:]]).max() > 100
        assert isL[1] == ph + 1 and (isL[-1] == N - 1 or ph == N - 1)  # the photon's warp and the last particle
    if opts.get("big_photon"):
        assert s.charge[ph] == di.BIG_PHOTON_CHARGE and tuple(s.image[ph]) == di.BIG_PHOTON_IMAGE
    # neutral molecules: the charge sums to zero
    mol = s.typeid != s.L_typeid
    assert math.fsum(s.charge[mol]) == 0.0
    # molecules intact when unwrapped: rebuild them from the layout and look at their bonds
    q = s.charge[mol]
    u = di.unwrapped(s.pos, s.image, s.box)[mol]
    size = opts["size"]
    lead = q == (di.Q_DIMER if size == 2 else -2.0 * di.Q_WATER)
    n_mol = int(lead.sum())
    assert n_mol == (N - len(isL)) // size
    if opts["order"] != "shuffled":
        idx = np.nonzero(q != 0.0)[0][:n_mol * size]
        atoms = idx.reshape(n_mol, size) if opts["order"] == "adjacent" else idx.reshape(size, n_mol).T
        bonds = np.linalg.norm(u[atoms[:, 1:]] - u[atoms[:, :1]], axis=2)
        want = 0.0 if opts.get("zero") else di.BOND
        assert np.abs(bonds - want).max() <= L[0] * 2.0 ** -22  # float32 rounding of the wrapped partner
        assert np.abs(s.image[mol][atoms[:, 1:]] - s.image[mol][atoms[:, :1]]).max() <= 1
    # cancellation: the dipole is a small remainder of large terms
    if opts.get("zero"):
        assert np.all(D == 0.0)
    elif N >= 1000000 and opts["images"] >= 50:
        assert np.all(S / np.abs(D) >= 1e7), S / np.abs(D)


@pytest.mark.parametrize("kind,N", _inputs(list(di.KINDS) + list(di.MORE_KINDS), CPU_SIZES))
def test_fsum_against_oracle_dipole_exact(coracle, kind, N):
    """orc_dipole_exact (long-double Neumaier) is within 1 ulp of the correctly rounded sum on every builder case."""
    s, ph, t, D, S = system(kind, N)
    o = coracle.dipole_exact(s.pos, s.charge, s.image, s.box, ph)
    if np.all(D == 0.0):
        assert np.all(o == 0.0)
    else:
        assert np.all(di.ulps(o, D) <= 1.0), di.ulps(o, D)


@pytest.mark.parametrize("kind,N", _inputs(list(di.KINDS) + list(di.MORE_KINDS), [33, 4096, 262145]))
def test_finalize_restates_the_reference(coracle, kind, N):
    """dipole_inputs.finalize / force_rows fed the oracle's own (serial-sum) dipole give the oracle's energies and force
    array bit for bit: the GPU tests may then demand the same of a kernel fed its own d."""
    s, ph, t, D, S = system(kind, N)
    ref = coracle.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, di.OMEGAC, di.G, di.PHMASS)
    assert ref["photon_idx"] == ph
    c = di.constants()
    en, Dq, FL = di.finalize(ref["dipole"], di.unwrapped(s.pos, s.image, s.box)[ph], c)
    assert np.array_equal(en.view(np.uint64), ref["energies"].view(np.uint64))
    f = di.force_rows(s.charge, s.typeid, s.L_typeid, ph, Dq, FL, c)
    assert np.array_equal(f.view(np.uint64), ref["force"].view(np.uint64))


@pytest.mark.parametrize("kind,N", _inputs(list(di.KINDS), GPU_SIZES))
def test_model_meets_tolerance_and_mutants_miss_it(kind, N):
    s, ph, t, D, S = system(kind, N)
    tol = di.tolerance(D, S, N)
    row = []
    for threads in MODEL_THREADS:
        for mode in ("kernel", "no_lo", "drop_fold"):
            d = np.array([di.model_sum(t[:, k], threads, mode) for k in range(3)])
            err = np.abs(d - D)
            row.append(f"{mode}/{threads}: {di.ulps(d, D).max():.3g} ulp")
            if mode == "kernel":
                assert np.all(err <= tol), (threads, err, tol)
            elif N >= 4096:
                # every component: a kernel that lost its low word must fail on each of them
                assert np.all(err >= 10 * tol), (mode, threads, err / tol)
    print(f"\n{kind:12s} N={N:8d} tol {(tol / np.spacing(np.abs(D))).max():.3g} ulp | " + " | ".join(row))


def test_model_at_16M():
    """The one 16M-particle input of the GPU tests."""
    test_model_meets_tolerance_and_mutants_miss_it("adj50", 16 * 2 ** 20 + 1)
    _CACHE.clear()


@pytest.mark.parametrize("kind", ["shuf1000", "shuf50"])
def test_serial_sum_is_not_the_judge(kind):
    """The reference adds index-ascending in plain doubles: on shuffled molecules at 1M particles that sum is more than
    1e-10 relative off the exact dipole, so "GPU against the oracle at 1e-10" cannot be asserted on these inputs."""
    s, ph, t, D, S = system(kind, 1000001)
    serial = np.cumsum(t, axis=0)[-1]
    assert np.abs(serial - D).max() / np.abs(D[np.argmax(np.abs(serial - D))]) > 1e-10
