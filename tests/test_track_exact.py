"""The tracker's field contract on the CPU (tests/track_inputs.py): the NumPy restatement of k_track_record against exact
Fractions, the C(t) bound against the 1e-10 tolerance it replaces, and mutants of the restatement -- a C(t) contracted
into fused multiply-adds, the photon's kinetic energy of the wrong particle, the dipole of the previous step -- that the
contract must reject."""
import math
from fractions import Fraction

import numpy as np
import pytest

import dipole_inputs as di
import track_inputs as ti
from cav_hoomd_b200 import synth

DT = synth.DT_1FS


def _ulp_err(x: float, exact: Fraction) -> float:
    return abs(Fraction(x) - exact) / Fraction(float(np.spacing(abs(float(exact)))))


def _vels(n, seed):
    rng = np.random.default_rng(seed)
    v = np.empty((n, 4))
    v[:, :3] = rng.standard_normal((n, 3)) * np.exp(rng.uniform(-30, 5, size=(n, 1)))
    v[:, 3] = rng.choice([1.0, di.MASS_MOL, 0.75, 3.0 ** 20], size=n)
    return v


# ---- 1. the restatement against Fractions --------------------------------------------------------------------------------
def test_photon_ke_within_gamma3_of_exact():
    for v in _vels(2000, 1):
        ke, exact = ti.photon_ke(v), ti.photon_ke_exact(v)
        assert abs(Fraction(ke) - exact) <= Fraction(ti.GAMMA3) * exact
        assert _ulp_err(ke, exact) <= 3


def test_autocorr_within_its_rounding_bound():
    rng = np.random.default_rng(2)
    for _ in range(2000):
        r, d = rng.standard_normal(3) * 1e3, rng.standard_normal(3) * 1e3
        if rng.random() < 0.5:  # cancelling terms
            d[2] = -(r[0] * d[0] + r[1] * d[1]) / r[2] * (1 + 1e-9 * rng.standard_normal())
        c, exact = ti.autocorr(r, d), ti.dot_exact(r, d)
        assert abs(Fraction(c) - exact) <= Fraction(ti.autocorr_rounding_bound(r, d))


def test_record_restatement_fields():
    s = ti.make_system(769, "middle")
    ph = di.photon_index(s)
    D, _ = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph)
    q = ti.photon_q(s.pos, s.image, s.box, ph)
    en = di.finalize(D, q, di.constants())[0]
    ref = D * (1 + 1e-3)
    bo = dict(ke=1.5, alpha=0.99, cumulative=-2e-5)
    r = ti.record(7, (en, D, ph), q, s.vel, ref, bo)
    assert r[0] == 7 and np.array_equal(r[1:4], D) and np.array_equal(r[4:7], q) and np.array_equal(r[7:10], en)
    assert r[10] == ti.autocorr(ref, D) and r[11] == ti.photon_ke(s.vel[ph]) and r[15] == ph
    assert list(r[12:15]) == [1.5, 0.99, -2e-5]
    # no thermostat handle; pending velocities; a shard whose rows start at global index 5000
    assert np.all(np.isnan(ti.record(7, (en, D, ph), q, s.vel, ref, None)[12:15]))
    rp = ti.record(7, (en, D, ph), q, s.vel, ref, bo, pending=True)
    assert np.isnan(rp[11]) and np.isnan(rp[12]) and rp[13] == 0.99 and rp[14] == -2e-5
    assert ti.record(7, (en, D, ph + 5000), q, s.vel, ref, bo, offset=5000)[11] == ti.photon_ke(s.vel[ph])
    assert ti.record(7, (en, D, ph + 5000), q, s.vel, ref, bo, offset=0)[11] == 0.0       # beyond the local rows
    assert ti.record(7, (en, D, 3), q, s.vel, ref, bo, offset=5000)[11] == 0.0            # below the local rows
    assert ti.same_bits(rp, rp.copy()) and not ti.same_bits(rp, r)


# ---- 2. the C(t) bound is far inside the old tolerance ------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["adj50", "water_blk50"])
@pytest.mark.parametrize("N", [769, 8193, 262145])
def test_autocorr_bound_beats_the_old_tolerance(kind, N):
    s0 = ti.make_system(N, "last", kind)
    ph = di.photon_index(s0)
    D0, S0 = di.exact_dipole(s0.pos, s0.charge, s0.image, s0.box, ph)
    pos = s0.pos.copy()
    pos[:, :3] += s0.vel[:, :3] * 5 * DT
    D, S = di.exact_dipole(pos, s0.charge, s0.image, s0.box, ph)
    bound = ti.autocorr_bound(D0, di.tolerance(D0, S0, N), D, di.tolerance(D, S, N))
    old = ti.OLD_TOL * float(np.abs(D0) @ S)  # tests/test_trackers_gpu.py: 1e-10 dot(|d0|, sum |q r|)
    assert bound * 10 <= old, (bound, old)


# ---- 3. mutants miss the contract -----------------------------------------------------------------------------------------
def test_fma_in_autocorr_is_caught():
    """On the dipoles of these systems a contracted C(t) differs from the kernel's order in some record: the bitwise
    contract of [10] rejects a kernel the compiler contracted."""
    differ = 0
    for N in (769, 8193):
        for seed in range(6):
            s = ti.make_system(N, "last", seed=seed)
            ph = di.photon_index(s)
            D0, _ = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph)
            for t in range(1, 6):
                pos = s.pos.copy()
                pos[:, :3] += s.vel[:, :3] * t * DT
                D, _ = di.exact_dipole(pos, s.charge, s.image, s.box, ph)
                differ += ti.autocorr(D0, D) != ti.autocorr_fma(D0, D)
    assert differ > 0


def test_wrong_photon_row_misses_its_bound():
    for where in ("last", "middle"):
        s = ti.make_system(8193, where)
        ph = di.photon_index(s)
        exact = ti.photon_ke_exact(s.vel[ph])
        for wrong in (ph - 1, 0, (ph + 1) % s.N):
            ke = ti.photon_ke(s.vel[wrong])
            assert abs(Fraction(ke) - exact) > Fraction(ti.GAMMA3) * exact


@pytest.mark.parametrize("kind", ["adj50", "water_blk50"])
@pytest.mark.parametrize("N", [769, 8193, 262145])
def test_dipole_of_the_previous_step_misses_its_bound(kind, N):
    """One femtosecond of thermal motion moves d by far more than its bound: a record of the previous step's d (or of
    another handle's) fails; C(t) formed from it fails its bound too."""
    s = ti.make_system(N, "last", kind)
    ph = di.photon_index(s)
    D_prev, S_prev = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph)
    pos = s.pos.copy()
    pos[:, :3] += s.vel[:, :3] * DT
    D, S = di.exact_dipole(pos, s.charge, s.image, s.box, ph)
    tol = di.tolerance(D, S, N)
    assert np.any(np.abs(D_prev - D) > tol)
    bound = ti.autocorr_bound(D_prev, di.tolerance(D_prev, S_prev, N), D, tol)
    exact = ti.dot_exact(D_prev, D)
    assert abs(Fraction(ti.autocorr(D_prev, D_prev)) - exact) > Fraction(bound)


def test_absent_photon_system_has_no_L():
    s = ti.make_system(769, "absent")
    assert di.photon_index(s) == -1 and math.isclose(float(s.charge.sum()), 0.0, abs_tol=1e-12)
