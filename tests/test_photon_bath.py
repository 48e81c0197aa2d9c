"""The cavity mode's Langevin bath in the CPU reference (tests/photon_bath_oracle.py): with a null bath it is the
oracle's thermostatted harness step bit for bit, with kT = 0 it drains the photon's energy, and with a free cavity mode
it gives each Cartesian component of the photon the bath temperature, in kinetic and in potential energy
(equipartition).  The last check is what pins the noise amplitude sqrt(6 gamma kT / dt) of uniform draws in [-1, 1]:
parity with the GPU cannot tell a wrong factor there."""
import os
import sys

import numpy as np
import pytest

from cav_hoomd_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from photon_bath_oracle import nvt_step_bath  # noqa: E402


def _fast(n_mol, replica, photon):
    s = synth.make_system(n_mol, replica=replica, photon=photon)
    mol = s.typeid != s.L_typeid
    s.vel[mol, :3] *= (s.box[0] / 6.0) / (np.abs(s.vel[mol, :3]).max() * synth.DT_1FS)  # many particles cross a face
    return s


@pytest.mark.parametrize("photon", ["last", "middle", "absent"])
@pytest.mark.parametrize("first,n", [(0, 500), (100, 301), (0, 0)])
def test_null_bath_is_the_oracle_step(coracle, photon, first, n):
    """gamma = 0, r = 0: every output of five steps equals orc_nvt_step_w's, bit for bit."""
    s = _fast(500, 13, photon)
    dof, dt, r, gm = 3.0 * max(n, 1) - 3.0, synth.DT_1FS, 0.7, 650.0
    f0 = coracle.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, 0.01, 1e-3)["force"]
    ke0 = coracle.kinetic_energy(s.vel, np.arange(first, first + n, dtype=np.uint32))
    arms = []
    for bath in (False, True):
        p, v, im, f = s.pos.copy(), s.vel.copy(), s.image.copy(), f0.copy()
        ke, res, bd = np.array([ke0]), np.zeros(2), np.zeros(3)
        out = []
        for _ in range(5):
            if bath:
                out.append(nvt_step_bath(coracle, p, v, s.charge, im, f, s.box, s.L_typeid, 0.01, 1e-3, 1.0, dt,
                                         np.arange(first, first + n), dof, synth.KT_100K, synth.TAU_5PS, r, gm, res, ke,
                                         0.0, synth.KT_100K, [0.0, 0.0, 0.0], bd))
            else:
                out.append(coracle.nvt_step(p, v, s.charge, im, f, s.box, s.L_typeid, 0.01, 1e-3, 1.0, dt, first, n, dof,
                                            synth.KT_100K, synth.TAU_5PS, r, gm, res, ke, wrap=True))
        arms.append((p, v, im, f, ke, res, out))
    (pa, va, ia, fa, ka, ra, oa), (pb, vb, ib, fb, kb, rb, ob) = arms
    assert np.any(ia != s.image)
    for x, y in ((pa, pb), (va, vb), (ia, ib), (fa, fb), (ka, kb), (ra, rb)):
        assert np.array_equal(x, y)
    for (alpha_a, en_a), (alpha_b, en_b) in zip(oa, ob):
        assert alpha_a == alpha_b and np.array_equal(en_a, en_b)


def _free_photon(v0=(0.0, 0.0, 0.0)):
    """One photon alone in a large box: with g = 0 it is a 3-D harmonic oscillator, K = phmass omegac^2."""
    pos = np.zeros((1, 4))
    pos[:, 3] = synth.typeid_to_w(np.array([synth.L_TYPEID]))
    vel = np.zeros((1, 4))
    vel[0, :3] = v0
    vel[0, 3] = 1.0  # mass
    return pos, vel, np.zeros(1), np.zeros((1, 3), dtype=np.int32), np.full(3, 1e6)


def _run_free(coracle, steps, gamma, kT, omegac, dt, draws, v0=(0.0, 0.0, 0.0)):
    pos, vel, charge, image, box = _free_photon(v0)
    force = coracle.cavity_force(pos, charge, image, box, synth.L_TYPEID, omegac, 0.0)["force"]
    ke, res, bd = np.zeros(1), np.zeros(2), np.zeros(3)
    q = np.empty((steps, 3))
    v = np.empty((steps, 3))
    for t in range(steps):
        nvt_step_bath(coracle, pos, vel, charge, image, force, box, synth.L_TYPEID, omegac, 0.0, 1.0, dt, [], 0.0, 0.0,
                      1.0, 0.0, 0.0, res, ke, gamma, kT, draws(t), bd)
        q[t] = pos[0, :3]
        v[t] = vel[0, :3]
    return q, v


def test_zero_temperature_bath_drains_the_photon(coracle):
    omegac, dt, gamma = 1.0, 0.05, 0.5
    q, v = _run_free(coracle, 400, gamma, 0.0, omegac, dt, lambda t: (0.7, -0.3, 0.9), v0=(1.0, -2.0, 0.5))
    e = 0.5 * (v ** 2).sum(axis=1) + 0.5 * omegac ** 2 * (q ** 2).sum(axis=1)
    ke = 0.5 * (v ** 2).sum(axis=1)
    assert e[-1] < 1e-3 * e[0]  # e^{-gamma t} of the energy, t = 20: ~5e-5
    assert ke[-100:].max() < 1e-3 * ke[0]
    assert np.all(np.diff(e[::20]) < 0.0)


def test_free_cavity_mode_equipartition(coracle):
    """10^5 steps of a free cavity mode (g = 0, omegac dt = 0.05) with uniform draws from NumPy: <m v_c^2> and
    <K q_c^2> of each component are the bath's kT.  Tolerance: 5 standard errors of the mean, estimated from 50 blocks
    of 2000 steps (a block is 100 friction times 1/gamma long, so the block means are independent), plus 1 % for the
    O((omegac dt)^2) bias of the discretisation; the standard error itself must be below 5 % of kT."""
    omegac, dt, gamma, kT = 1.0, 0.05, 1.0, 1.0
    steps, burn, blocks = 102000, 2000, 50
    u = np.random.default_rng(2024).uniform(-1.0, 1.0, size=(steps, 3))
    q, v = _run_free(coracle, steps, gamma, kT, omegac, dt, lambda t: u[t])
    K = 1.0 * omegac * omegac
    for name, x in (("m v^2", v[burn:] ** 2), ("K q^2", K * q[burn:] ** 2)):
        for c in range(3):
            b = x[:, c].reshape(blocks, -1).mean(axis=1)
            mean, sem = b.mean(), b.std(ddof=1) / np.sqrt(blocks)
            assert sem < 0.05 * kT, (name, c, sem)
            assert abs(mean - kT) <= 5.0 * sem + 0.01 * kT, (name, c, mean, sem)
    # a noise amplitude off by sqrt(3) (the Gaussian-draw coefficient sqrt(2 gamma kT / dt) used with uniform draws)
    # gives a third of kT: far outside the tolerance above
    q3, v3 = _run_free(coracle, 22000, gamma, kT, omegac, dt, lambda t: u[t] / np.sqrt(3.0))
    assert abs((v3[burn:] ** 2).mean() - kT / 3.0) < 0.1 * kT
