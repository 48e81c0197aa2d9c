"""The thermostatted harness step with the cavity mode's Langevin bath (HOOMD's TwoStepLangevin on the photon, type 'L'),
restated in NumPy on top of the C oracle's pieces: orc_bussi_rescale_factor, orc_cavity_force, orc_find_photon and
orc_kinetic_energy.  It is orc_nvt_step_w (oracle/cavity_oracle.c) in the same operation order -- every product and
sum rounded on its own, as NumPy's element-wise float64 operations are -- with the bath added to the photon's kicks:

    step two at timestep t:  bd_c = coeff r_c - gamma v_c   (v: the photon's velocity BEFORE its second half kick)
                             coeff = sqrt(6 gamma kT / dt)  (left to right, as the library forms it on the host)
                             the photon kicks with f = (f_other + F_L) + bd
    step one at t + 1:       the photon kicks with the same bd (HOOMD keeps the sum as the acceleration); bd = 0
                             before the first step two

[HOOMD-upstream, not in the reference tree: TwoStepLangevin restated from its definition.]  tests/test_photon_bath.py
shows that with gamma = 0 and r = 0 it is bit-identical to orc_nvt_step_w."""
import ctypes as C
import math

import numpy as np


def langevin_coeff(gamma, kT, dt):
    return math.sqrt(6.0 * gamma * kT / dt)


def wrap(pos, image, box):
    """orc_wrap over all particles: one shift per direction into [-L/2, L/2), the image flag follows."""
    for c in range(3):
        L = float(box[c])
        hi = 0.5 * L
        x = pos[:, c]
        up = x >= hi
        dn = ~up & (x < -hi)
        x[up] = x[up] - L
        x[dn] = x[dn] + L
        image[up, c] += 1
        image[dn, c] -= 1


def find_photon(co, pos, L_typeid):
    p = np.ascontiguousarray(pos)
    return co.lib.orc_find_photon(p.ctypes.data_as(C.POINTER(C.c_double)), p.shape[0], L_typeid)


def nvt_step_bath(co, pos, vel, charge, image, force, box, L_typeid, omegac, couplstr, phmass, dt, idx, dof, kT,
                  tau, r_normal, gamma_draw, reservoir, ke_io, gamma, bath_kT, r, bd_io, wrap_box=True, force_other=None):
    """One step in place on pos / vel / image / force (the cavity force of the current positions); reservoir =
    float64[2], ke_io = float64[1] and bd_io = float64[3] (the photon's bath force, 0 before the first step) are updated
    in place.  force_other: float64[N, 4] added to the cavity force before the bath, or None.  idx: the thermostatted
    group as an index list (a range gives orc_nvt_step_w's window).  Returns (alpha, energies)."""
    idx = np.ascontiguousarray(idx, dtype=np.uint32)
    alpha = 1.0
    ke = float(ke_io[0])
    if len(idx) and dof != 0.0:
        if ke == 0.0:
            return math.nan, None
        alpha = co.bussi_rescale_factor(ke, dof, dt, kT, tau, r_normal, gamma_draw)
        delta = ke * (1.0 - alpha * alpha)
        reservoir[0] += delta
        reservoir[1] = delta
    ph = find_photon(co, pos, L_typeid)
    hm = (0.5 * dt) / vel[:, 3]

    def kick_force():
        f = force[:, :3].copy()
        if force_other is not None:
            f = force_other[:, :3] + f
        return f

    # step one: v <- alpha v (group), v += hm f, r += dt v
    f = kick_force()
    if ph >= 0:
        f[ph] = f[ph] + bd_io
    v = vel[:, :3].copy()
    v[idx] = v[idx] * alpha
    v = v + hm[:, None] * f
    vel[:, :3] = v
    pos[:, :3] = pos[:, :3] + dt * v
    if wrap_box:
        wrap(pos, image, box)
    res = co.cavity_force(pos, charge, image, box, L_typeid, omegac, couplstr, phmass)
    force[:] = res["force"]
    # step two: the bath force from the velocity before the kick, then v += hm f
    f = kick_force()
    if ph >= 0:
        coeff = langevin_coeff(gamma, bath_kT, dt)
        bd = coeff * np.asarray(r, dtype=np.float64) - gamma * vel[ph, :3]
        f[ph] = f[ph] + bd
        bd_io[:] = bd
    vel[:, :3] = vel[:, :3] + hm[:, None] * f
    ke_io[0] = co.kinetic_energy(vel, idx)
    return alpha, res["energies"]
