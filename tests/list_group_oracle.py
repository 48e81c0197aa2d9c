"""The thermostatted harness step with the group given as an index list (HOOMD's ParticleGroup index array), built
from the C oracle's own pieces: orc_bussi_step over the list (KE, alpha, reservoir bookkeeping, v <- alpha v),
orc_nve_step_w over all N (kick, drift, box wrap, cavity force, kick) and orc_kinetic_energy over the list.  This is
orc_nvt_step_w's sequence with [first, first + n) replaced by the list; tests/test_group_list.py shows that it is
bit-identical to orc_nvt_step_w when the list is a range."""
import numpy as np


def nvt_step_list(co, pos, vel, charge, image, force, box, L_typeid, omegac, couplstr, phmass, dt, idx, dof, kT, tau,
                  r_normal, gamma_draw, reservoir, ke_io, wrap=True):
    """One step in place on pos / vel / image / force; reservoir = float64[2], ke_io = float64[1] (1/2 sum m|v|^2 of the
    group, left by the previous step or by COracle.kinetic_energy) updated in place.  Returns (alpha, energies)."""
    idx = np.ascontiguousarray(idx, dtype=np.uint32)
    alpha = 1.0
    if len(idx) and dof != 0.0:
        alpha, ke = co.bussi_step(vel, idx, dof, dt, kT, tau, r_normal, gamma_draw, reservoir)
        assert ke == ke_io[0]  # the group's velocities have not changed since ke_io was summed
    en = co.nve_step(pos, vel, charge, image, force, box, L_typeid, omegac, couplstr, phmass, dt, wrap=wrap)
    ke_io[0] = co.kinetic_energy(vel, idx)
    return alpha, en
