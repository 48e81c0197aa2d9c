"""The list-group harness step of tests/list_group_oracle.py (the thermostatted group as an index list, the way HOOMD's
ParticleGroup hands it out, composed from the C oracle's orc_bussi_step, orc_nve_step_w and orc_kinetic_energy) is
bit-identical to the window step orc_nvt_step_w when the list is a range."""
import os
import sys

import numpy as np
import pytest

from cav_hoomd_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from list_group_oracle import nvt_step_list  # noqa: E402


@pytest.mark.parametrize("first,n", [(0, 500), (100, 301), (0, 0)])
def test_list_step_with_a_range_is_the_window_step(coracle, first, n):
    s = synth.make_system(500, replica=12)
    mol = s.typeid != s.L_typeid
    s.vel[mol, :3] *= (s.box[0] / 6.0) / (np.abs(s.vel[mol, :3]).max() * synth.DT_1FS)  # many particles cross a face
    dof, dt, r, gm = 3.0 * max(n, 1) - 3.0, synth.DT_1FS, 0.7, 650.0
    idx = np.arange(first, first + n, dtype=np.uint32)
    f0 = coracle.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, 0.01, 1e-3)["force"]
    ke0 = coracle.kinetic_energy(s.vel, idx)
    arms = []
    for use_list in (False, True):
        p, v, im, f = s.pos.copy(), s.vel.copy(), s.image.copy(), f0.copy()
        ke, res = np.array([ke0]), np.zeros(2)
        out = []
        for _ in range(5):
            if use_list:
                out.append(nvt_step_list(coracle, p, v, s.charge, im, f, s.box, s.L_typeid, 0.01, 1e-3, 1.0, dt, idx, dof,
                                         synth.KT_100K, synth.TAU_5PS, r, gm, res, ke))
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
