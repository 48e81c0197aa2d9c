"""Index-list groups and particle sorts on the fused integration path: the group mask of cavb200_group_set taken by the
ten window entry points (group_first = CAVB200_GROUP_MASK), cavb200_rank1_reindex after a permutation of the particle
arrays, and TwoStepConstantVolumeCavity with index_list_group = True driven through sorts of hoomd_shim's ParticleData."""
import os
import sys

import numpy as np
import pytest

from cav_hoomd_b200 import capi, rng, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from list_group_oracle import nvt_step_list  # noqa: E402

pytestmark = pytest.mark.gpu
BUILD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "plugin", "build")
OMEGAC, G, PHMASS = 0.01, 1e-8, 1.0  # weak coupling: the fast charges below would otherwise be thrown many box lengths
KT, TAU, DT = synth.KT_100K, synth.TAU_5PS, synth.DT_1FS
INVALID_VALUE, NOT_SUPPORTED = 1, 801  # cudaError_t


@pytest.fixture(scope="module")
def mods():
    sys.path.insert(0, BUILD)
    import _hoomd_shim  # noqa: F401  (registers ForceCompute / Thermostat bases first)
    import _bussi_reservoir
    import _cavitymd
    return _hoomd_shim, _cavitymd, _bussi_reservoir


def fast_system(n_mol, replica, photon="last"):
    """A particle travels ~L/6 per step: a large share of them crosses a face within a few steps."""
    s = synth.make_system(n_mol, replica=replica, photon=photon)
    mol = s.typeid != s.L_typeid
    s.vel[mol, :3] *= (s.box[0] / 6.0) / (np.abs(s.vel[mol, :3]).max() * DT)
    return s


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def run_path(h, s, path, wrap, first, n, steps, d_idx=None, st=None):
    """`steps` harness steps through one family of entry points; first == GROUP_MASK: the group is the mask built from
    d_idx.  Returns positions, velocities, images and the per-step (bussi_read, rank1_read) of the device."""
    p = capi.Params.make(OMEGAC, G, PHMASS)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    d_f = capi.DeviceArray((s.N, 4), np.float64)
    image, box = (d["image"], s.box) if wrap else (None, None)
    dof = 3.0 * n - 3.0
    draws = [capi.BussiArgs(KT, TAU, DT, dof, *rng.bussi_draws(t, 9, 0, dof)) for t in range(steps)]
    h.bussi_reset(st)
    if first == capi.Handle.GROUP_MASK:
        h.group_set(d_idx, n, s.N, st)
        h.bussi_ke(d["vel"], d_idx, 0, n, st)
    else:
        h.bussi_ke(d["vel"], None, first, n, st)
    hist = []

    def record():
        hist.append((h.bussi_read(st), h.rank1_read(st)))

    if path == "stored":
        h.force(d["pos"], d["charge"], d["image"], d_f, s.N, s.box, s.L_typeid, p, st)
        for t in range(steps):
            h.nvt_step_one(d["pos"], d["vel"], d_f, s.N, DT, first, n, draws[t], st, image=image, box=box)
            h.force(d["pos"], d["charge"], d["image"], d_f, s.N, s.box, s.L_typeid, p, st)
            h.nvt_step_two(d["vel"], d_f, s.N, DT, first, n, st)
            record()
    elif path == "rank1":
        h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p, st)
        for t in range(steps):
            h.nvt_step_one_rank1(d["pos"], d["vel"], None, d["charge"], s.N, DT, s.L_typeid, G, first, n, draws[t], st,
                                 image=image, box=box)
            h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p, st)
            h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], s.N, DT, s.L_typeid, G, first, n, st)
            record()
    else:  # md_step_one ; md_step_fused x (steps - 1) ; nvt_step_two_rank1
        h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p, st)
        h.md_step_one(d["pos"], d["vel"], None, d["charge"], d["image"], s.N, DT, s.box, s.L_typeid, p, first, n, draws[0],
                      st, wrap=wrap)
        record()
        for t in range(1, steps):
            h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], s.N, DT, s.box, s.L_typeid, p, first, n,
                            draws[t], st, wrap=wrap)
            record()
        h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], s.N, DT, s.L_typeid, G, first, n, st)
        record()
    return d["pos"].numpy(st), d["vel"].numpy(st), d["image"].numpy(st), hist


# ---- a mask that holds a range is the window, bit for bit ---------------------------------------------------------------
@pytest.mark.parametrize("path", ["stored", "rank1", "md"])
@pytest.mark.parametrize("wrap", [False, True])
@pytest.mark.parametrize("N", [300, 40000, 1048576])
def test_mask_of_a_range_is_the_window(N, wrap, path):
    s = fast_system(N - 1, replica=21)
    first, n = 5, N - 12  # a range that starts and ends inside a mask word
    h = capi.Handle(0)
    d_idx = capi.DeviceArray.from_numpy(np.arange(first, first + n, dtype=np.uint32))
    win = run_path(h, s, path, wrap, first, n, 3)
    msk = run_path(h, s, path, wrap, capi.Handle.GROUP_MASK, n, 3, d_idx)
    for a, b in zip(win[:3], msk[:3]):
        assert np.array_equal(a, b)
    if wrap:
        assert np.any(win[2] != s.image)
    for (bw, rw), (bm, rm) in zip(win[3], msk[3]):
        assert bw == bm
        assert all(np.array_equal(x, y) for x, y in zip(rw, rm))
    assert h.fault_count == 0
    h.close()


# ---- an index list with holes against the oracle's list step -------------------------------------------------------------
@pytest.mark.parametrize("path", ["stored", "rank1", "md"])
def test_index_list_matches_the_oracle(coracle, path):
    """Photon in the middle, about a tenth of the molecules left out of the group; six steps with the wrap against
    the oracle's list step (tests/list_group_oracle.py) with the same draws."""
    steps = 6
    s = fast_system(40000, replica=22, photon="middle")
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    idx = np.sort(np.random.default_rng(3).choice(mol, size=int(0.9 * len(mol)), replace=False)).astype(np.uint32)
    n = len(idx)
    h = capi.Handle(0)
    gp, gv, gi, hist = run_path(h, s, path, True, capi.Handle.GROUP_MASK, n, steps, capi.DeviceArray.from_numpy(idx))
    dof = 3.0 * n - 3.0
    pos, vel, image, force = s.pos.copy(), s.vel.copy(), s.image.copy(), np.zeros((s.N, 4))
    force[:] = coracle.cavity_force(pos, s.charge, image, s.box, s.L_typeid, OMEGAC, G, PHMASS)["force"]
    ke, res = np.array([coracle.kinetic_energy(vel, idx)]), np.zeros(2)
    for t in range(steps):
        r, gm = rng.bussi_draws(t, 9, 0, dof)
        nvt_step_list(coracle, pos, vel, s.charge, image, force, s.box, s.L_typeid, OMEGAC, G, PHMASS, DT, idx, dof, KT,
                      TAU, r, gm, res, ke)
    assert np.any(image != s.image, axis=1).sum() > 0.2 * s.N and np.array_equal(gi, image)
    assert _rel(gp[:, :3], pos[:, :3]) <= 1e-10 and _rel(gv[:, :3], vel[:, :3]) <= 1e-10
    b = hist[-1][0]
    assert abs(b["cumulative"] - res[0]) <= 1e-9 * abs(res[0])
    assert abs(b["ke"] - ke[0]) <= 1e-10 * ke[0]
    assert h.fault_count == 0
    h.close()


# ---- argument checks ----------------------------------------------------------------------------------------------------
def _code(fn, *a, **kw):
    try:
        fn(*a, **kw)
    except capi.CavbError as e:
        return e.code
    return 0


def test_group_and_reindex_argument_checks():
    s = synth.make_system(999)
    N = s.N
    h = capi.Handle(0)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "vel")}
    d_f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    M = capi.Handle.GROUP_MASK
    # the sentinel before any cavb200_group_set
    assert _code(h.nvt_step_one, d["pos"], d["vel"], d_f, N, DT, M, 10) == INVALID_VALUE
    assert _code(h.nvt_step_two, d["vel"], d_f, N, DT, M, 10) == INVALID_VALUE
    # an index >= N, an index listed twice
    assert _code(h.group_set, capi.DeviceArray.from_numpy(np.array([0, 3, N], np.uint32)), 3, N) == INVALID_VALUE
    assert _code(h.group_set, capi.DeviceArray.from_numpy(np.array([7, 2, 7], np.uint32)), 3, N) == INVALID_VALUE
    assert _code(h.nvt_step_one, d["pos"], d["vel"], d_f, N, DT, M, 3) == INVALID_VALUE  # a failed set leaves no mask
    # a valid mask: n_group and N must be the ones it was built for
    h.group_set(capi.DeviceArray.from_numpy(np.array([9, 1, 500, 998], np.uint32)), 4, N)
    h.nvt_step_one(d["pos"], d["vel"], d_f, N, DT, M, 4)
    h.nvt_step_two(d["vel"], d_f, N, DT, M, 4)
    assert _code(h.nvt_step_one, d["pos"], d["vel"], d_f, N, DT, M, 5) == INVALID_VALUE
    assert _code(h.nvt_step_two, d["vel"], d_f, N - 1, DT, M, 4) == INVALID_VALUE
    # the window entry points keep their own check
    assert _code(h.nvt_step_two, d["vel"], d_f, N, DT, 1, N) == INVALID_VALUE
    # re-index: one 'L' particle is found wherever it is; two are refused
    h.rank1_reindex(d["pos"], N, s.L_typeid)
    two = synth.make_system(999, photon="duplicated")
    assert (two.typeid == two.L_typeid).sum() == 2
    assert _code(h.rank1_reindex, capi.DeviceArray.from_numpy(two.pos), two.N, two.L_typeid) == NOT_SUPPORTED
    capi.sync()
    assert h.fault_count == 0
    h.close()


def test_reindex_moves_the_photon_of_the_last_rank1_result():
    """force_rank1, then a permutation that moves the photon: after the re-index the rank-1 net force of the permuted
    arrays is the permuted net force of the original ones, bit for bit."""
    s = synth.make_system(5000, photon="middle")
    p = capi.Params.make(OMEGAC, 1e-3, PHMASS)
    h = capi.Handle(0)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image")}
    h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p)
    net0 = capi.DeviceArray.from_numpy(np.zeros((s.N, 4)))
    h.net_force_add_rank1(net0, d["charge"], d["pos"], s.N, s.L_typeid, 1e-3)
    order = np.random.default_rng(8).permutation(s.N)
    ph = int(np.flatnonzero(s.typeid == s.L_typeid)[0])
    assert int(np.flatnonzero(order == ph)[0]) != ph
    dp = {"pos": capi.DeviceArray.from_numpy(s.pos[order]), "charge": capi.DeviceArray.from_numpy(s.charge[order])}
    h.rank1_reindex(dp["pos"], s.N, s.L_typeid)
    net1 = capi.DeviceArray.from_numpy(np.zeros((s.N, 4)))
    h.net_force_add_rank1(net1, dp["charge"], dp["pos"], s.N, s.L_typeid, 1e-3)
    f0, f1 = net0.numpy(), net1.numpy()
    assert np.any(f0[ph] != 0.0) and np.array_equal(f1, f0[order])
    h.close()


# ---- the integration method with particle sorts ---------------------------------------------------------------------------
def _sorted_run(mods, coracle, mode, members, index_list, n_mol, photon, sorts=(3, 6), steps=8):
    shim, cav, bus = mods
    s = fast_system(n_mol, replica=23, photon=photon)
    members = np.asarray(members, dtype=np.uint32)
    n = len(members)
    dof = 3.0 * n - 3.0
    exec_conf = shim.ExecutionConfiguration(True, 0)
    pd = shim.ParticleData(s.N, s.box[0], s.box[1], s.box[2], list(s.types), exec_conf)
    pd.setPositions(s.pos)
    pd.setVelocities(s.vel)
    pd.setCharges(s.charge)
    pd.setImages(s.image)
    sysdef = shim.SystemDefinition(pd, 7)
    group = shim.ParticleGroup(sysdef, [int(x) for x in members])
    group.setTranslationalDOF(dof)
    th = bus.BussiReservoirThermostat(shim.VariantConstant(KT), group, shim.ComputeThermo(sysdef, group), sysdef, TAU)
    fc = cav.CavityForceComputeGPU(sysdef, OMEGAC, G)
    method = cav.TwoStepConstantVolumeCavity(sysdef, group, th, fc, mode)
    assert method.index_list_group is False
    method.index_list_group = index_list
    method.setDeltaT(DT)
    draws = [rng.bussi_draws(t, 11, 0, dof) for t in range(steps)]
    perm = np.random.default_rng(17)
    fc.compute(0)
    pd.setNetForce(fc.getForces())
    for t in range(steps):
        if t in sorts:
            ph = int(np.flatnonzero(pd.getPositions()[:, 3].view(np.uint64) & 0xFFFFFFFF == s.L_typeid)[0])
            order = perm.permutation(s.N)
            while order[ph] == ph:
                order = perm.permutation(s.N)
            pd.sortParticles([int(o) for o in order])
        bus._inject_draws(list(draws[t]))
        method.integrateStepOne(t)
        fc.compute(t + 1)
        pd.setNetForce(fc.getForces())
        method.integrateStepTwo(t)
    method.flush()
    tags = np.asarray(pd.getTags())
    assert not np.array_equal(tags, np.arange(s.N))

    pos, vel, image, force = s.pos.copy(), s.vel.copy(), s.image.copy(), np.zeros((s.N, 4))
    force[:] = coracle.cavity_force(pos, s.charge, image, s.box, s.L_typeid, OMEGAC, G)["force"]
    ke, res = np.array([coracle.kinetic_energy(vel, members)]), np.zeros(2)
    for t in range(steps):
        _, en_ref = nvt_step_list(coracle, pos, vel, s.charge, image, force, s.box, s.L_typeid, OMEGAC, G, PHMASS, DT,
                                  members, dof, KT, TAU, draws[t][0], draws[t][1], res, ke)
    gp, gv, gi = pd.getPositions(), pd.getVelocities(), pd.getImages()
    pos, vel, image = pos[tags], vel[tags], image[tags]
    assert np.any(image != s.image[tags], axis=1).sum() > 0.2 * s.N and np.array_equal(gi, image)
    assert _rel(gp[:, :3], pos[:, :3]) <= 1e-10 and _rel(gv[:, :3], vel[:, :3]) <= 1e-10
    assert np.isclose(fc.getHarmonicEnergy(), en_ref[0], rtol=1e-10) and np.isclose(fc.getCouplingEnergy(), en_ref[1], rtol=1e-10)
    assert np.isclose(th.getReservoirEnergyTranslational(), res[0], rtol=1e-9, atol=1e-18)
    assert np.isclose(th.getInstantaneousReservoirTranslational(), res[1], rtol=1e-9, atol=1e-18)
    return method.getLaunchCount()


@pytest.mark.parametrize("mode", ["stored", "rank1", "one_launch"])
def test_method_with_an_index_list_group_through_sorts(mods, coracle, mode):
    n_mol, steps = 4000, 8
    s = fast_system(n_mol, replica=23, photon="middle")
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    members = np.sort(np.random.default_rng(4).choice(mol, size=int(0.9 * len(mol)), replace=False))
    launches = _sorted_run(mods, coracle, mode, members, True, n_mol, "middle", steps=steps)
    # as without sorts (tests/test_plugin_gpu.py), plus one mask build at the start and after each of the two sorts and,
    # in the rank-1 modes, one re-index after each sort
    base = {"stored": 1 + 2 * steps, "rank1": 1 + 2 * steps + steps + 1, "one_launch": 1 + steps + 1 + 1}[mode]
    assert launches == base + 3 + (0 if mode == "stored" else 2)


def test_method_rank1_all_particles_window_through_sorts(mods, coracle):
    """The group stays a contiguous range (all particles) and index_list_group stays False: the sorts still move the
    photon, and the rank-1 kicks follow it."""
    n_mol, steps = 4000, 8
    launches = _sorted_run(mods, coracle, "rank1", np.arange(n_mol + 1), False, n_mol, "middle", steps=steps)
    assert launches == 1 + 2 * steps + steps + 1 + 2
