"""The cavity mode's Langevin bath on the fused integration path: the four *_bath entry points against the CPU reference
of tests/photon_bath_oracle.py over 8 steps (the three-launch rank-1 step and md_step_one ; md_step_fused x 7 ;
step_two), the two paths against each other, the null bath and the photon-less system against the siblings bit for bit,
and the argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from cav_hoomd_b200 import capi, rng, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from photon_bath_oracle import nvt_step_bath  # noqa: E402

pytestmark = pytest.mark.gpu
OMEGAC, G, PHMASS = 0.01, 1e-8, 1.0  # weak coupling: the fast charges below would otherwise be thrown many box lengths
KT, TAU, DT = synth.KT_100K, synth.TAU_5PS, synth.DT_1FS
GAMMA = 1e-3  # the bath force is then of the order of F_L: a bath left out or misplaced is far outside the tolerances
STEPS = 8
INVALID_VALUE = 1


def fast_system(n_mol, replica, photon):
    s = synth.make_system(n_mol, replica=replica, photon=photon)
    mol = s.typeid != s.L_typeid
    s.vel[mol, :3] *= (s.box[0] / 6.0) / (np.abs(s.vel[mol, :3]).max() * DT)
    return s


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def group_of(s, kind):
    """window: every particle (the photon, wherever it sits, is then inside the group); mask: about a tenth of the
    molecules left out, the photon out."""
    if kind == "window":
        return np.arange(s.N, dtype=np.uint32)
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    keep = np.random.default_rng(5).random(len(mol)) >= 0.1
    return mol[keep].astype(np.uint32)


def draws_for(dof, steps=STEPS, gamma=GAMMA, seed=31):
    u = np.random.default_rng(seed).uniform(-1.0, 1.0, size=(steps, 3))
    bussi = [rng.bussi_draws(t, 9, 0, dof) for t in range(steps)]
    return bussi, [capi.LangevinArgs.make(gamma, KT, u[t]) for t in range(steps)]


def run_gpu(s, path, group, fo, bath, shape=0, steps=STEPS, bath_on=True):
    """`steps` steps on a fresh handle (its bath slot starts at 0).  path: "rank1" (nvt_step_one_rank1 ; force_rank1 ;
    nvt_step_two_rank1) or "md" (md_step_one ; md_step_fused x (steps - 1) ; nvt_step_two_rank1).  bath_on = False runs
    the siblings.  group: ("window", idx) or ("mask", idx).  Returns pos, vel, image, bussi_read, rank1_read."""
    kind, idx = group
    n = len(idx)
    dof = 3.0 * n - 3.0
    bussi, lang = bath
    h = capi.Handle(0)
    h.set_tuning(md_shape=shape)
    p = capi.Params.make(OMEGAC, G, PHMASS)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    d_fo = capi.DeviceArray.from_numpy(fo) if fo is not None else None
    if kind == "mask":
        d_idx = capi.DeviceArray.from_numpy(idx)
        h.group_set(d_idx, n, s.N)
        first = capi.Handle.GROUP_MASK
        h.bussi_ke(d["vel"], d_idx, 0, n)
    else:
        first = int(idx[0]) if n else 0
        h.bussi_ke(d["vel"], None, first, n)
    args = [capi.BussiArgs(KT, TAU, DT, dof, *bussi[t]) for t in range(steps)]
    lb = (lambda t: lang[t]) if bath_on else (lambda t: None)
    h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p)
    if path == "rank1":
        for t in range(steps):
            h.nvt_step_one_rank1(d["pos"], d["vel"], d_fo, d["charge"], s.N, DT, s.L_typeid, G, first, n, args[t],
                                 image=d["image"], box=s.box, bath=bath_on)
            h.force_rank1(d["pos"], d["charge"], d["image"], s.N, s.box, s.L_typeid, p)
            h.nvt_step_two_rank1(d["vel"], d_fo, d["charge"], d["pos"], s.N, DT, s.L_typeid, G, first, n, bath=lb(t))
    else:
        h.md_step_one(d["pos"], d["vel"], d_fo, d["charge"], d["image"], s.N, DT, s.box, s.L_typeid, p, first, n, args[0],
                      wrap=True, bath=bath_on)
        for t in range(1, steps):
            h.md_step_fused(d["pos"], d["vel"], d_fo, d["charge"], d["image"], s.N, DT, s.box, s.L_typeid, p, first, n,
                            args[t], wrap=True, bath=lb(t - 1))
        h.nvt_step_two_rank1(d["vel"], d_fo, d["charge"], d["pos"], s.N, DT, s.L_typeid, G, first, n, bath=lb(steps - 1))
    out = (d["pos"].numpy(), d["vel"].numpy(), d["image"].numpy(), h.bussi_read(), h.rank1_read())
    assert h.fault_count == 0
    h.close()
    return out


def run_oracle(co, s, idx, fo, bath, gamma_scale=1.0, steps=STEPS):
    bussi, lang = bath
    dof = 3.0 * len(idx) - 3.0
    pos, vel, image = s.pos.copy(), s.vel.copy(), s.image.copy()
    force = co.cavity_force(pos, s.charge, image, s.box, s.L_typeid, OMEGAC, G, PHMASS)["force"].copy()
    ke, res, bd = np.array([co.kinetic_energy(vel, idx)]), np.zeros(2), np.zeros(3)
    for t in range(steps):
        nvt_step_bath(co, pos, vel, s.charge, image, force, s.box, s.L_typeid, OMEGAC, G, PHMASS, DT, idx, dof, KT, TAU,
                      bussi[t][0], bussi[t][1], res, ke, lang[t].gamma * gamma_scale, lang[t].kT, list(lang[t].r), bd,
                      force_other=fo)
    return pos, vel, image, res, ke, force


def other_forces(s, seed=6):
    """A stand-in for the pair forces: random, of the order of the cavity force on the photon."""
    fo = np.random.default_rng(seed).normal(scale=1e-3, size=(s.N, 4))
    fo[:, 3] = 0.0
    return fo


# ---- parity with the CPU reference -------------------------------------------------------------------------------------
GRID = [(path, shape) for path in ("rank1", "md") for shape in ((0, 1) if path == "md" else (0,))]


@pytest.mark.parametrize("path,shape", GRID)
@pytest.mark.parametrize("n_mol", [1, 300, 20000, 200000])
@pytest.mark.parametrize("other", [False, True])
@pytest.mark.parametrize("kind", ["window", "mask"])
@pytest.mark.parametrize("photon", ["last", "middle", "absent"])
def test_bath_matches_the_oracle(coracle, photon, kind, other, n_mol, path, shape):
    s = fast_system(n_mol, replica=41, photon=photon)
    idx = group_of(s, kind)
    fo = other_forces(s) if other else None
    bath = draws_for(3.0 * len(idx) - 3.0)
    gp, gv, gi, b, (_, FL, ph, _) = run_gpu(s, path, (kind, idx), fo, bath, shape)
    pos, vel, image, res, ke, force = run_oracle(coracle, s, idx, fo, bath)
    if n_mol >= 300:
        assert np.any(image != s.image, axis=1).sum() > 0.2 * s.N
    assert np.array_equal(gi, image)
    assert _rel(gp[:, :3], pos[:, :3]) <= 1e-10 and _rel(gv[:, :3], vel[:, :3]) <= 1e-10
    assert abs(b["ke"] - ke[0]) <= 1e-10 * max(ke[0], 1e-300)
    assert abs(b["cumulative"] - res[0]) <= 1e-9 * abs(res[0]) + 1e-18
    if photon != "absent":
        p = int(np.flatnonzero(s.typeid == s.L_typeid)[0])
        assert ph == p and _rel(np.asarray(FL), force[p, :3]) <= 1e-10
        # the photon on its own scale, and the bath visibly in it: the same run without the bath is far off
        assert _rel(gv[p, :3], vel[p, :3]) <= 1e-10 and _rel(gp[p, :3], pos[p, :3]) <= 1e-10
        _, vel0, _, _, _, _ = run_oracle(coracle, s, idx, fo, bath, gamma_scale=0.0)
        assert _rel(vel0[p, :3], vel[p, :3]) > 1e-6


@pytest.mark.parametrize("n_mol", [300, 20000, 200000])
@pytest.mark.parametrize("photon", ["last", "middle"])
def test_fused_path_is_the_three_launch_path(photon, n_mol):
    s = fast_system(n_mol, replica=42, photon=photon)
    idx = group_of(s, "mask")
    fo = other_forces(s)
    bath = draws_for(3.0 * len(idx) - 3.0)
    a = run_gpu(s, "rank1", ("mask", idx), fo, bath)
    for shape in (0, 1):
        m = run_gpu(s, "md", ("mask", idx), fo, bath, shape)
        assert np.array_equal(a[2], m[2])
        assert _rel(m[0][:, :3], a[0][:, :3]) <= 1e-13 and _rel(m[1][:, :3], a[1][:, :3]) <= 1e-13
        p = int(np.flatnonzero(s.typeid == s.L_typeid)[0])
        assert _rel(m[1][p, :3], a[1][p, :3]) <= 1e-13
        assert abs(m[3]["ke"] - a[3]["ke"]) <= 1e-13 * a[3]["ke"]


# ---- the null bath and the photon-less system are the siblings, bit for bit ---------------------------------------------
@pytest.mark.parametrize("path,shape", GRID)
@pytest.mark.parametrize("case", ["null_bath", "no_photon"])
def test_bath_entry_points_reduce_to_their_siblings(case, path, shape):
    s = fast_system(20000, replica=43, photon="absent" if case == "no_photon" else "middle")
    idx = group_of(s, "window")
    fo = other_forces(s)
    bath = draws_for(3.0 * len(idx) - 3.0)
    if case == "null_bath":
        bath = (bath[0], [capi.LangevinArgs.make(0.0, KT, (0.0, 0.0, 0.0)) for _ in bath[1]])
    a = run_gpu(s, path, ("window", idx), fo, bath, shape, bath_on=False)
    b = run_gpu(s, path, ("window", idx), fo, bath, shape, bath_on=True)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)
    assert a[3] == b[3]
    assert all(np.array_equal(x, y) for x, y in zip(a[4], b[4]))


# ---- argument checks ---------------------------------------------------------------------------------------------------
def _code(fn, *a):
    return fn(*a)


def test_bath_argument_checks():
    s = synth.make_system(999)
    N = s.N
    h = capi.Handle(0)
    lib = h.lib
    p = capi.Params.make(OMEGAC, G, PHMASS)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    P = {k: capi._ptr(v) for k, v in d.items()}
    h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, p)
    ok = capi.LangevinArgs.make(GAMMA, KT, (0.1, 0.2, 0.3))
    L = s.L_typeid

    def two(bath, dt=DT):
        return lib.cavb200_nvt_step_two_rank1_bath(h.h, P["vel"], None, P["charge"], P["pos"], N, dt, L, G, 0, N, bath,
                                                   None)

    def fused(bath, dt=DT):
        return lib.cavb200_md_step_fused_wrap_bath(h.h, P["pos"], P["vel"], None, P["charge"], P["image"], N, dt,
                                                   s.box[0], s.box[1], s.box[2], L, C.byref(p), 0, N, None, bath, None)

    launches = h.launch_count
    for fn in (two, fused):
        assert fn(None) == INVALID_VALUE
        assert fn(C.byref(capi.LangevinArgs.make(-1e-3, KT, (0, 0, 0)))) == INVALID_VALUE
        assert fn(C.byref(capi.LangevinArgs.make(GAMMA, -KT, (0, 0, 0)))) == INVALID_VALUE
        assert fn(C.byref(ok), 0.0) == INVALID_VALUE
    assert h.launch_count == launches
    assert lib.cavb200_nvt_step_two_rank1_bath(None, P["vel"], None, P["charge"], P["pos"], N, DT, L, G, 0, N,
                                               C.byref(ok), None) == INVALID_VALUE
    # N == 0 is a no-op, as for every entry point
    assert lib.cavb200_nvt_step_two_rank1_bath(h.h, P["vel"], None, P["charge"], P["pos"], 0, DT, L, G, 0, 0, None,
                                               None) == 0
    # valid calls launch one kernel each
    assert two(C.byref(ok)) == 0
    assert lib.cavb200_nvt_step_one_rank1_wrap_bath(h.h, P["pos"], P["vel"], None, P["charge"], P["image"], N, DT,
                                                    s.box[0], s.box[1], s.box[2], L, G, 0, N, None, None) == 0
    assert lib.cavb200_md_step_one_wrap_bath(h.h, P["pos"], P["vel"], None, P["charge"], P["image"], N, DT, s.box[0],
                                             s.box[1], s.box[2], L, C.byref(p), 0, N, None, None) == 0
    assert fused(C.byref(ok)) == 0
    assert h.launch_count == launches + 4
    # the wrappers: the bath comes with the wrapped steps only
    with pytest.raises(ValueError):
        h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, L, p, 0, N, bath=ok)
    capi.sync()
    assert h.fault_count == 0
    h.close()


# ---- the integration method: TwoStepConstantVolumeCavity.setPhotonBath ----------------------------------------------------
BUILD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "plugin", "build")


@pytest.fixture(scope="module")
def mods():
    sys.path.insert(0, BUILD)
    import _hoomd_shim  # noqa: F401  (registers ForceCompute / Thermostat bases first)
    import _bussi_reservoir
    import _cavitymd
    return _hoomd_shim, _cavitymd, _bussi_reservoir


def _method(mods, s, mode, members):
    shim, cav, bus = mods
    exec_conf = shim.ExecutionConfiguration(True, 0)
    pd = shim.ParticleData(s.N, s.box[0], s.box[1], s.box[2], list(s.types), exec_conf)
    pd.setPositions(s.pos)
    pd.setVelocities(s.vel)
    pd.setCharges(s.charge)
    pd.setImages(s.image)
    sysdef = shim.SystemDefinition(pd, 7)
    group = shim.ParticleGroup(sysdef, [int(x) for x in members])
    group.setTranslationalDOF(3.0 * len(members) - 3.0)
    th = bus.BussiReservoirThermostat(shim.VariantConstant(KT), group, shim.ComputeThermo(sysdef, group), sysdef, TAU)
    fc = cav.CavityForceComputeGPU(sysdef, OMEGAC, G)
    method = cav.TwoStepConstantVolumeCavity(sysdef, group, th, fc, mode)
    method.index_list_group = True
    method.setDeltaT(DT)
    return pd, sysdef, group, th, fc, method


@pytest.mark.parametrize("mode", ["rank1", "one_launch"])
def test_method_with_the_photon_bath_through_sorts(mods, coracle, mode):
    """The method with a photon bath, driven with injected draws through two particle sorts that move the photon and
    through flush(), against the CPU reference; the photon in the middle, a tenth of the molecules out of the group."""
    shim, cav, bus = mods
    steps, sorts = 8, (3, 6)
    s = fast_system(4000, replica=44, photon="middle")
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    members = np.sort(np.random.default_rng(4).choice(mol, size=int(0.9 * len(mol)), replace=False)).astype(np.uint32)
    ph = int(np.flatnonzero(s.typeid == s.L_typeid)[0])
    dof = 3.0 * len(members) - 3.0
    pd, sysdef, group, th, fc, method = _method(mods, s, mode, members)
    photon = shim.ParticleGroup(sysdef, [ph])
    method.setPhotonBath(photon, shim.VariantConstant(KT), GAMMA)
    assert method.photon_bath
    bussi = [rng.bussi_draws(t, 11, 0, dof) for t in range(steps)]
    u = np.random.default_rng(45).uniform(-1.0, 1.0, size=(steps, 3))
    perm = np.random.default_rng(17)
    fc.compute(0)
    pd.setNetForce(fc.getForces())
    for t in range(steps):
        if t in sorts:
            cur = int(np.flatnonzero(pd.getPositions()[:, 3].view(np.uint64) & 0xFFFFFFFF == s.L_typeid)[0])
            order = perm.permutation(s.N)
            while order[cur] == cur:
                order = perm.permutation(s.N)
            pd.sortParticles([int(o) for o in order])
        bus._inject_draws(list(bussi[t]))
        method.integrateStepOne(t)
        fc.compute(t + 1)
        pd.setNetForce(fc.getForces())
        cav._inject_draws(list(u[t]))
        method.integrateStepTwo(t)
    method.flush()
    tags = np.asarray(pd.getTags())
    assert not np.array_equal(tags, np.arange(s.N))

    pos, vel, image = s.pos.copy(), s.vel.copy(), s.image.copy()
    force = coracle.cavity_force(pos, s.charge, image, s.box, s.L_typeid, OMEGAC, G)["force"].copy()
    ke, res, bd = np.array([coracle.kinetic_energy(vel, members)]), np.zeros(2), np.zeros(3)
    for t in range(steps):
        nvt_step_bath(coracle, pos, vel, s.charge, image, force, s.box, s.L_typeid, OMEGAC, G, PHMASS, DT, members, dof,
                      KT, TAU, bussi[t][0], bussi[t][1], res, ke, GAMMA, KT, u[t], bd)
    gp, gv, gi = pd.getPositions(), pd.getVelocities(), pd.getImages()
    pos, vel, image = pos[tags], vel[tags], image[tags]
    assert np.any(image != s.image[tags], axis=1).sum() > 0.2 * s.N and np.array_equal(gi, image)
    assert _rel(gp[:, :3], pos[:, :3]) <= 1e-10 and _rel(gv[:, :3], vel[:, :3]) <= 1e-10
    p = int(np.flatnonzero(tags == ph)[0])
    assert _rel(gv[p, :3], vel[p, :3]) <= 1e-10
    assert np.isclose(th.getReservoirEnergyTranslational(), res[0], rtol=1e-9, atol=1e-18)
    # launches as without the bath (tests/test_group_list_gpu.py): the bath rides in the same kernels
    base = {"rank1": 1 + 2 * steps + steps + 1, "one_launch": 1 + steps + 1 + 1}[mode]
    assert method.getLaunchCount() == base + 3 + 2


def test_method_photon_bath_refusals(mods):
    shim, cav, bus = mods
    s = fast_system(300, replica=46, photon="middle")
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    ph = int(np.flatnonzero(s.typeid == s.L_typeid)[0])
    pd, sysdef, group, th, fc, method = _method(mods, s, "stored", mol)
    kT = shim.VariantConstant(KT)
    with pytest.raises(ValueError, match="mode"):
        method.setPhotonBath(shim.ParticleGroup(sysdef, [ph]), kT, GAMMA)
    for mode in ("rank1", "one_launch"):
        pd, sysdef, group, th, fc, method = _method(mods, s, mode, mol)
        with pytest.raises(ValueError, match="exactly one"):
            method.setPhotonBath(shim.ParticleGroup(sysdef, [ph, int(mol[0])]), kT, GAMMA)
        with pytest.raises(ValueError, match="type 'L'"):
            method.setPhotonBath(shim.ParticleGroup(sysdef, [int(mol[3])]), kT, GAMMA)
        with pytest.raises(ValueError, match="gamma"):
            method.setPhotonBath(shim.ParticleGroup(sysdef, [ph]), kT, -1e-3)
        with pytest.raises(ValueError, match="kT"):
            method.setPhotonBath(shim.ParticleGroup(sysdef, [ph]), shim.VariantConstant(-KT), GAMMA)
        assert not method.photon_bath
        # the photon inside the thermostatted group
        pd, sysdef, group, th, fc, method = _method(mods, s, mode, np.arange(s.N))
        with pytest.raises(ValueError, match="thermostatted group"):
            method.setPhotonBath(shim.ParticleGroup(sysdef, [ph]), kT, GAMMA)
        method.clearPhotonBath()
        assert not method.photon_bath
