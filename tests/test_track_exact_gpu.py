"""The scalar tracker (cavb200_track_record / _record_from) after every entry point that leaves results on a handle, each
record held to the field contract of tests/track_inputs.py: bit for bit the values read back right after that step
(force_read, bussi_read, the photon's row of the velocities, C(t) in the kernel's order), and within stated bounds of the
exact dipole, the exact D(ref) . D(t), the exact photon kinetic energy and math.fsum of the group's kinetic energy.

Inputs are neutral molecules (dipole_inputs.make_molecules), where d cancels heavily: a record of the wrong step or of
the wrong handle misses by far more than the bounds.  Then the ring (capacity, wrap, read(0), read(k), re-open), stream
order (pdl on and off, a CUDA graph), and the plugin classes through hoomd_shim: the drop-in force with the Bussi
thermostat, and TwoStepConstantVolumeCavity in every mode, with the photon bath and through particle sorts."""
import functools
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

import dipole_inputs as di
import track_inputs as ti
from cav_hoomd_b200 import capi, rng, synth

pytestmark = pytest.mark.gpu
C = di.constants()
PARAMS = capi.Params.make(di.OMEGAC, di.G, di.PHMASS)
KT, TAU, DT = synth.KT_100K, synth.TAU_5PS, synth.DT_1FS
PENDING = capi.Handle.TRACK_VELOCITIES_PENDING
BUILD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "plugin", "build")


@functools.lru_cache(maxsize=None)
def system(N, photon, kind="adj50"):
    return ti.make_system(N, photon, kind)


def upload(s, keys=("pos", "charge", "image", "vel")):
    return {k: capi.DeviceArray.from_numpy(np.ascontiguousarray(getattr(s, k))) for k in keys}


def bussi_args(t, n, seed=5):
    dof = max(3.0 * n - 3.0, 3.0)
    return capi.BussiArgs(KT, TAU, DT, dof, *rng.bussi_draws(t, seed, 0, dof))


class Expect:
    """What one record must hold, gathered right after the step it records."""

    def __init__(self, h, t, d, s, bussi_h="self", group=None, offset=0, pending=False, force_h=None):
        fh = force_h or h
        self.t = t
        self.force = fh.force_read()
        self.bussi = None if bussi_h is None else (h if bussi_h == "self" else bussi_h).bussi_read()
        self.pos, self.image, self.vel = d["pos"].numpy(), d["image"].numpy(), d["vel"].numpy()
        self.charge, self.box = s.charge, s.box
        self.group, self.offset, self.pending = group, offset, pending

    @property
    def ph_local(self):
        ph = self.force[2]
        return ph - self.offset if ph >= 0 else -1

    def exact(self):
        """-> (D, tol) of the arrays this step left."""
        D, S = di.exact_dipole(self.pos, self.charge, self.image, self.box, self.ph_local)
        return D, di.tolerance(D, S, len(self.charge))


def check(row, e: Expect, ref_d, ref_exact=None, photon_expected=None):
    """row against the contract: bit for bit the restatement on what was read back, and the exact bounds.  ref_d: the
    stored reference (the d recorded when it was taken); ref_exact: its (D0, tol0)."""
    ph = e.force[2]
    if photon_expected is not None:
        assert ph == photon_expected, (ph, photon_expected)
    q = ti.photon_q(e.pos, e.image, e.box, e.ph_local)
    want = ti.record(e.t, e.force, q, e.vel, ref_d, e.bussi, e.offset, e.pending)
    assert ti.same_bits(row, want), (e.t, row, want)
    if ph < 0:
        assert np.all(row[1:12] == 0.0) or (e.pending and np.all(row[1:11] == 0.0) and np.isnan(row[11]))
        return
    d = row[1:4]
    D, tol = e.exact()
    assert np.all(np.abs(d - D) <= tol), (e.t, d - D, tol)
    assert ti.same_bits(row[7:10], di.finalize(d, q, C)[0])  # [4..6] is the q the energies were formed from
    if ref_exact is not None:
        D0, tol0 = ref_exact
        assert abs(Fraction(row[10]) - ti.dot_exact(D0, D)) <= Fraction(ti.autocorr_bound(D0, tol0, D, tol))
    assert abs(Fraction(row[10]) - ti.dot_exact(ref_d, d)) <= Fraction(ti.autocorr_rounding_bound(ref_d, d))
    if not e.pending:
        ke = ti.photon_ke_exact(e.vel[e.ph_local])
        assert abs(Fraction(row[11]) - ke) <= Fraction(ti.GAMMA3) * ke
        if e.group is not None and e.bussi is not None:
            KE = ti.group_ke_exact(e.vel, e.group)
            assert abs(row[12] - KE) <= ti.group_ke_bound(KE, len(e.group)), (row[12], KE)


def take_reference(h, s, d, offset=0):
    """track_set_reference and what it stored: (the d of the handle's last result, the exact D0 and its bound).  offset:
    the global index of the arrays' row 0."""
    h.track_set_reference()
    _, d0, ph = h.force_read()
    if ph < 0:
        return d0, None
    pos, image = d["pos"].numpy(), d["image"].numpy()
    D0, S0 = di.exact_dipole(pos, s.charge, image, s.box, ph - offset)
    return d0, (D0, di.tolerance(D0, S0, s.N))


# ---- 1. force-side calls under every schedule ---------------------------------------------------------------------------
FORCE_CASES = [("k_small", 2, {}), ("k_small", 768, {}), ("k_cluster", 769, {}), ("k_cluster", 8192, {}),
               ("k_split", 8193, dict(variant=2)), ("k_split_folder", 8193, {}), ("k_split", 262145, dict(variant=2)),
               ("k_split_folder", 262145, {}), ("k_split_folder", 1048577, {})]


@pytest.mark.parametrize("call", ["force", "step", "force_rank1"])
@pytest.mark.parametrize("sched,N,tuning", FORCE_CASES, ids=[f"{c[0]}-{c[1]}" for c in FORCE_CASES])
def test_force_side_calls(call, sched, N, tuning):
    """nve_kick_drift moves the particles, then the call reduces the dipole; one record per step."""
    s = system(N, "last")
    h = capi.Handle(0)
    if tuning:
        h.set_tuning(**tuning)
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    h.track_open(8)
    h.bussi_reset()

    def run(t):
        if call == "force":
            h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
        elif call == "step":
            h.step(d["pos"], d["charge"], d["image"], f, d["vel"], N, s.box, s.L_typeid, PARAMS, 0, N - 1,
                   bussi_args(t, N - 1))
        else:
            h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, PARAMS)

    run(0)
    ref = take_reference(h, s, d)
    want = []
    for t in range(1, 4):
        h.nve_kick_drift(d["pos"], d["vel"], f, N, DT)
        run(t)
        h.track_record(t, d["vel"], N)
        want.append(Expect(h, t, d, s))  # (cavb200_step publishes the KE of the velocities before its rescale)
    rec, total = h.track_read(8)
    assert total == 3 and len(rec) == 3
    for row, e in zip(rec, want):
        check(row, e, *ref, photon_expected=N - 1)
    assert h.fault_count == 0
    h.close()


# ---- 2. harness steps ---------------------------------------------------------------------------------------------------
def run_harness(h, s, path, wrap, group, steps=3, bath=False, record_pending=True):
    """The documented sequences with a record after every step.  path: stored (nvt_step_one ; force ; nvt_step_two),
    rank1 (nvt_step_one_rank1 ; force_rank1 ; nvt_step_two_rank1), md_one (md_step_one ; nvt_step_two_rank1), fused
    (md_step_one ; md_step_fused x (steps - 1) ; nvt_step_two_rank1: records between fused steps carry the pending
    flag).  Returns (records, expectations, reference)."""
    N = s.N
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    ph0 = di.photon_index(s)
    mol = np.flatnonzero(s.typeid != s.L_typeid).astype(np.uint32)
    if group == "window":
        first, n, d_idx, idx = 0, N - 1 if ph0 == N - 1 else N, None, np.arange(N - 1 if ph0 == N - 1 else N)
    else:
        idx = mol[::2] if len(mol) > 2 else mol
        d_idx = capi.DeviceArray.from_numpy(idx)
        first, n = capi.Handle.GROUP_MASK, len(idx)
        h.group_set(d_idx, n, N)
    image, box = (d["image"], s.box) if wrap else (None, None)
    lang = (lambda t: capi.LangevinArgs.make(0.5, KT, np.random.default_rng(t).uniform(-1, 1, 3))) if bath else (lambda t: None)
    h.track_open(16)
    h.bussi_reset()
    if path == "stored":
        h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
    else:
        h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, PARAMS)
    h.bussi_ke(d["vel"], d_idx, 0 if d_idx is not None else first, n)
    ref = take_reference(h, s, d)
    want = []

    def rec(t, pending=False):
        if pending:
            h.track_record_from(h, h, t, d["vel"], N, PENDING)
        else:
            h.track_record(t, d["vel"], N)
        want.append(Expect(h, t, d, s, group=idx, pending=pending))

    for t in range(1, steps + 1):
        a = bussi_args(t, n)
        if path == "stored":
            h.nvt_step_one(d["pos"], d["vel"], f, N, DT, first, n, a, image=image, box=box)
            h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
            h.nvt_step_two(d["vel"], f, N, DT, first, n)
            rec(t)
        elif path == "rank1":
            h.nvt_step_one_rank1(d["pos"], d["vel"], None, d["charge"], N, DT, s.L_typeid, di.G, first, n, a,
                                 image=image, box=box, bath=bath and t > 1)
            h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, PARAMS)
            h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], N, DT, s.L_typeid, di.G, first, n, bath=lang(t))
            rec(t)
        elif path == "md_one":
            h.md_step_one(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS, first, n,
                          a, wrap=wrap, bath=bath and t > 1)
            h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], N, DT, s.L_typeid, di.G, first, n, bath=lang(t))
            rec(t)
        else:
            if t == 1:
                h.md_step_one(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS, first,
                              n, a, wrap=wrap)
            else:
                h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS,
                                first, n, a, wrap=wrap, bath=lang(t - 1))
            if record_pending:
                rec(t, pending=True)
    if path == "fused":
        h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], N, DT, s.L_typeid, di.G, first, n, bath=lang(steps))
        rec(steps + 1)
    got, total = h.track_read(16)
    assert total == len(want) and h.fault_count == 0
    return got, want, ref


HARNESS = [(path, wrap, group, photon, N) for N in (769, 8193) for path in ("stored", "rank1", "md_one", "fused")
           for wrap in (False, True) for group in ("window", "mask") for photon in ("last", "middle", "absent")]
HARNESS += [(path, True, group, "middle", N) for N in (2, 262145, 1048577) for path in ("stored", "rank1", "md_one", "fused")
            for group in ("window", "mask") if not (N == 2 and group == "mask")]


@pytest.mark.parametrize("path,wrap,group,photon,N", HARNESS, ids=["-".join(map(str, c)) for c in HARNESS])
def test_harness_steps(path, wrap, group, photon, N):
    s = system(N, photon)
    h = capi.Handle(0)
    got, want, ref = run_harness(h, s, path, wrap, group)
    for row, e in zip(got, want):
        check(row, e, *ref, photon_expected=di.photon_index(s))
    h.close()


@pytest.mark.parametrize("path", ["rank1", "md_one", "fused"])
@pytest.mark.parametrize("photon", ["last", "middle"])
@pytest.mark.parametrize("md_shape", [0, 1])
def test_harness_steps_with_the_photon_bath(path, photon, md_shape):
    if md_shape and path != "fused":
        pytest.skip("md_shape shapes the fused step only")
    s = system(8193, photon)
    h = capi.Handle(0)
    h.set_tuning(md_shape=md_shape)
    got, want, ref = run_harness(h, s, path, True, "mask", steps=4, bath=True)
    for row, e in zip(got, want):
        check(row, e, *ref, photon_expected=di.photon_index(s))
    h.close()


# ---- 3. the sharded step on one device ------------------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0, 5000, 100000])
@pytest.mark.parametrize("photon", ["last", "middle", "absent"])
@pytest.mark.parametrize("N", [8193, 262145])
def test_shard_step_photon_row(offset, photon, N):
    """[15] is the global index offset + local row; [11] reads the local row.  With offset 5000 and the photon at local
    row 3072 of 8193, the global index 8072 is itself a row of the local array: a tracker that indexes the local array
    with the global index reads a molecule there."""
    s = system(N, photon)
    h = capi.Handle(0)
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    h.track_open(4)
    h.bussi_reset()
    n = N - 1
    h.shard_step(d["pos"], d["charge"], d["image"], f, d["vel"], N, offset, s.box, s.L_typeid, PARAMS, 0, n, bussi_args(0, n))
    ref = take_reference(h, s, d, offset)
    want = []
    for t in range(1, 3):
        h.nve_kick_drift(d["pos"], d["vel"], f, N, DT)
        h.shard_step(d["pos"], d["charge"], d["image"], f, d["vel"], N, offset, s.box, s.L_typeid, PARAMS, 0, n,
                     bussi_args(t, n))
        h.track_record(t, d["vel"], N)
        want.append(Expect(h, t, d, s, offset=offset))
    got, total = h.track_read(4)
    ph = di.photon_index(s)
    for row, e in zip(got, want):
        check(row, e, *ref, photon_expected=ph + offset if ph >= 0 else -1)
        if ph >= 0:
            assert row[11] == ti.photon_ke(e.vel[ph]) and row[11] > 0
    h.close()


# ---- 4. the reference taken mid-run ---------------------------------------------------------------------------------------
def test_reference_taken_mid_run():
    s = system(8193, "middle")
    N = s.N
    h = capi.Handle(0)
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    h.track_open(8)
    h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
    refs, want = [take_reference(h, s, d)], []
    for t in range(1, 7):
        h.nve_kick_drift(d["pos"], d["vel"], f, N, DT)
        h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
        h.nve_half_kick(d["vel"], f, N, DT)
        if t == 3:
            refs.append(take_reference(h, s, d))  # the records from here on use this step's d, not the current one
        h.track_record(t, d["vel"], N)
        want.append((Expect(h, t, d, s), refs[-1]))
    got, _ = h.track_read(8)
    for row, (e, ref) in zip(got, want):
        check(row, e, *ref)
    assert got[3][10] != ti.autocorr(got[3][1:4], got[3][1:4])  # not d(t) . d(t)
    assert got[2][10] == ti.autocorr(got[2][1:4], got[2][1:4])  # the step the reference was taken at: d . d
    h.close()


# ---- 5. the ring -----------------------------------------------------------------------------------------------------------
def test_ring_capacity_read_and_reopen():
    s = system(769, "last")
    N = s.N
    h = capi.Handle(0)
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)

    def steps(t0, t1):
        rows = []
        for t in range(t0, t1):
            h.nve_kick_drift(d["pos"], d["vel"], f, N, DT)
            h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
            h.track_record(t, d["vel"], N)
            rows.append(t)
        return rows

    h.track_open(1)  # capacity 1: always the newest
    steps(1, 4)
    got, total = h.track_read(5)
    assert total == 3 and len(got) == 1 and got[0][0] == 3
    h.track_open(5)  # re-open: ring and reference emptied
    got, total = h.track_read(5)
    assert total == 0 and len(got) == 0
    h.track_record(0, d["vel"], N)
    got, _ = h.track_read(1)
    assert got[0][10] == 0.0  # the reference is zero again: C = 0 . d
    h.track_set_reference()
    steps(1, 13)  # 13 records in a ring of 5
    got, total = h.track_read(0)
    assert total == 13 and len(got) == 0  # read(0): only the total
    for k in (1, 3, 5, 9):
        got, total = h.track_read(k)
        assert total == 13 and list(got[:, 0]) == list(range(13 - min(k, 5), 13))  # the newest k, oldest first
    h.close()


# ---- 6. stream order ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pdl", [1, 0])
def test_records_interleaved_with_the_fused_step(pdl):
    s = system(262145, "middle")
    h = capi.Handle(0)
    h.set_tuning(pdl=pdl)
    got, want, ref = run_harness(h, s, "fused", True, "window", steps=6)
    for row, e in zip(got, want):
        check(row, e, *ref)
    h.close()


def test_steps_and_records_in_a_graph():
    """20 fused steps with a record after each, captured in one CUDA graph and replayed: the same records as the eager
    run, bit for bit."""
    s = system(8193, "middle")
    N, n = s.N, s.N

    def setup():
        h = capi.Handle(0)
        d = upload(s)
        h.track_open(32)
        h.bussi_reset()
        h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, PARAMS)
        h.bussi_ke(d["vel"], None, 0, n)
        h.track_set_reference()
        h.md_step_one(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS, 0, n,
                      bussi_args(0, n), wrap=True)
        h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS, 0, n,
                        bussi_args(0, n), wrap=True)
        capi.sync()
        return h, d

    a = bussi_args(1, n)

    def steps(h, d, st):
        for t in range(1, 21):
            h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, PARAMS, 0, n, a,
                            st, wrap=True)
            capi.check(h.lib.cavb200_track_record_from(h.h, h.h, h.h, t, d["vel"].ptr, N, PENDING, st), "record")

    eager, de = setup()
    steps(eager, de, None)
    want, total = eager.track_read(32)
    assert total == 20
    h, d = setup()
    stream = capi.Stream()
    capi.sync()
    g = h.graph_capture(stream.ptr, lambda: steps(h, d, stream.ptr))
    assert h.track_read(32, stream.ptr)[1] == 0  # capturing launches nothing
    h.graph_launch(g, stream.ptr)
    got, total = h.track_read(32, stream.ptr)
    assert total == 20 and ti.same_bits(got, want)
    assert np.array_equal(d["pos"].numpy(), de["pos"].numpy())
    h.graph_destroy(g)
    assert h.fault_count == 0 and eager.fault_count == 0
    h.close()
    eager.close()


def test_record_from_argument_checks():
    h, other = capi.Handle(0), capi.Handle(0)
    with pytest.raises(capi.CavbError):
        h.track_record_from(other, other, 0, None, 0)  # ring not opened
    h.track_open(2)
    with pytest.raises(capi.CavbError):
        h.track_record_from(other, other, 0, None, 0, flags=2)  # unknown flag
    with pytest.raises(capi.CavbError):
        capi.check(h.lib.cavb200_track_record_from(h.h, None, None, 0, None, 0, 0, None), "record")  # no force handle
    with pytest.raises(capi.CavbError):
        capi.check(h.lib.cavb200_track_set_reference_from(h.h, None, None), "reference")
    h.track_record_from(other, None, 5, None, 0)
    got, _ = h.track_read(2)
    assert got[0][0] == 5 and np.all(np.isnan(got[0][12:15])) and got[0][15] == 0.0  # other's zeroed Scalars
    h.close()
    other.close()


# ---- 7. the plugin classes through hoomd_shim ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mods():
    sys.path.insert(0, BUILD)
    import _hoomd_shim  # noqa: F401  (registers ForceCompute / Thermostat bases first)
    import _bussi_reservoir
    import _cavitymd
    return _hoomd_shim, _cavitymd, _bussi_reservoir


def _sysdef(shim, s, seed=7):
    exec_conf = shim.ExecutionConfiguration(True, 0)
    pd = shim.ParticleData(s.N, s.box[0], s.box[1], s.box[2], list(s.types), exec_conf)
    pd.setPositions(s.pos)
    pd.setVelocities(s.vel)
    pd.setCharges(s.charge)
    pd.setImages(s.image)
    return shim.SystemDefinition(pd, seed), pd


def _typeid(pos):
    return (pos[:, 3].view(np.uint64) & 0xFFFFFFFF).astype(np.int64)


class Snap:
    """Host snapshot of the shim's arrays after a step: what check() needs, with force_read / bussi_read from the
    plugin objects' getters."""

    def __init__(self, pd, s, t, dipole, energies, cumulative, group_tags, pending):
        self.t = t
        pos = pd.getPositions()
        ph = np.flatnonzero(_typeid(pos) == s.L_typeid)
        self.force = (np.asarray(energies), np.asarray(dipole), int(ph[0]) if len(ph) else -1)
        self.cumulative = cumulative  # None: no method, so no thermostat handle
        self.bussi = None
        self.pos, self.image, self.vel = pos, pd.getImages(), pd.getVelocities()
        tags = np.asarray(pd.getTags())
        self.charge = s.charge[tags]  # the charges move with their particles in a sort
        self.box = s.box
        rtag = np.argsort(tags)
        self.group = rtag[group_tags]
        self.offset, self.pending = 0, pending

    ph_local = Expect.ph_local
    exact = Expect.exact


def _plugin_run(mods, mode, photon="last", n_mol=4000, steps=6, flush=False, bath=False, sorts=(), thermostat=True):
    """TwoStepConstantVolumeCavity (mode None: the drop-in force + BussiReservoirThermostat, no method) driven as
    IntegratorTwoStep::update does, trackRecord(t) after each integrateStepTwo(t)."""
    shim, cav, bus = mods
    s = ti.make_system(n_mol + 1, photon)
    mol = np.flatnonzero(s.typeid != s.L_typeid)
    ph0 = di.photon_index(s)
    dof = 3.0 * len(mol) - 3.0
    sysdef, pd = _sysdef(shim, s)
    group = shim.ParticleGroup(sysdef, [int(x) for x in mol])
    group.setTranslationalDOF(dof)
    th = bus.BussiReservoirThermostat(shim.VariantConstant(KT), group, shim.ComputeThermo(sysdef, group), sysdef, TAU)
    fc = cav.CavityForceComputeGPU(sysdef, di.OMEGAC, di.G)
    method = None
    if mode is not None:
        method = cav.TwoStepConstantVolumeCavity(sysdef, group, th if thermostat else None, fc, mode)
        method.index_list_group = True
        method.setDeltaT(DT)
        if bath:
            method.setPhotonBath(shim.ParticleGroup(sysdef, [ph0]), shim.VariantConstant(KT), 0.5)
    fc.trackOpen(steps + 8)
    fc.compute(0)
    pd.setNetForce(fc.getForces())
    fc.trackSetReference()
    d0 = np.asarray(fc.getDipole())
    D0, S0 = di.exact_dipole(pd.getPositions(), s.charge, pd.getImages(), s.box, ph0)
    ref = (d0, (D0, di.tolerance(D0, S0, s.N)))
    draws = [rng.bussi_draws(t, 11, 0, dof) for t in range(steps)]
    perm = np.random.default_rng(17)
    u = np.random.default_rng(45).uniform(-1.0, 1.0, size=(steps, 3))  # the photon bath's draws
    snaps, photon_rows = [], []
    for t in range(steps):
        if t in sorts:
            ph = int(np.flatnonzero(_typeid(pd.getPositions()) == s.L_typeid)[0])
            order = perm.permutation(s.N)
            while order[ph] == ph:
                order = perm.permutation(s.N)
            pd.sortParticles([int(o) for o in order])
        if method is None:
            bus._inject_draws(list(draws[t]))
            th.getRescalingFactorsOne(t, DT)
            fc.compute(t + 1)
        else:
            bus._inject_draws(list(draws[t]))
            method.integrateStepOne(t)
            fc.compute(t + 1)
            pd.setNetForce(fc.getForces())
            if bath:
                cav._inject_draws(list(u[t]))
            method.integrateStepTwo(t)
            if flush:
                method.flush()
        fc.trackRecord(t)
        pending = mode == "one_launch" and not flush
        # the reservoir getter reads cavb200_bussi_read of the method's handle (the fused path keeps no host part)
        cum = th.getReservoirEnergyTranslational() if method is not None else None
        snaps.append(Snap(pd, s, t, fc.getDipole(), [fc.getHarmonicEnergy(), fc.getCouplingEnergy(),
                                                      fc.getDipoleSelfEnergy()], cum, mol, pending))
        photon_rows.append(snaps[-1].force[2])
    rows = np.array(fc.trackRead(steps + 8))
    return rows, snaps, ref, photon_rows, (fc, th, method, pd)


@pytest.mark.parametrize("mode", ["stored", "rank1", "one_launch"])
@pytest.mark.parametrize("flush", [False, True])
@pytest.mark.parametrize("photon", ["last", "middle"])
def test_plugin_method_records(mods, mode, flush, photon):
    if flush and mode != "one_launch":
        pytest.skip("flush() only matters in the one_launch mode")
    rows, snaps, ref, _, _ = _plugin_run(mods, mode, photon, flush=flush)
    _check_plugin_rows(rows, snaps, ref)


def _check_plugin_rows(rows, snaps, ref):
    """The method's records: [12] (when complete) against math.fsum of the group's kinetic energy, [13] a Bussi factor,
    [14] bit for bit the thermostat object's reservoir getter, everything else through check()."""
    assert len(rows) == len(snaps)
    for row, e in zip(rows, snaps):
        e.bussi = dict(ke=row[12], alpha=row[13], cumulative=e.cumulative)
        check(row, e, *ref, photon_expected=e.force[2])
        assert 0.9 < row[13] < 1.1 and row[14] != 0.0
        assert np.isnan(row[12]) == e.pending


def test_plugin_drop_in_force_without_method(mods):
    """The drop-in force next to BussiReservoirThermostat: the force object cannot know the thermostat, so [12..14] are
    NaN, never zeros; everything else is the force's."""
    rows, snaps, ref, _, _ = _plugin_run(mods, None, "middle", steps=4)
    for row, e in zip(rows, snaps):
        check(row, e, *ref, photon_expected=e.force[2])
        assert np.all(np.isnan(row[12:15]))


def test_plugin_one_launch_flush_completes_the_velocity_fields(mods):
    """one_launch: without flush() [11] / [12] are NaN in every record, the rest complete; a record after flush() has
    the full-step photon kinetic energy."""
    rows, snaps, ref, _, (fc, th, method, pd) = _plugin_run(mods, "one_launch", "middle", steps=4)
    assert np.all(np.isnan(rows[:, 11])) and np.all(np.isnan(rows[:, 12]))
    assert np.all(np.isfinite(rows[:, 1:11])) and np.all(np.isfinite(rows[:, 13:16]))
    method.flush()
    fc.trackRecord(99)
    last = np.array(fc.trackRead(1))[0]
    vel = pd.getVelocities()
    ph = int(last[15])
    assert _typeid(pd.getPositions())[ph] == synth.L_TYPEID
    assert last[11] == ti.photon_ke(vel[ph])
    KE = ti.group_ke_exact(vel, snaps[-1].group)
    assert abs(last[12] - KE) <= ti.group_ke_bound(KE, len(snaps[-1].group))


def test_plugin_photon_bath(mods):
    for mode in ("rank1", "one_launch"):
        rows, snaps, ref, _, _ = _plugin_run(mods, mode, "middle", bath=True, flush=mode == "one_launch")
        _check_plugin_rows(rows, snaps, ref)


@pytest.mark.parametrize("mode", ["stored", "rank1", "one_launch"])
def test_plugin_records_follow_the_photon_through_sorts(mods, mode):
    rows, snaps, ref, photon_rows, _ = _plugin_run(mods, mode, "last", sorts=(2, 4), flush=mode == "one_launch")
    _check_plugin_rows(rows, snaps, ref)
    assert len(set(photon_rows)) == 3 and photon_rows[0] == len(snaps[0].vel) - 1  # two sorts moved the photon
    assert [int(r[15]) for r in rows] == photon_rows


def test_dipole_autocorrelation_against_host_snapshots(mods):
    """The reference's DipoleAutocorrelation output d(0) . d(t) over 50 steps of the one_launch method, from host
    snapshots taken in the test (np.dot of exact dipoles), against the device records' C(t)."""
    rows, snaps, ref, _, _ = _plugin_run(mods, "one_launch", "middle", steps=50, n_mol=2000)
    D0, tol0 = ref[1]
    for row, e in zip(rows, snaps):
        D, tol = e.exact()
        c_host = float(np.dot(D0, D))
        assert abs(row[10] - c_host) <= ti.autocorr_bound(D0, tol0, D, tol) + ti.autocorr_rounding_bound(D0, D)
