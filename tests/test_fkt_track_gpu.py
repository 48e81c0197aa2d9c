"""The F(k,t) tracker without snapshots (cavb200_fkt_track_*): every record against the calls it is built from, bit for
bit (rho against cavb200_rhok on the same Scalar4 frame with T = 1, each F against cavb200_fkt on the pair (stored
reference, this frame)), against exact sums (tests/fkt_inputs.py), against the schedule of the host mirror
analysis.FieldAutocorrelationTracker, interleaved with the fused MD step in both launch modes, inside a CUDA graph,
under a permutation of the particles, the argument checks, and the plugin class through hoomd_shim."""
import ctypes as C
import importlib.util
import os
import sys

import numpy as np
import pytest

import fkt_inputs as fi
from cav_hoomd_b200 import analysis, capi, rng, synth

pytestmark = pytest.mark.gpu

INVALID_VALUE = 1
MISALIGNED = 716
REC, ADD = capi.Handle.FKT_RECORD, capi.Handle.FKT_ADD_REFERENCE
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def extras():
    spec = importlib.util.spec_from_file_location("cavb200_extras", os.path.join(ROOT, "plugin", "python",
                                                                                  "cavb200_extras.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def scalar4(frame, typeid=None):
    """[N, 3] -> HOOMD Scalar4 [N, 4] (type id in the low 32 bits of w)."""
    p = np.zeros((frame.shape[0], 4))
    p[:, :3] = frame
    if typeid is not None:
        p[:, 3] = np.asarray(typeid, dtype=np.int64).view(np.float64)
    return p


def rhok_one(h, d_pos, N, d_k, K):
    """cavb200_rhok of one Scalar4 frame (T = 1): what the tracker must reproduce bit for bit."""
    d_rho = capi.DeviceArray((K, 2), np.float64)
    h.rhok(d_pos, 4, 4 * N, N, 1, d_k, K, d_rho)
    return d_rho.numpy()


def fkt_pair(h, a, b):
    """cavb200_fkt F[0][1] of the two-frame table (a, b), fields [K, 2]."""
    K = a.shape[0]
    d_rho = capi.DeviceArray.from_numpy(np.stack([a, b]))
    d_out = capi.DeviceArray((1, 2), np.float64)
    h.fkt(d_rho, 2, K, 1, 2, d_out)
    return d_out.numpy()[0, 1]


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def fields(rec, M, K):
    return rec[:, 2 + M:].reshape(len(rec), K, 2)


# ---- 1. bit for bit against cavb200_rhok and cavb200_fkt ---------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 50, 64, 1030])
@pytest.mark.parametrize("N", [1, 700, 40000, 1048576])
def test_records_are_the_existing_calls(N, K):
    h = capi.Handle(0)
    M = 3
    frames = fi.walk_frames(N, 3, seed=N + K)
    kvec = fi.kvectors(K)
    d_k = capi.DeviceArray.from_numpy(kvec)
    d_pos = [capi.DeviceArray.from_numpy(scalar4(f)) for f in frames]
    h.fkt_track_open(kvec, M, 4, N)
    h.fkt_track_step(d_pos[0], N, 0, ADD)
    h.fkt_track_step(d_pos[1], N, 1, REC | ADD)
    h.fkt_track_step(d_pos[2], N, 2, REC)
    rec, total = h.fkt_track_read(4)
    assert total == 2 and rec.shape == (2, 2 + M + 2 * K)
    rho = [rhok_one(h, d, N, d_k, K) for d in d_pos]
    assert np.array_equal(rec[:, 0], [1.0, 2.0]) and np.array_equal(rec[:, 1], [1.0, 2.0])
    for i, t in enumerate((1, 2)):
        assert np.array_equal(bits(fields(rec, M, K)[i]), bits(rho[t]))
        for r in range(t):
            assert bits(rec[i, 2 + r]) == bits(fkt_pair(h, rho[r], rho[t])), (t, r)
        assert np.all(np.isnan(rec[i, 2 + t:2 + M]))
    assert h.fault_count == 0
    h.close()


# ---- 2. against exact sums ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,K", [(700, 50), (40000, 64)])
def test_records_against_exact_sums(N, K):
    import torch
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    h = capi.Handle(0)
    M = 2
    frames = fi.walk_frames(N, 3, seed=3 * N)
    kvec = fi.kvectors(K)
    h.fkt_track_open(kvec, M, 8, N)
    for t, f in enumerate(frames):
        h.fkt_track_step(capi.DeviceArray.from_numpy(scalar4(f)), N, t, ADD if t == 0 else (REC | ADD if t == 1 else REC))
    rec, _ = h.fkt_track_read(8)
    geo = fi.geometry(N, 1, K, num_sms)
    rho = {}
    for t in range(3):
        (R, tol_re, tol_im, _), = fi.reference(frames[t:t + 1], kvec, geo).values()
        rho[t] = R
        if t:
            got = fields(rec, M, K)[t - 1]
            assert np.all(np.abs(got[:, 0] - R.real) <= tol_re) and np.all(np.abs(got[:, 1] - R.imag) <= tol_im)
            rho[t] = got[:, 0] + 1j * got[:, 1]
    # F against the exact sum of the products of the fields the tracker holds (its references are bitwise rho, test 1)
    ref0 = rhok_one(h, capi.DeviceArray.from_numpy(scalar4(frames[0])), N, capi.DeviceArray.from_numpy(kvec), K)
    refs = [ref0[:, 0] + 1j * ref0[:, 1], rho[1]]
    for i, t in enumerate((1, 2)):
        for r in range(t):
            Fs, b = fi.fkt_exact(np.stack([refs[r], rho[t]]), 0, 1)
            assert abs(rec[i, 2 + r] - Fs) <= b, (t, r, rec[i, 2 + r], Fs, b)
    h.close()


# ---- 3. the schedule of the host mirror ------------------------------------------------------------------------------
class _State:
    def __init__(self, N):
        self.N, self.device = N, 0
        self.pos = capi.DeviceArray((N, 4), np.float64)


class _HandleAsForce:
    """The C++ force's fkt* methods on a capi.Handle and a device state: drives cavb200_extras.FieldAutocorrelation
    without HOOMD."""

    def __init__(self, h, st):
        self.h, self.st = h, st

    def fktOpen(self, kvectors, max_references, capacity):
        self.h.fkt_track_open(np.array(kvectors), max_references, capacity, self.st.N)

    def fktStep(self, timestep, record, add_reference):
        self.h.fkt_track_step(self.st.pos, self.st.N, timestep, (REC if record else 0) | (ADD if add_reference else 0))

    def fktRead(self, max_records):
        return self.h.fkt_track_read(max_records)


def test_schedule_matches_the_mirror():
    N, K, steps = 5000, 50, 12
    frames = fi.walk_frames(N, steps + 1, seed=12)
    st = _State(N)
    st.pos.upload(scalar4(frames[0]))
    h = capi.Handle(0)
    mirror = analysis.FieldAutocorrelationTracker(st, kmag=1.0, num_wavevectors=K, reference_interval_steps=2,
                                                  max_references=3, handle=h)
    X = extras()
    dev = X.FieldAutocorrelation(_HandleAsForce(h, st), mirror.wavevectors, reference_interval_steps=2,
                                 max_references=3, capacity=64)
    want, refs = [], [mirror.references[0]["field"]]
    for t in range(steps + 1):
        st.pos.upload(scalar4(frames[t]))
        n_before = len(mirror.references)
        want += [(r, t, lag, v) for r, lag, v in mirror.act(t)]
        dev.act(t)
        if len(mirror.references) > n_before:
            refs.append(mirror.references[-1]["field"])
    rows, rho = dev.read()
    assert [(r, t, lag) for r, t, lag, _ in rows] == [(r, t, lag) for r, t, lag, _ in want]
    assert len(rows) == 1 + 1 + 2 + 2 + 3 * (steps - 4) and rho.shape == (steps, K, 2)
    assert dev.reference_timesteps == [0, 2, 4]
    for (r, t, _, F), (_, _, _, Fm) in zip(rows, want):
        cur = rho[t - 1, :, 0] + 1j * rho[t - 1, :, 1]
        Fs, b = fi.fkt_exact(np.stack([refs[r], cur]), 0, 1)
        assert abs(F - Fs) <= b and abs(Fm - Fs) <= 1e-12 * N * N, (r, t, F, Fs, b, Fm)
    assert dev.read()[0] == []  # nothing new since the last read
    h.close()


# ---- 4. the ring ---------------------------------------------------------------------------------------------------------
def test_ring_wraps():
    N, K, M, cap, steps = 700, 8, 4, 5, 12
    h = capi.Handle(0)
    frames = fi.walk_frames(N, steps + 1, seed=4)
    d = [capi.DeviceArray.from_numpy(scalar4(f)) for f in frames]
    h.fkt_track_open(fi.kvectors(K), M, cap, N)
    h.fkt_track_step(d[0], N, 0, ADD)
    for t in range(1, steps + 1):
        h.fkt_track_step(d[t], N, t, REC | (ADD if t in (3, 6) else 0))
    rec, total = h.fkt_track_read(100)
    assert total == steps and len(rec) == cap
    assert np.array_equal(rec[:, 0], np.arange(steps - cap + 1, steps + 1))
    assert np.array_equal(rec[:, 1], [3.0] * cap)
    assert np.all(np.isfinite(rec[:, 2:5])) and np.all(np.isnan(rec[:, 5]))
    rec3, total3 = h.fkt_track_read(3)
    assert total3 == steps and np.array_equal(rec3, rec[-3:], equal_nan=True)
    none, total0 = h.fkt_track_read(0)
    assert len(none) == 0 and total0 == steps
    # before the wrap: records 1..3 with 1, 1, 1 references and NaN beyond
    h.fkt_track_open(fi.kvectors(K), M, cap, N)
    h.fkt_track_step(d[0], N, 0, ADD)
    for t in range(1, 4):
        h.fkt_track_step(d[t], N, t, REC)
    rec, total = h.fkt_track_read(100)
    assert total == 3 and np.array_equal(rec[:, 0], [1, 2, 3]) and np.all(rec[:, 1] == 1.0)
    assert np.all(np.isnan(rec[:, 3:2 + M]))
    h.close()


# ---- 5. interleaved with the fused MD step ----------------------------------------------------------------------------
OMEGAC, G = 0.01, 1e-3
KT, TAU, DT = synth.KT_100K, synth.TAU_5PS, synth.DT_1FS


def _flags(t):
    return ADD if t == 0 else (REC | (ADD if t % 3 == 0 else 0))


def replay(frames_dev, N, kvec, M, cap):
    """The tracker run afterwards, on a fresh handle, on positions copied out at each step."""
    h = capi.Handle(0)
    h.fkt_track_open(kvec, M, cap, N)
    for t, d in enumerate(frames_dev):
        h.fkt_track_step(d, N, t, _flags(t))
    rec, total = h.fkt_track_read(cap)
    h.close()
    return rec, total


@pytest.mark.parametrize("pdl", [1, 0])
def test_interleaved_with_the_fused_step(pdl):
    n_mol, steps, K, M = 100000, 8, 64, 4
    s = synth.make_system(n_mol, replica=61)
    N = s.N
    kvec = fi.kvectors(K)
    dof = 3.0 * n_mol - 3.0
    h = capi.Handle(0)
    h.set_tuning(pdl=pdl)
    p = capi.Params.make(OMEGAC, G)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    copies = [capi.DeviceArray((N, 4), np.float64) for _ in range(steps + 1)]
    lib = capi.load()
    h.fkt_track_open(kvec, M, 16, N)
    h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, p)
    h.bussi_ke(d["vel"], None, 0, n_mol)
    h.fkt_track_step(d["pos"], N, 0, _flags(0))
    capi.check(lib.cavb200_memcpy_d2d(copies[0].ptr, d["pos"].ptr, copies[0].nbytes, None), "d2d")
    for t in range(1, steps + 1):
        args = capi.BussiArgs(KT, TAU, DT, dof, *rng.bussi_draws(t, 9, 0, dof))
        step = h.md_step_one if t == 1 else h.md_step_fused
        step(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s.box, s.L_typeid, p, 0, n_mol, args, wrap=True)
        h.fkt_track_step(d["pos"], N, t, _flags(t))
        capi.check(lib.cavb200_memcpy_d2d(copies[t].ptr, d["pos"].ptr, copies[t].nbytes, None), "d2d")
    rec, total = h.fkt_track_read(16)
    assert h.fault_count == 0 and total == steps
    want, want_total = replay(copies, N, kvec, M, 16)
    assert want_total == total and np.array_equal(bits(rec), bits(want))
    assert not np.array_equal(copies[0].numpy(), copies[steps].numpy())  # the particles moved
    assert np.array_equal(rec[:, 1], [1, 1, 1, 2, 2, 2, 3, 3])
    h.close()


# ---- 6. no synchronisation inside a step: a captured graph ------------------------------------------------------------
def test_steps_captured_in_a_graph():
    K, M, cap = 64, 3, 8
    kvec = fi.kvectors(K)
    sizes = (40000, 700, 40000)
    frames = [fi.walk_frames(n, 1, seed=n + i)[0] for i, n in enumerate(sizes)]
    d = [capi.DeviceArray.from_numpy(scalar4(f)) for f in frames]
    ref = capi.DeviceArray.from_numpy(scalar4(fi.walk_frames(40000, 1, seed=99)[0]))

    def setup(h):
        h.fkt_track_open(kvec, M, cap, 40000)
        h.fkt_track_step(ref, 40000, 0, ADD)
        h.fkt_track_step(d[0], 40000, 1, ADD)

    direct = capi.Handle(0)
    setup(direct)
    for i, n in enumerate(sizes):
        direct.fkt_track_step(d[i], n, 10 + i, REC)
    want, _ = direct.fkt_track_read(cap)

    h = capi.Handle(0)
    setup(h)
    stream = capi.Stream()
    stream.sync()
    capi.sync()
    g = h.graph_capture(stream.ptr, lambda: [h.fkt_track_step(d[i], n, 10 + i, REC, stream.ptr)
                                             for i, n in enumerate(sizes)])
    got0, total0 = h.fkt_track_read(cap, stream.ptr)
    assert total0 == 0  # capturing launches nothing
    h.graph_launch(g, stream.ptr)
    got, total = h.fkt_track_read(cap, stream.ptr)
    assert total == 3 and np.array_equal(bits(got), bits(want))
    h.graph_launch(g, stream.ptr)  # a replay appends again, after the first three
    again, total = h.fkt_track_read(cap, stream.ptr)
    assert total == 6 and np.array_equal(bits(again[3:]), bits(want))
    h.graph_destroy(g)
    assert h.fault_count == 0
    h.close()
    direct.close()


# ---- 7. a sort of the particles ---------------------------------------------------------------------------------------
def test_permutation_changes_rho_within_the_bound():
    import torch
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    N, K, M = 40000, 64, 1
    frame = fi.walk_frames(N, 1, seed=77)[0]
    perm = np.random.default_rng(78).permutation(N)
    kvec = fi.kvectors(K)
    geo = fi.geometry(N, 1, K, num_sms)
    out = []
    for f in (frame, frame[perm]):
        h = capi.Handle(0)
        h.fkt_track_open(kvec, M, 2, N)
        h.fkt_track_step(capi.DeviceArray.from_numpy(scalar4(f)), N, 0, ADD)
        h.fkt_track_step(capi.DeviceArray.from_numpy(scalar4(f)), N, 1, REC)
        rec, _ = h.fkt_track_read(2)
        (R, tol_re, tol_im, _), = fi.reference(f[None], kvec, geo).values()
        got = fields(rec, M, K)[0]
        assert np.all(np.abs(got[:, 0] - R.real) <= tol_re) and np.all(np.abs(got[:, 1] - R.imag) <= tol_im)
        out.append((got, tol_re, tol_im))
        h.close()
    (a, ta_re, ta_im), (b, tb_re, tb_im) = out
    assert np.all(np.abs(a[:, 0] - b[:, 0]) <= ta_re + tb_re) and np.all(np.abs(a[:, 1] - b[:, 1]) <= ta_im + tb_im)


# ---- 8. argument checks ------------------------------------------------------------------------------------------------
def test_argument_checks():
    h = capi.Handle(0)
    lib = h.lib
    N, K = 64, 4
    kvec = np.ascontiguousarray(fi.kvectors(K))
    kp = kvec.ctypes.data_as(C.POINTER(C.c_double))
    pos = capi.DeviceArray.from_numpy(scalar4(fi.walk_frames(N, 1, seed=1)[0]))
    n0 = h.launch_count
    out = np.zeros((4, 2 + 2 + 2 * K))
    n, tot = C.c_uint32(0), C.c_uint64(0)
    # no open yet
    assert lib.cavb200_fkt_track_step(h.h, pos.ptr, N, 1, REC, None) == INVALID_VALUE
    assert lib.cavb200_fkt_track_read(h.h, out.ctypes.data_as(C.POINTER(C.c_double)), 4, C.byref(n), C.byref(tot),
                                      None) == INVALID_VALUE
    for args in ((kp, 0, 2, 4, N), (kp, K, 0, 4, N), (kp, K, 1025, 4, N), (kp, K, 2, 0, N), (None, K, 2, 4, N)):
        assert lib.cavb200_fkt_track_open(h.h, *args) == INVALID_VALUE, args
    assert lib.cavb200_fkt_track_open(None, kp, K, 2, 4, N) == INVALID_VALUE
    assert lib.cavb200_fkt_track_open(h.h, kp, K, 1024, 4, N) == 0
    h.fkt_track_open(kvec, 2, 4, N)  # (through the binding, which sizes its read buffer from the open)
    for flags in (0, 4, 7):
        assert lib.cavb200_fkt_track_step(h.h, pos.ptr, N, 1, flags, None) == INVALID_VALUE
    assert lib.cavb200_fkt_track_step(h.h, None, N, 1, REC, None) == INVALID_VALUE
    assert lib.cavb200_fkt_track_step(h.h, pos.ptr + 8, N, 1, REC, None) == MISALIGNED
    assert h.launch_count == n0
    h.fkt_track_step(pos, N, 0, ADD)
    h.fkt_track_step(pos, N, 1, REC | ADD)
    assert lib.cavb200_fkt_track_step(h.h, pos.ptr, N, 2, ADD, None) == INVALID_VALUE  # two stored: the cap
    assert lib.cavb200_fkt_track_step(h.h, pos.ptr, N, 2, REC | ADD, None) == INVALID_VALUE
    h.fkt_track_step(pos, N, 2, REC)
    # N == 0: rho = 0 (a NULL pos is fine then), F against the stored references is then 0
    h.fkt_track_step(None, 0, 3, REC)
    rec, total = h.fkt_track_read(4)
    assert total == 3 and len(rec) == 3
    assert np.all(rec[2, 4:] == 0.0) and np.all(rec[2, 2:4] == 0.0) and rec[2, 1] == 2.0
    assert rec[0, 1] == 1.0 and np.isnan(rec[0, 3])
    # re-open drops the references
    h.fkt_track_open(kvec, 2, 4, N)
    h.fkt_track_step(pos, N, 0, ADD)
    h.fkt_track_step(pos, N, 1, REC | ADD)
    rec, total = h.fkt_track_read(4)
    assert total == 1 and rec[0, 1] == 1.0
    assert lib.cavb200_fkt_track_read(h.h, None, 4, C.byref(n), C.byref(tot), None) == INVALID_VALUE
    capi.sync()
    assert h.fault_count == 0
    h.close()


# ---- 9. the plugin class through hoomd_shim ---------------------------------------------------------------------------
BUILD = os.path.join(ROOT, "plugin", "build")


@pytest.fixture(scope="module")
def mods():
    sys.path.insert(0, BUILD)
    import _hoomd_shim  # noqa: F401  (registers ForceCompute / Thermostat bases first)
    import _bussi_reservoir  # noqa: F401
    import _cavitymd
    return _hoomd_shim, _cavitymd


def test_plugin_tracker_in_one_launch_mode_without_flush(mods):
    shim, cav = mods
    n_mol, steps, K, M, interval = 20000, 8, 50, 3, 2
    s = synth.make_system(n_mol, replica=62, photon="middle")
    exec_conf = shim.ExecutionConfiguration(True, 0)
    pd = shim.ParticleData(s.N, s.box[0], s.box[1], s.box[2], list(s.types), exec_conf)
    pd.setPositions(s.pos)
    pd.setVelocities(s.vel)
    pd.setCharges(s.charge)
    pd.setImages(s.image)
    sysdef = shim.SystemDefinition(pd, 7)
    group = shim.ParticleGroup(sysdef, [int(x) for x in np.flatnonzero(s.typeid != s.L_typeid)])
    fc = cav.CavityForceComputeGPU(sysdef, OMEGAC, G)
    method = cav.TwoStepConstantVolumeCavity(sysdef, group, None, fc, "one_launch")
    method.index_list_group = True
    method.setDeltaT(DT)
    kvec = synth.fibonacci_sphere(K) * 1.1
    X = extras()
    tracker = X.FieldAutocorrelation(fc, kvec, reference_interval_steps=interval, max_references=M, capacity=32)
    snaps = [pd.getPositions()]
    fc.compute(0)
    pd.setNetForce(fc.getForces())
    for t in range(steps):
        method.integrateStepOne(t)
        fc.compute(t + 1)
        pd.setNetForce(fc.getForces())
        method.integrateStepTwo(t)
        tracker.act(t + 1)  # no flush(): the positions are complete after the launch
        snaps.append(pd.getPositions())
    rows, rho = tracker.read()
    assert not np.array_equal(snaps[0], snaps[-1])

    # test 5's reference: the tracker afterwards on the positions of every step
    h = capi.Handle(0)
    h.fkt_track_open(kvec, M, 32, s.N)
    flags = [ADD] + [REC | (ADD if t in (2, 4) else 0) for t in range(1, steps + 1)]
    for t, snap in enumerate(snaps):
        h.fkt_track_step(capi.DeviceArray.from_numpy(snap), s.N, t, flags[t])
    want, total = h.fkt_track_read(32)
    assert total == steps
    assert np.array_equal(bits(rho), bits(fields(want, M, K)))
    assert rows == X.records_to_rows(want, [0, 2, 4], M)
    assert [(r, t, lag) for r, t, lag, _ in rows][:4] == [(0, 1, 1), (0, 2, 2), (0, 3, 3), (1, 3, 1)]
    assert fc.getFaultCount() == 0

    # a second tracker on the same force re-opens: the earlier references are gone
    again = X.FieldAutocorrelation(fc, kvec, reference_interval_steps=100, max_references=M, capacity=4)
    again.act(steps + 1)
    rows2, rho2 = again.read()
    assert [(r, t, lag) for r, t, lag, _ in rows2] == [(0, steps + 1, steps + 1)]
    assert abs(rows2[0][3] - float(np.mean(rho2[0, :, 0] ** 2 + rho2[0, :, 1] ** 2))) <= 1e-12 * s.N * s.N
    h.close()
