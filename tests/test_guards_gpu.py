"""Out-of-bounds canaries (compute-sanitizer is closed on this GPU pool, DESIGN.md section 5): every array a kernel
writes sits between two 4 KB guard zones inside one allocation; after each call the guards must still hold their
pattern and every byte of the arrays a call must not touch must be unchanged.  Sizes are ragged around the warp,
CTA and full-grid boundaries (150001 runs the folder step kernel on a full grid)."""
import numpy as np
import pytest

from cav_hoomd_b200 import capi, synth

pytestmark = pytest.mark.gpu

GUARD = 4096
PATTERN = 0xA5


class Guarded:
    """One device allocation: guard | payload | guard (payload 32-byte aligned)."""

    def __init__(self, a: np.ndarray):
        a = np.ascontiguousarray(a)
        self.shape, self.dtype, self.n = a.shape, a.dtype, a.nbytes
        pad = (-self.n) % 32
        self.buf = capi.DeviceArray((GUARD + self.n + pad + GUARD,), np.uint8)
        self.buf.fill_bytes(PATTERN)
        capi.sync()
        self.ptr = self.buf.offset(GUARD)
        if self.n:
            capi.check(capi.load().cavb200_memcpy_h2d(self.ptr, a.ctypes.data, self.n, None), "h2d")
        capi.sync()
        self.pad = pad

    def get(self):
        raw = self.buf.numpy()
        return raw[GUARD:GUARD + self.n].view(self.dtype).reshape(self.shape).copy()

    def guards_intact(self):
        raw = self.buf.numpy()
        return bool(np.all(raw[:GUARD] == PATTERN) and np.all(raw[GUARD + self.n:] == PATTERN))


def _setup(n_mol, photon="last"):
    s = synth.make_system(n_mol, replica=n_mol % 5, photon=photon)
    g = {k: Guarded(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    g["force"] = Guarded(np.full((s.N, 4), np.nan))
    g["net"] = Guarded(np.zeros((s.N, 4)))
    return s, g


def _check(g, s, untouched):
    for k, a in g.items():
        assert a.guards_intact(), f"guard of {k} overwritten"
    for k in untouched:
        assert np.array_equal(g[k].get().view(np.uint8), np.ascontiguousarray(getattr(s, k)).view(np.uint8)), f"{k} was modified"


@pytest.mark.parametrize("n_mol", [1, 31, 33, 383, 385, 1025, 150001])
def test_guards_single_calls_and_step(handle, n_mol):
    s, g = _setup(n_mol)
    p = capi.Params.make(0.01, 1e-3)
    dof = max(3.0 * n_mol - 3.0, 1.0)
    a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof, 0.3, max(dof - 1.0, 0.0) / 2)
    P = {k: v.ptr for k, v in g.items()}
    handle.bussi_reset()
    for variant in (0, 1, 2, 3):
        handle.set_tuning(variant=variant, threads=384, ctas_per_sm=2, unroll=2)
        handle.force(P["pos"], P["charge"], P["image"], P["force"], s.N, s.box, s.L_typeid, p)
        capi.sync()
        _check(g, s, ("pos", "charge", "image", "vel"))
        assert not np.isnan(g["force"].get()).any()
    handle.set_tuning(variant=3)
    handle.bussi_ke(P["vel"], None, 0, n_mol)
    handle.force_rank1(P["pos"], P["charge"], P["image"], s.N, s.box, s.L_typeid, p)
    handle.net_force_add_rank1(P["net"], P["charge"], P["pos"], s.N, s.L_typeid, 1e-3)
    capi.sync()
    _check(g, s, ("pos", "charge", "image", "vel"))
    for variant in (0, 1, 2, 3):
        handle.set_tuning(variant=variant, threads=384, ctas_per_sm=2, unroll=2)
        handle.step(P["pos"], P["charge"], P["image"], P["force"], P["vel"], s.N, s.box, s.L_typeid, p, 0, n_mol, a)
        capi.sync()
        _check(g, s, ("pos", "charge", "image"))
    v = g["vel"].get()
    assert np.array_equal(v[:, 3], s.vel[:, 3]) and np.array_equal(v[n_mol:], s.vel[n_mol:])  # masses, photon untouched


@pytest.mark.parametrize("n_mol", [1, 33, 257, 1025, 150001])
def test_guards_harness_steps(handle, n_mol):
    s, g = _setup(n_mol)
    p = capi.Params.make(0.01, 1e-3)
    dof = max(3.0 * n_mol - 3.0, 1.0)
    a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, 1.0, dof, -0.2, max(dof - 1.0, 0.0) / 2)
    P = {k: v.ptr for k, v in g.items()}
    handle.set_tuning(variant=3, threads=384, ctas_per_sm=2, unroll=2)
    handle.bussi_reset()
    handle.force(P["pos"], P["charge"], P["image"], P["force"], s.N, s.box, s.L_typeid, p)
    handle.bussi_ke(P["vel"], None, 0, n_mol)
    handle.nve_kick_drift(P["pos"], P["vel"], P["force"], s.N, 1.0)
    handle.nve_half_kick(P["vel"], P["force"], s.N, 1.0)
    handle.nvt_step_one(P["pos"], P["vel"], P["force"], s.N, 1.0, 0, n_mol, a)
    handle.nvt_step_two(P["vel"], P["force"], s.N, 1.0, 0, n_mol)
    handle.force_rank1(P["pos"], P["charge"], P["image"], s.N, s.box, s.L_typeid, p)
    handle.nvt_step_one_rank1(P["pos"], P["vel"], P["net"], P["charge"], s.N, 1.0, s.L_typeid, 1e-3, 0, n_mol, a)
    handle.md_step_one(P["pos"], P["vel"], None, P["charge"], P["image"], s.N, 1.0, s.box, s.L_typeid, p, 0, n_mol, a)
    for shape in (0, 1):
        handle.set_tuning(md_shape=shape)
        handle.md_step_fused(P["pos"], P["vel"], P["net"], P["charge"], P["image"], s.N, 1.0, s.box, s.L_typeid, p, 0, n_mol, a)
    handle.set_tuning(md_shape=0)
    handle.nvt_step_two_rank1(P["vel"], P["net"], P["charge"], P["pos"], s.N, 1.0, s.L_typeid, 1e-3, 0, n_mol)
    handle.track_open(4)
    handle.track_set_reference()
    handle.track_record(1, P["vel"], s.N)
    capi.sync()
    _check(g, s, ("charge", "image"))
    assert np.array_equal(g["pos"].get()[:, 3].view(np.uint64), s.pos[:, 3].view(np.uint64))   # type words
    assert np.array_equal(g["vel"].get()[:, 3], s.vel[:, 3])                                     # masses
    assert np.all(g["net"].get() == 0.0)                                                         # read-only here
    assert np.isfinite(g["pos"].get()[:, :3]).all() and np.isfinite(g["vel"].get()[:, :3]).all()
    assert handle.bussi_read()["err"] == 0.0


# F(k,t): (N, T, K, rhok_threads, frame padding) -- direct multi-tile, folded, multi-slab, 128 threads
RHOK_SHAPES = [(1537, 8000, 5, 256, 0), (1537, 8000, 5, 128, 1), (20001, 2, 64, 256, 0), (20001, 2, 1025, 256, 1),
               (5000, 2, 2051, 128, 1), (100001, 3, 64, 128, 1)]


@pytest.mark.parametrize("N,T,K,threads,pad", RHOK_SHAPES)
@pytest.mark.parametrize("layout", ["xyz", "scalar4", "f32"])
def test_guards_rhok(handle, N, T, K, threads, pad, layout):
    """cavb200_rhok / _rhok_f32 write rho only inside its array; positions (padding between frames included) and the
    wave vectors are unchanged byte for byte."""
    rng = np.random.default_rng(N + T + K)
    w, dt = (4, np.float64) if layout == "scalar4" else (3, np.float32 if layout == "f32" else np.float64)
    fs = w * N + pad * (8 if layout == "scalar4" else 5 if layout == "xyz" else 1)
    pos = np.full((T, fs), np.nan, dt)
    pos[:, :w * N].reshape(T, N, w)[:, :, :3] = rng.uniform(-20, 20, size=(T, N, 3))
    kvec = synth.fibonacci_sphere(max(K, 2))[:K]
    g = {"pos": Guarded(pos), "kvec": Guarded(kvec), "rho": Guarded(np.full((T, K, 2), np.nan))}
    handle.set_tuning(rhok_threads=threads)
    if layout == "f32":
        handle.rhok_f32(g["pos"].ptr, fs, N, T, g["kvec"].ptr, K, g["rho"].ptr)
    else:
        handle.rhok(g["pos"].ptr, w, fs, N, T, g["kvec"].ptr, K, g["rho"].ptr)
    capi.sync()
    handle.set_tuning(rhok_threads=0)
    for k, a in g.items():
        assert a.guards_intact(), f"guard of {k} overwritten"
    assert np.array_equal(g["pos"].get().view(np.uint8), pos.view(np.uint8))
    assert np.array_equal(g["kvec"].get().view(np.uint8), kvec.view(np.uint8))
    assert np.isfinite(g["rho"].get()).all()


@pytest.mark.parametrize("T,K,n_or,n_lag", [(12, 1, 8, 10), (1200, 64, 1000, 1000), (5, 4096, 9, 3)])
def test_guards_fkt(handle, T, K, n_or, n_lag):
    rng = np.random.default_rng(T + K)
    rho = rng.standard_normal((T, K, 2)) * 100.0
    g = {"rho": Guarded(rho), "out": Guarded(np.zeros((n_or, n_lag)))}
    handle.fkt(g["rho"].ptr, T, K, n_or, n_lag, g["out"].ptr)
    capi.sync()
    for k, a in g.items():
        assert a.guards_intact(), f"guard of {k} overwritten"
    assert np.array_equal(g["rho"].get().view(np.uint8), rho.view(np.uint8))
    o, l = np.meshgrid(np.arange(n_or), np.arange(n_lag), indexing="ij")
    assert np.array_equal(np.isnan(g["out"].get()), o + l >= T)
