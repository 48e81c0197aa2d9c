"""Every entry point that reduces the dipole, under every schedule its launcher picks, against the exact dipole of
neutral-molecule inputs (tests/dipole_inputs.py; the CPU side of the argument is tests/test_dipole_exact.py).

For each call:
  1. the photon index is the reference's (the first particle of type 'L');
  2. d (cavb200_force_read) is within |d_k - D_k| <= 2 ulp(D_k) + (n_c u)^2 S_k of the correctly rounded sum D;
  3. the energies and, where the call gives them, Dq, F_L and the force array equal BIT FOR BIT the reference's
     operation order evaluated on the kernel's own d (dipole_inputs.finalize / force_rows);
  4. energies, Dq, F_L and forces are within the tolerance carried through from D (dipole_inputs.propagated) -- on these
     inputs this replaces "1e-10 against the serial-sum oracle", which the oracle itself misses on the shuffled ones.
The kinetic energy of cavb200_bussi_ke and of the step is held to (n_c + 4) u KE against math.fsum of 1/2 m |v|^2.
At the end of the module the largest |d - D| of each path is printed, in ulp of D.
"""
import functools
import math

import numpy as np
import pytest

import dipole_inputs as di
from cav_hoomd_b200 import capi, synth

pytestmark = pytest.mark.gpu

C = di.constants()
PARAMS = capi.Params.make(di.OMEGAC, di.G, di.PHMASS)
KINDS = list(di.KINDS)
MD_KINDS = ["adj50", "shuf1000", "water_blk50"]  # the big charged photon would tear the molecules apart in one kick
KT, TAU, DT = synth.KT_100K, synth.TAU_5PS, synth.DT_1FS
U = di.U
WORST = {}  # path -> [largest |d - D| in ulp of D (D != 0), largest |d - D| / tolerance]


@functools.lru_cache(maxsize=None)  # every input is built once per module (~1 GB of host memory up to 1M particles)
def inputs(kind, N):
    s = di.build(kind, N)
    ph = di.photon_index(s)
    D, S = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph)
    return s, ph, D, S


@pytest.fixture(scope="module", autouse=True)
def worst_per_path(pytestconfig):
    yield
    if not WORST:
        return
    lines = ["", "largest |d - D| per path (ulp of D over inputs with D != 0; fraction of the tolerance over all inputs)"]
    lines += [f"  {path:44s} {u:6.2f} ulp   {r:6.3f} of tol" for path, (u, r) in sorted(WORST.items())]
    capman = pytestconfig.pluginmanager.getplugin("capturemanager")
    with capman.global_and_fixture_disabled():
        print("\n".join(lines))


@pytest.fixture
def h():
    handle = capi.Handle(0)
    yield handle
    handle.close()


def upload(s, keys=("pos", "charge", "image", "vel")):
    return {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in keys}


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def check(path, s, D, S, ph_ref, d, en, ph, Dq=None, FL=None, force=None, index_offset=0):
    """Assertions 1-4 of the module docstring for one call on system s (whose pos / image are the ones reduced)."""
    assert ph == (ph_ref + index_offset if ph_ref >= 0 else -1), (path, ph, ph_ref)
    tol = di.tolerance(D, S, s.N)
    err = np.abs(np.asarray(d) - D)
    w = WORST.setdefault(path, [0.0, 0.0])
    nz = D != 0.0
    if nz.any():
        w[0] = max(w[0], float(di.ulps(d, D)[nz].max()))
    w[1] = max(w[1], float((err / tol).max()))
    assert np.all(err <= tol), f"{path}: |d - D| = {err} > tolerance {tol} ({di.ulps(d, D)} ulp of D)"
    q = di.unwrapped(s.pos, s.image, s.box)[ph_ref] if ph_ref >= 0 else np.zeros(3)
    en_d, Dq_d, FL_d = di.finalize(d, q, C)
    en_D, Dq_D, FL_D = di.finalize(D, q, C)
    b = di.propagated(D, tol, q, s.charge, C)
    assert np.array_equal(bits(en), bits(en_d)), (path, en, en_d)
    assert np.all(np.abs(en - en_D) <= b["energies"]), (path, en - en_D, b["energies"])
    if Dq is not None:
        assert np.array_equal(bits(Dq), bits(Dq_d)), (path, Dq, Dq_d)
        assert np.all(np.abs(Dq - Dq_D) <= b["Dq"])
    if FL is not None:
        assert np.array_equal(bits(FL), bits(FL_d)), (path, FL, FL_d)
        assert np.all(np.abs(FL - FL_D) <= b["FL"])
    if force is not None:
        want = di.force_rows(s.charge, s.typeid, s.L_typeid, ph_ref, Dq_d, FL_d, C)
        bad = np.nonzero(np.any(bits(force) != bits(want), axis=1))[0]
        assert len(bad) == 0, (path, bad[:5], force[bad[:5]], want[bad[:5]])
        f_D = di.force_rows(s.charge, s.typeid, s.L_typeid, ph_ref, Dq_D, FL_D, C)
        mol = s.typeid != s.L_typeid
        assert np.all(np.abs(force[mol, :2] - f_D[mol, :2]) <= b["force"][mol] + 4 * U * np.abs(f_D[mol, :2]))
        if ph_ref >= 0:
            assert np.all(np.abs(force[ph_ref, :3] - f_D[ph_ref, :3]) <= b["FL"])


def check_ke(path, vel, idx, ke):
    v = vel[idx]
    terms = 0.5 * v[:, 3] * (v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
    KE = math.fsum(terms)
    assert abs(ke - KE) <= (di.n_c(len(idx)) + 4) * U * KE, (path, ke, KE, (ke - KE) / KE)


def bussi_args(n_group, dt=DT):
    dof = 3.0 * n_group - 3.0
    return capi.BussiArgs(KT, TAU, dt, dof, 0.3, (dof - 1.0) / 2.0)


# ---- cavb200_force -------------------------------------------------------------------------------------------------------
NO_SMALL = dict(small_n=0, cluster_n=0)
FORCE_CASES = [
    ("k_small", 33, {}), ("k_small", 700, {}), ("k_small", 768, {}),
    ("k_cluster", 769, {}), ("k_cluster", 4096, {}), ("k_cluster", 8192, {}),
    ("k_cluster(8)", 4096, dict(cluster_ctas=8)),  # (up to 2048 particles the default cluster is 8 CTAs already)
    ("variant0", 8192, dict(variant=0, **NO_SMALL)), ("variant0", 262145, dict(variant=0, **NO_SMALL)),
    ("variant1", 8192, dict(variant=1, **NO_SMALL)), ("variant1", 262145, dict(variant=1, **NO_SMALL)),
    ("default", 262145, {}), ("default", 1000001, {}),
]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("sched,N,tuning", FORCE_CASES, ids=[f"{c[0]}-{c[1]}" for c in FORCE_CASES])
def test_force(h, kind, sched, N, tuning):
    s, ph_ref, D, S = inputs(kind, N)
    if tuning:
        h.set_tuning(**tuning)
    d = upload(s, ("pos", "charge", "image"))
    f = capi.DeviceArray.from_numpy(np.full((N, 4), np.nan))
    h.force(d["pos"], d["charge"], d["image"], f, N, s.box, s.L_typeid, PARAMS)
    en, dip, ph = h.force_read()
    check(f"cavb200_force {sched}", s, D, S, ph_ref, dip, en, ph, force=f.numpy())


# ---- cavb200_step --------------------------------------------------------------------------------------------------------
STEP_CASES = [("variant%d" % v, 150001, dict(variant=v)) for v in range(4)] + [
    ("default", 262145, {}), ("default", 500000, {}), ("default", 1000001, {}),
    ("k_small", 33, {}), ("k_small", 768, {}), ("k_cluster", 4096, {}), ("k_cluster", 8192, {}),
]


def run_step(h, s):
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.full((s.N, 4), np.nan))
    h.bussi_reset()
    h.step(d["pos"], d["charge"], d["image"], f, d["vel"], s.N, s.box, s.L_typeid, PARAMS, 0, s.N, bussi_args(s.N))
    en, dip, ph = h.force_read()
    return en, dip, ph, f.numpy(), h.bussi_read()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("sched,N,tuning", STEP_CASES, ids=[f"{c[0]}-{c[1]}" for c in STEP_CASES])
def test_step(h, kind, sched, N, tuning):
    s, ph_ref, D, S = inputs(kind, N)
    if tuning:
        h.set_tuning(**tuning)
    en, dip, ph, force, bo = run_step(h, s)
    check(f"cavb200_step {sched}", s, D, S, ph_ref, dip, en, ph, force=force)
    assert bo["err"] == 0.0
    check_ke(f"cavb200_step {sched}", s.vel, np.arange(N), bo["ke"])


@pytest.mark.timeout(900)
def test_step_16M(h):
    """One case at 16M particles: the default step, the automatic CTA size, the folder CTA."""
    N = 16 * 2 ** 20 + 1
    s, ph_ref, D, S = inputs("adj50", N)
    en, dip, ph, force, bo = run_step(h, s)
    check("cavb200_step default 16M", s, D, S, ph_ref, dip, en, ph, force=force)
    inputs.cache_clear()


# ---- cavb200_force_rank1 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N", [700, 4096, 262145, 1000001])
def test_force_rank1(h, kind, N):
    s, ph_ref, D, S = inputs(kind, N)
    d = upload(s, ("pos", "charge", "image"))
    h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, PARAMS)
    Dq, FL, ph1, n_L = h.rank1_read()
    en, dip, ph = h.force_read()
    count = int((s.typeid == s.L_typeid).sum())
    assert ph1 == ph and (n_L == count or (count > 1 and n_L == 2))  # a merge of records keeps "more than one" as 2
    check("cavb200_force_rank1", s, D, S, ph_ref, dip, en, ph, Dq=Dq, FL=FL)


# ---- cavb200_md_step_one / _fused: the dipole of the positions they have just drifted ---------------------------------
@pytest.mark.parametrize("kind", MD_KINDS)
@pytest.mark.parametrize("N", [4096, 262145])
@pytest.mark.parametrize("wrap", [False, True])
@pytest.mark.parametrize("group", ["window", "mask"])
@pytest.mark.parametrize("md_shape", [0, 1])
def test_md_steps(h, kind, N, wrap, group, md_shape):
    """The documented sequence force_rank1 ; bussi_ke ; md_step_one ; md_step_fused.  After each md call the reference
    is D over the terms of the positions and images the call wrote back."""
    s0, ph_ref, _, _ = inputs(kind, N)
    h.set_tuning(md_shape=md_shape)
    d = upload(s0)
    idx = np.nonzero(s0.typeid != s0.L_typeid)[0].astype(np.uint32)
    if group == "window":
        first, n, d_idx = 0, N, None
    else:
        d_idx = capi.DeviceArray.from_numpy(idx)
        first, n = capi.Handle.GROUP_MASK, len(idx)
        h.group_set(d_idx, n, N)
    h.bussi_reset()
    h.force_rank1(d["pos"], d["charge"], d["image"], N, s0.box, s0.L_typeid, PARAMS)
    h.bussi_ke(d["vel"], d_idx, 0, n)
    check_ke("cavb200_bussi_ke (md sequence)", s0.vel, idx if d_idx is not None else np.arange(N), h.bussi_read()["ke"])
    prev = s0
    for name, fn in (("cavb200_md_step_one", h.md_step_one), ("cavb200_md_step_fused", h.md_step_fused)):
        fn(d["pos"], d["vel"], None, d["charge"], d["image"], N, DT, s0.box, s0.L_typeid, PARAMS, first, n,
           bussi_args(n), wrap=wrap)
        s = synth.System(d["pos"].numpy(), d["vel"].numpy(), s0.charge, d["image"].numpy(), s0.box)
        assert not np.array_equal(s.pos, prev.pos)
        crossed = int(np.any(s.image != prev.image, axis=1).sum())
        if not wrap:
            assert crossed == 0
        elif N >= 262145:
            # tens of particles cross a face per step at this size: the wrap's image update takes part in the reduce
            assert crossed > 0, f"{name}: no particle crossed a face, the wrap branch was not exercised"
        prev = s
        D, S = di.exact_dipole(s.pos, s.charge, s.image, s.box, ph_ref)
        Dq, FL, ph1, _ = h.rank1_read()
        en, dip, ph = h.force_read()
        assert ph1 == ph
        path = f"{name}{'_wrap' if wrap else ''} shape{md_shape}"
        check(path, s, D, S, ph_ref, dip, en, ph, Dq=Dq, FL=FL)
        assert h.bussi_read()["err"] == 0.0


# ---- cavb200_shard_step, one rank --------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N", [4096, 262145])
def test_shard_step_one_rank(h, kind, N):
    s, ph_ref, D, S = inputs(kind, N)
    d = upload(s)
    f = capi.DeviceArray.from_numpy(np.full((N, 4), np.nan))
    h.shard_step(d["pos"], d["charge"], d["image"], f, d["vel"], N, 5000, s.box, s.L_typeid, PARAMS, 0, 0,
                 bussi_args(1, dt=0.0))
    en, dip, ph = h.force_read()
    check("cavb200_shard_step offset 5000", s, D, S, ph_ref, dip, en, ph, force=f.numpy(), index_offset=5000)


# ---- the host-buffer step --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("rank1", [False, True])
def test_step_host_submit_ex(h, kind, rank1):
    N = 262145
    s, ph_ref, D, S = inputs(kind, N)
    bufs = {k: capi.PinnedArray.from_numpy(getattr(s, k)) for k in ("pos", "charge", "image", "vel")}
    force = None if rank1 else capi.PinnedArray.from_numpy(np.full((N, 4), np.nan))
    h.bussi_reset()
    h.step_host_submit_ex(0, bufs["pos"], bufs["charge"], bufs["image"], force, bufs["vel"], N, s.box, s.L_typeid,
                          PARAMS, 0, N, bussi_args(N), h.HOST_RANK1_RESULT if rank1 else 0)
    en, bo, r1 = h.step_host_wait_ex(0)
    _, dip, ph = h.force_read()
    assert r1["photon_idx"] == ph
    check(f"cavb200_step_host_submit_ex{' rank1' if rank1 else ''}", s, D, S, ph_ref, dip, en, ph, Dq=r1["Dq"],
          FL=r1["F_L"], force=None if rank1 else force.array.copy())
    check_ke("cavb200_step_host_submit_ex", s.vel, np.arange(N), bo["ke"])


# ---- kinetic energy: a photon of mass 1 next to masses of 29166 -------------------------------------------------------
@pytest.mark.parametrize("kind", ["adj50", "water_blk50"])
@pytest.mark.parametrize("N", [700, 4096, 262145, 1000001])
@pytest.mark.parametrize("group", ["window", "list"])
def test_bussi_ke(h, kind, N, group):
    s, _, _, _ = inputs(kind, N)
    d = upload(s, ("vel",))
    if group == "window":
        idx = np.arange(N)
        h.bussi_ke(d["vel"], None, 0, N)
    else:
        idx = np.arange(0, N, 3)  # every third particle, the photon among them or not
        h.bussi_ke(d["vel"], capi.DeviceArray.from_numpy(idx.astype(np.uint32)), 0, len(idx))
    check_ke(f"cavb200_bussi_ke {group}", s.vel, idx, h.bussi_read()["ke"])
