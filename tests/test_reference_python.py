"""Pin of the Python-side oracle (SURVEY.md 8a rows a12-a14, 8f.4) on the REFERENCE'S OWN PYTHON.

The reference's src/cavitymd/{analysis,utils,cavity_force_python}.py are executed unmodified, from where they
lie under /root/reference, under a stub `hoomd` module (oracle/refpy.py).  Every NumPy restatement in
oracle/oracle.py must agree with them BIT FOR BIT on the same inputs, and the committed fixture
tests/golden/fkt.npz (what the GPU parity tests compare against on the GPU box, where /root/reference does
not exist) must be exactly what the imported reference produces.  Skipped where the reference tree is absent.

The tests at the end need no reference tree: they hold the same restatements bit for bit to the reference's own
outputs stored in tests/golden/fkt.npz (generate_fibonacci_sphere for 50 and 64 points, compute_density_field on
six frames of a 401-particle system, compute_field_autocorr over every origin and lag of those frames).
"""
import os

import numpy as np
import pytest

from cav_hoomd_b200 import synth
from oracle import oracle as O
from oracle import refpy

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ref():
    if not refpy.available():
        pytest.skip("the reference source tree is not present (CAVB_REFERENCE_ROOT); the stored outputs carry the pin")
    return refpy.load()


@pytest.fixture(scope="module")
def fkt():
    return np.load(os.path.join(GOLD, "fkt.npz"))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.mark.parametrize("n", [2, 50, 64, 100, 257])
def test_fibonacci_sphere_bitwise(ref, n):
    """reference src/cavitymd/analysis.py:50-66"""
    assert np.array_equal(_bits(ref.analysis.generate_fibonacci_sphere(n)), _bits(O.numpy_fibonacci_sphere(n)))
    assert np.array_equal(_bits(ref.analysis.generate_fibonacci_sphere(n)), _bits(synth.fibonacci_sphere(n)))


@pytest.mark.parametrize("n_mol,K", [(1, 3), (33, 8), (400, 50), (5000, 64)])
def test_density_field_bitwise(ref, n_mol, K):
    """reference src/cavitymd/analysis.py:34-47 (all particles, wrapped positions, photon included)"""
    s = synth.make_system(n_mol, replica=4)
    kvec = ref.analysis.generate_fibonacci_sphere(K) * 1.3
    pos = np.ascontiguousarray(s.pos[:, :3])
    a = ref.analysis.compute_density_field(refpy.Snapshot(pos), kvec)
    b = O.numpy_density_field(pos, kvec)
    assert np.array_equal(_bits(a.real.copy()), _bits(b.real.copy())) and np.array_equal(_bits(a.imag.copy()), _bits(b.imag.copy()))
    # float32 positions, the way a GSD trajectory holds them: np.dot(float32, float64) widens exactly
    pos32 = pos.astype(np.float32)
    a32 = ref.analysis.compute_density_field(refpy.Snapshot(pos32), kvec)
    b32 = O.numpy_density_field(pos32.astype(np.float64), kvec)
    assert np.allclose(a32, b32, rtol=1e-13, atol=1e-9)


def test_field_autocorr_bitwise(ref):
    """reference src/cavitymd/analysis.py:359-364 (ndarray branch: mean_k Re(rho0 conj rho_t))"""
    rng = np.random.default_rng(3)
    f0 = rng.standard_normal(64) + 1j * rng.standard_normal(64)
    ft = rng.standard_normal(64) + 1j * rng.standard_normal(64)
    fa = ref.analysis.FieldAutocorrelationTracker.compute_field_autocorr
    assert fa(None, f0, ft) == O.numpy_field_autocorr(f0, ft)


@pytest.mark.parametrize("n_mol", [1, 100, 3001])
def test_total_dipole_bitwise(ref, n_mol):
    """reference src/cavitymd/analysis.py:18-31 + utils.py unwrap_positions"""
    s = synth.make_system(n_mol, replica=9)
    pos = np.ascontiguousarray(s.pos[:, :3])
    snap = refpy.Snapshot(pos, s.image, s.charge, box=np.array(s.box))
    a = ref.analysis.compute_total_dipole_moment(snap)
    b = O.numpy_total_dipole(pos, s.image, s.charge, np.array(s.box))
    assert np.array_equal(_bits(a), _bits(b))
    assert np.array_equal(_bits(ref.utils.unwrap_positions(pos, s.image, np.array(s.box))),
                          _bits(O.numpy_unwrap(pos, s.image, np.array(s.box))))


def test_committed_fkt_fixture_is_the_reference_output(ref):
    """tests/golden/fkt.npz == what the imported reference computes from the stored frames (bitwise)."""
    g = np.load(os.path.join(GOLD, "fkt.npz"))
    frames, kvec = g["frames"], g["kvec"]
    assert np.array_equal(_bits(kvec), _bits(ref.analysis.generate_fibonacci_sphere(len(kvec)) * 1.0))
    rho = np.array([ref.analysis.compute_density_field(refpy.Snapshot(frames[t]), kvec) for t in range(len(frames))])
    assert np.array_equal(_bits(rho.view(np.float64)), _bits(g["rho"].view(np.float64)))
    fa = ref.analysis.FieldAutocorrelationTracker.compute_field_autocorr
    T, L = g["F"].shape
    F = np.array([[fa(None, rho[o], rho[o + l]) if o + l < T else np.nan for l in range(L)] for o in range(T)])
    assert np.array_equal(F, g["F"], equal_nan=True)
    assert np.array_equal(_bits(g["fib64"]), _bits(ref.analysis.generate_fibonacci_sphere(64)))


@pytest.mark.parametrize("n_mol,photon", [(40, "last"), (500, "middle"), (2000, "first")])
def test_python_fallback_force_agrees_with_cpp_semantics(ref, coracle, n_mol, photon):
    """The reference's pure-Python force (src/cavitymd/cavity_force_python.py:65-149), run as shipped on one frame,
    against the C++ class's semantics (oracle).  It looks for typeid == 1 (:75) and includes the photon in the
    dipole sum (harmless: charge 0), so the frame labels the photon 1 for it; NumPy's dot sums in another order
    than the serial loop of CavityForceCompute.cc:120-126, hence a tolerance."""
    s = synth.make_system(n_mol, replica=21, photon=photon)
    tid = s.typeid
    tid_py = np.where(tid == s.L_typeid, 1, 0)
    pos = np.ascontiguousarray(s.pos[:, :3])
    py = refpy.python_cavity_force(pos, s.image, s.charge, tid_py, np.array(s.box), 0.01, 1e-3)
    c = coracle.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, 0.01, 1e-3)
    scale = np.abs(c["force"]).max()
    assert np.abs(py["force"] - c["force"][:, :3]).max() <= 1e-11 * scale
    assert np.allclose(py["energies"], c["energies"], rtol=1e-11)
    # and the repo's NumPy restatement of that file is the same arithmetic
    b = O.numpy_cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, 0.01, 1e-3)
    assert np.allclose(py["force"], b["force"], rtol=1e-13, atol=1e-300)
    assert np.allclose(py["energies"], b["energies"], rtol=1e-13)


# ---- the same pins on the reference's stored outputs (no reference tree needed) ---------------------------------
@pytest.mark.parametrize("n,key", [(50, "kvec"), (64, "fib64")])
def test_fibonacci_sphere_matches_stored_reference(fkt, n, key):
    """reference src/cavitymd/analysis.py:50-66; kvec was stored as generate_fibonacci_sphere(50) * 1.0 (exact)"""
    assert np.array_equal(_bits(fkt[key]), _bits(O.numpy_fibonacci_sphere(n)))
    assert np.array_equal(_bits(fkt[key]), _bits(synth.fibonacci_sphere(n)))


def test_density_field_matches_stored_reference(fkt):
    """reference src/cavitymd/analysis.py:34-47 on every stored frame and wave vector"""
    for t, frame in enumerate(fkt["frames"]):
        b = O.numpy_density_field(frame, fkt["kvec"])
        assert np.array_equal(_bits(b.view(np.float64)), _bits(fkt["rho"][t].view(np.float64)))


def test_field_autocorr_matches_stored_reference(fkt):
    """reference src/cavitymd/analysis.py:359-364 for every origin and lag of the stored density fields"""
    rho, F = fkt["rho"], fkt["F"]
    T, L = F.shape
    ours = np.array([[O.numpy_field_autocorr(rho[o], rho[o + l]) if o + l < T else np.nan for l in range(L)]
                     for o in range(T)])
    assert np.array_equal(ours, F, equal_nan=True)
