"""The scalar tracker's record (cavb200_track_record / _record_from, csrc/track.cu), field by field: what each field must
equal bit for bit, the exact value it must be near, and the systems the tests record on.

Field contract (include/cavb200.h documents the layout):
  [0]      the timestep argument
  [1..3]   d, [7..9] the energies: bit for bit cavb200_force_read of the handle that holds the force result, read right
           after the step; d within the Sum2 bound of tests/dipole_inputs.py of the correctly rounded dipole D
  [4..6]   q: bit for bit the photon's unwrapped position pos + image L of the arrays the step left (the q the energies
           were formed from: dipole_inputs.finalize(d, q) gives [7..9] bit for bit)
  [10]     C(t) = fl(fl(fl(r_x d_x) + r_y d_y) + r_z d_z), no fused multiply-add, on the recorded d and the stored
           reference r (`autocorr`); within gamma_3 sum |r_k d_k| of the exact dot product of those two vectors, and within
           `autocorr_bound` of the exact D(ref) . D(t) of the snapshots
  [11]     fl(fl(0.5 m) fl(fl(v_x^2 + v_y^2) + v_z^2)) of the photon's velocity after the full step (`photon_ke`), within
           gamma_3 of the exact value; 0 without a photon on this rank; NaN while a second half kick is pending
  [12..14] KE, alpha, cumulative reservoir: bit for bit cavb200_bussi_read of the handle that ran the thermostat; KE within
           (n_c + 4) u KE of math.fsum of 1/2 m |v|^2 over the group; NaN without a thermostat handle ([12] also while a
           half kick is pending)
  [15]     the photon's global index (force_read's), -1 without one

`record` restates k_track_record in NumPy from those sources; the GPU tests compare every record with it.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

import dipole_inputs as di
from cav_hoomd_b200 import synth

U = di.U
NAN = float("nan")
GAMMA3 = 3 * U / (1 - 3 * U)
OLD_TOL = 1e-10  # the relative tolerance tests/test_trackers_gpu.py holds d and C(t) to


# ---- the kernel's arithmetic, restated --------------------------------------------------------------------------------
def autocorr(ref, d) -> float:
    """[10]: fl(fl(fl(r_x d_x) + r_y d_y) + r_z d_z), each product and sum rounded on its own (no FMA)."""
    c = 0.0
    for k in range(3):
        c = float(np.float64(c) + np.float64(float(ref[k]) * float(d[k])))
    return c


def autocorr_fma(ref, d) -> float:
    """A kernel that let the compiler contract C(t) into fused multiply-adds (a mutant: must miss the contract)."""
    c = 0.0
    for k in range(3):
        c = float(Fraction(float(ref[k])) * Fraction(float(d[k])) + Fraction(c))
    return c


def dot_exact(a, b) -> Fraction:
    return sum((Fraction(float(x)) * Fraction(float(y)) for x, y in zip(a, b)), Fraction(0))


def autocorr_rounding_bound(ref, d) -> float:
    """|autocorr(ref, d) - ref . d| <= gamma_3 sum |r_k d_k| (recursive summation of three rounded products)."""
    return GAMMA3 * float(np.sum(np.abs(np.asarray(ref, float) * np.asarray(d, float)))) * (1 + 4 * U)


def autocorr_bound(D0, tol0, D, tol) -> float:
    """Bound on |C - D0 . D| (exact) for C = autocorr(d0, d) with |d0_k - D0_k| <= tol0_k and |d_k - D_k| <= tol_k:
    the first-order change, the product of the two errors, and the rounding of the dot product itself."""
    D0, tol0, D, tol = (np.abs(np.asarray(x, float)) for x in (D0, tol0, D, tol))
    prop = float(np.sum(D0 * tol + tol0 * D + tol0 * tol))
    return prop * (1 + 4 * U) + autocorr_rounding_bound(D0 + tol0, D + tol)


def photon_ke(v) -> float:
    """[11]: fl(fl(0.5 m) fl(fl(v_x^2 + v_y^2) + v_z^2)) of one Scalar4 velocity row (vx, vy, vz, m)."""
    x, y, z, m = (np.float64(a) for a in v[:4])
    v2 = (x * x + y * y) + z * z
    return float((np.float64(0.5) * m) * v2)


def photon_ke_exact(v) -> Fraction:
    x, y, z, m = (Fraction(float(a)) for a in v[:4])
    return Fraction(1, 2) * m * (x * x + y * y + z * z)


def group_ke_bound(KE: float, n: int) -> float:
    return (di.n_c(n) + 4) * U * KE


def group_ke_exact(vel, idx) -> float:
    v = vel[idx]
    return math.fsum(0.5 * v[:, 3] * (v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2]))


# ---- k_track_record in NumPy --------------------------------------------------------------------------------------------
def record(timestep, force, q, vel, ref, bussi=None, offset: int = 0, pending: bool = False) -> np.ndarray:
    """The 16 doubles k_track_record appends.
    force   (energies[3], dipole[3], photon_idx) as cavb200_force_read returns them for the handle holding the result
    q       the photon's unwrapped position (zeros without a photon)
    vel     the velocity array (Scalar4 rows) passed to the record, or None
    ref     the stored reference dipole
    bussi   cavb200_bussi_read of the thermostat handle as a dict, or None (no thermostat handle)
    offset  the global index of vel's row 0 (cavb200_shard_step's index_offset)
    pending the velocities lack the deferred second half kick (CAVB200_TRACK_VELOCITIES_PENDING)"""
    en, d, ph = force
    r = np.zeros(16)
    r[0] = float(timestep)
    r[1:4] = d
    r[4:7] = q
    r[7:10] = en
    r[10] = autocorr(ref, d)
    ke = 0.0
    if vel is not None and ph >= 0 and 0 <= ph - offset < len(vel):
        ke = photon_ke(vel[ph - offset])
    r[11] = NAN if pending else ke
    r[12] = bussi["ke"] if bussi is not None and not pending else NAN
    r[13] = bussi["alpha"] if bussi is not None else NAN
    r[14] = bussi["cumulative"] if bussi is not None else NAN
    r[15] = float(ph)
    return r


def bits(x) -> np.ndarray:
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def same_bits(a, b) -> bool:
    """Bit-for-bit equal, with every NaN equal to every NaN (the kernel's NaN need not be NumPy's)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(bits(a[~na]), bits(b[~nb])))


# ---- the systems -------------------------------------------------------------------------------------------------------
def make_system(N: int, photon: str = "last", kind: str = "adj50", seed: int = 0) -> synth.System:
    """Neutral molecules (dipole_inputs.make_molecules): d cancels heavily, so a dipole of the wrong step or handle cannot
    hide in a relative tolerance.  photon: "last", "middle" (a CTA boundary), or "absent" (the photon becomes an
    uncharged molecular particle: no particle of type 'L')."""
    opts = dict(di.KINDS[kind])
    opts["photon"] = {"last": "last", "middle": "cta", "absent": "last"}[photon]
    s = di.make_molecules(N, seed=seed, **opts)
    if photon == "absent":
        ph = di.photon_index(s)
        t = s.typeid.copy()
        t[ph] = 0
        s.pos[:, 3] = synth.typeid_to_w(t)
        s.charge[ph] = 0.0
        s.vel[ph, 3] = di.MASS_MOL
        s = synth.System(s.pos, s.vel, s.charge, s.image, s.box)
    return s


def photon_q(pos, image, box, ph: int) -> np.ndarray:
    return di.unwrapped(pos, image, box)[ph] if ph >= 0 else np.zeros(3)
