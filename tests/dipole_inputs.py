"""Neutral-molecule inputs for the dipole sum, its exact value, and the tolerance a kernel's dipole is held to.

Why these inputs.  The dipole d = sum_{i != photon} c_i (r_i + n_i L) of a system of neutral molecules is a small
remainder of large terms: each molecule adds one bond length times a charge, while each term is a charge times an
unwrapped position of up to |n| L.  `synth.make_system` places particles independently, so there |d| ~ sqrt(N) L and the
condition number sum|t_i| / |d| is ~4e5; here it is >= 1e7 at 1M particles with images of +-50 or more.  On such inputs
a reduction that loses its compensation at one fold is off by 1e2-1e6 ulp, which is still far inside the 1e-10 relative
force tolerance -- and the reference's own serial sum may be off by more than 1e-10 (the shuffled cases).  So the
kernels' dipole is judged against the correctly rounded sum of the same terms, not against the reference.

Layouts are HOOMD's, as in `synth`: pos float64[N,4] (type id in the low 32 bits of w), vel float64[N,4] (mass in w),
charge float64[N], image int32[N,3].  Positions are float32-rounded and inside [-L/2, L/2), charges are float32-exact.

Exact reference.  The terms are formed as the kernels form them (hotpath.cuh unwrap_term, CavityForceCompute.cc:107-109,
124): u = pos + double(image) * L, then t = c * u, each operation rounded once (NumPy's element-wise operations do not
fuse).  D_k = math.fsum(t_k) over every particle except the first of type 'L' is the correctly rounded sum;
S_k = sum |t_k|.

Tolerance.  |d_k - D_k| <= 2 ulp(D_k) + (n_c u)^2 S_k,  u = 2^-53,  n_c = ceil(N / 1024) + 64.
The kernels accumulate each thread's strided subset with error-free two-sums and merge the (hi, lo) pairs in fixed trees
-- Ogita, Rump and Oishi's Sum2 arranged as a tree.  Sum2's bound, |res - s| <= u |s| + gamma_{n-1}^2 sum|p_i|, holds for
any such arrangement with n the longest chain of additions a partial sum takes; n_c bounds that chain generously: at
most ceil(N / 1024) strided terms per thread (no launch shape streams with fewer than 1024 threads once N is past the
one-CTA size; below it a thread takes one term) plus < 64 tree levels (warp, CTA, grid, extra 'L' terms).  The u |s|
part and the final rounding fit in 2 ulp(D).  At 1M particles with images +-1000 that is ~2.1 ulp; at 16M with images
+-50 ~40 ulp, against ~3.6e5 ulp for a reduction with no low word there and the 1e2-1e6 ulp that
tests/test_dipole_exact.py prints for the other inputs.

Downstream of d everything follows the reference's operation order (hotpath.cuh finalize, CavityForceCompute.cc:174-207;
apply_stream / force_of, :188-200), so `finalize` and `force_rows` restate it and the kernels must match them bit for bit
when fed the kernel's own d.
"""
from __future__ import annotations

import math

import numpy as np

from cav_hoomd_b200 import synth

U = 2.0 ** -53
BOND = 2.1                              # Bohr
Q_DIMER = 0.5                           # +-q dimers
Q_WATER = float(np.float32(0.4238))     # -2q, +q, +q
Q_EXTRA_L = 0.75                        # further 'L' particles, in +- pairs at one position
MASS_MOL = synth.MASS_O                 # 29166
MASS_L = 1.0
BIG_PHOTON_CHARGE = float(np.float32(0.7))
BIG_PHOTON_IMAGE = (100000, -100000, 100000)
OMEGAC, G, PHMASS = 0.01, 1e-3, 1.0

# grid strides (CTAs x threads) of default launch shapes on a 148-SM device: the folder step (295 x 320 / 352 / 384, the
# CTA size auto_threads picks) and the fused force kernel (296 x 384): an 'L' particle this far behind the photon lands
# in the photon's thread
STRIDES = (295 * 320, 295 * 352, 295 * 384, 296 * 384)


def n_c(N: int) -> int:
    return -(-int(N) // 1024) + 64


def _f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def _inside(x, L):
    """float32-round into [-L/2, L/2): a value the rounding pushed onto a face is moved one float32 step inwards."""
    x = _f32(x)
    hi = float(np.nextafter(np.float32(L / 2), np.float32(0)))
    lo = float(np.nextafter(np.float32(-L / 2), np.float32(0)))
    return np.where(x >= L / 2, hi, np.where(x < -L / 2, lo, x))


def photon_slot(N: int, where: str) -> int:
    if where == "first":
        return 0
    if where == "last":
        return N - 1
    if where == "cta":  # a multiple of 256, 384, 768 and 1024 threads: the first particle of some CTA
        for b in (3072, 768, 64):
            if b < N // 2:
                return b
        return 0
    raise ValueError(where)


def extra_L_slots(N: int, ph: int) -> list:
    """Further 'L' particles: the photon's warp, two other CTAs, the photon's thread under the default strides, N - 1.
    An even number of them (they come in +- pairs): when the count is odd, the second-to-last slot goes, so that the
    particle at N - 1 stays."""
    want = [ph + 1, ph + 1029, ph + 1157] + [ph + s for s in STRIDES] + [N - 1]
    slots = sorted({i for i in want if ph < i < N})
    if len(slots) % 2:
        del slots[-2 if len(slots) > 1 else -1]
    return slots


def make_molecules(N: int, *, size: int = 2, images: int = 50, order: str = "adjacent", photon: str = "last",
                   extra_L: bool = False, big_photon: bool = False, zero: bool = False, seed: int = 0) -> synth.System:
    """N particles: neutral molecules of `size` atoms (2: +-q dimers, 3: water-like -2q, +q, +q) plus the photon and,
    with `extra_L`, further 'L' particles in +- charge pairs.  Atoms left over when N does not divide are uncharged.

    images  first atoms take image flags in [-images, images]; a partner that falls across a face is wrapped back and
            its image adjusted, so the unwrapped molecule stays intact
    order   "adjacent" (partners next to each other), "blocked" (all first atoms, then all second atoms, ...: partners
            N/size apart, in different CTAs) or "shuffled" (a seeded random permutation)
    photon  "first", "last" or "cta" (index 3072 / 768 / 64, a CTA boundary); it is the first particle of type 'L'
    big_photon  the photon has charge 0.7 and image (1e5, -1e5, 1e5): a term ~1e5 |d| that must stay out of d
    zero    partners sit at identical unwrapped positions: d = 0 exactly
    """
    rng = np.random.Generator(np.random.PCG64(7919 * seed + 104729 * size + images + 31 * N))
    L = (max(N, 1) / synth.NUMBER_DENSITY) ** (1.0 / 3.0)
    box = np.array([L, L, L])
    ph = photon_slot(N, photon)
    extra = extra_L_slots(N, ph) if extra_L else []
    special = [ph] + extra
    n_atoms = N - len(special)
    n_mol = n_atoms // size

    # molecules: first atom inside the box, partners at a bond vector (or on top of it), wrapped back with their image
    x0 = _inside(rng.uniform(-L / 2, L / 2, size=(n_mol, 3)), L)
    n0 = rng.integers(-images, images + 1, size=(n_mol, 3)).astype(np.int32)
    xs, ns = [x0], [n0]
    for _ in range(size - 1):
        if zero:
            xs.append(x0.copy())
            ns.append(n0.copy())
            continue
        b = rng.standard_normal((n_mol, 3))
        b *= BOND / np.linalg.norm(b, axis=1)[:, None]
        raw = x0 + b
        shift = np.floor((raw + L / 2) / L)
        xs.append(_inside(raw - shift * L, L))
        ns.append((n0 + shift).astype(np.int32))
    if size == 2:
        qs = [Q_DIMER, -Q_DIMER]
    elif size == 3:
        qs = [-2.0 * Q_WATER, Q_WATER, Q_WATER]
    else:
        raise ValueError(size)
    ax = np.stack(xs, axis=1)                                   # [mol, atom, 3]
    an = np.stack(ns, axis=1)
    aq = np.broadcast_to(np.array(qs), (n_mol, size))
    if order == "blocked":
        ax, an, aq = (np.swapaxes(a, 0, 1) for a in (ax, an, aq))
    ax, an, aq = ax.reshape(-1, 3), an.reshape(-1, 3), aq.reshape(-1)
    if order == "shuffled":
        p = rng.permutation(len(aq))
        ax, an, aq = ax[p], an[p], aq[p]
    elif order not in ("adjacent", "blocked"):
        raise ValueError(order)
    pad = n_atoms - len(aq)                                     # uncharged filler atoms
    ax = np.concatenate([ax, _inside(rng.uniform(-L / 2, L / 2, size=(pad, 3)), L)])
    an = np.concatenate([an, np.zeros((pad, 3), np.int32)])
    aq = np.concatenate([aq, np.zeros(pad)])

    pos = np.empty((N, 4))
    vel = np.empty((N, 4))
    charge = np.empty(N)
    image = np.empty((N, 3), np.int32)
    typeid = np.zeros(N, np.int32)
    mol = np.ones(N, bool)
    mol[special] = False
    pos[mol, :3], image[mol], charge[mol] = ax, an, aq
    typeid[mol] = 0
    vel[mol, :3] = rng.standard_normal((n_atoms, 3)) * math.sqrt(synth.KT_100K / MASS_MOL)
    vel[mol, 3] = MASS_MOL

    K = PHMASS * OMEGAC * OMEGAC
    pos[ph, :3] = _f32(rng.standard_normal(3) * math.sqrt(synth.KT_100K / K))
    charge[ph] = BIG_PHOTON_CHARGE if big_photon else 0.0
    image[ph] = BIG_PHOTON_IMAGE if big_photon else (0, 0, 0)
    for j in range(0, len(extra), 2):  # a +- pair at one position: terms of 1e3 L that cancel exactly
        x = _inside(rng.uniform(-L / 2, L / 2, size=3), L)
        n = rng.integers(-1000, 1001, size=3).astype(np.int32)
        for i, c in ((extra[j], Q_EXTRA_L), (extra[j + 1], -Q_EXTRA_L)):
            pos[i, :3], image[i], charge[i] = x, n, c
    typeid[special] = synth.L_TYPEID
    vel[special, :3] = rng.standard_normal((len(special), 3)) * math.sqrt(synth.KT_100K / MASS_L)
    vel[special, 3] = MASS_L
    pos[:, 3] = synth.typeid_to_w(typeid)
    return synth.System(pos, vel, charge, image, (L, L, L))


# the input kinds the tests run, by name
KINDS = {
    "adj50": dict(size=2, images=50, order="adjacent", photon="last"),
    "shuf1000": dict(size=2, images=1000, order="shuffled", photon="first", extra_L=True),
    "water_blk50": dict(size=3, images=50, order="blocked", photon="cta"),
    "bigph": dict(size=2, images=1000, order="adjacent", photon="cta", extra_L=True, big_photon=True),
    "zero": dict(size=2, images=50, order="shuffled", photon="last", zero=True),
}
# the builder options not in KINDS, for the CPU checks of the builders and of the oracle
MORE_KINDS = {
    "adj1": dict(size=2, images=1, order="adjacent", photon="first"),
    "shuf50": dict(size=2, images=50, order="shuffled", photon="cta"),
    "blk1000": dict(size=2, images=1000, order="blocked", photon="last", extra_L=True),
    "water_adj1000": dict(size=3, images=1000, order="adjacent", photon="first", extra_L=True),
    "water_shuf1": dict(size=3, images=1, order="shuffled", photon="last"),
    "water_zero": dict(size=3, images=1000, order="blocked", photon="cta", zero=True),
}


def build(kind: str, N: int) -> synth.System:
    return make_molecules(N, **{**MORE_KINDS, **KINDS}[kind])


# ---- exact reference --------------------------------------------------------------------------------------------------
def photon_index(s: synth.System) -> int:
    isL = np.nonzero(s.typeid == s.L_typeid)[0]
    return int(isL[0]) if len(isL) else -1


def unwrapped(pos, image, box) -> np.ndarray:
    """u = pos + double(image) * L, one rounding each (unwrap_term)."""
    return pos[:, :3] + image.astype(np.float64) * np.asarray(box, dtype=np.float64)


def dipole_terms(pos, charge, image, box, photon: int) -> np.ndarray:
    """t = c * u of every particle but the photon, float64[N - 1, 3] (float64[N, 3] without a photon)."""
    t = charge[:, None] * unwrapped(pos, image, box)
    return np.delete(t, photon, axis=0) if photon >= 0 else t


def exact_dipole(pos, charge, image, box, photon: int):
    """-> (D, S): the correctly rounded dipole and sum |t|, per component."""
    t = dipole_terms(pos, charge, image, box, photon)
    D = np.array([math.fsum(t[:, k]) for k in range(3)])
    S = np.array([math.fsum(np.abs(t[:, k])) for k in range(3)])
    return D, S


def tolerance(D, S, N: int) -> np.ndarray:
    return 2.0 * np.spacing(np.abs(D)) + (n_c(N) * U) ** 2 * S


def ulps(d, D) -> np.ndarray:
    """|d - D| in units of ulp(D)."""
    with np.errstate(over="ignore", divide="ignore"):
        return np.abs(np.asarray(d) - D) / np.spacing(np.abs(D))


# ---- downstream of d: the reference's operation order -----------------------------------------------------------------
def constants(omegac=OMEGAC, g=G, phmass=PHMASS) -> dict:
    """The host-evaluated constants (capi.Params.make, api.cu fill_force_constants)."""
    K = phmass * omegac * omegac
    return dict(g=g, K=K, gk=g / K, half_K=0.5 * K, half_g2K=0.5 * (g * g / K))


def finalize(d, q, c: dict):
    """hotpath.cuh finalize (CavityForceCompute.cc:174-183, 203) on the dipole d and the photon's unwrapped position q:
    -> (energies[3], Dq[2], F_L[3]), every operation rounded as the kernel rounds it."""
    d = [float(x) for x in d]
    q = [float(x) for x in q]
    qq = (q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]
    dq = (d[0] * q[0] + d[1] * q[1]) + 0.0
    dd = (d[0] * d[0] + d[1] * d[1]) + 0.0
    en = np.array([c["half_K"] * qq, c["g"] * dq, c["half_g2K"] * dd])
    Dq = np.array([q[0] + c["gk"] * d[0], q[1] + c["gk"] * d[1]])
    FL = np.array([(-c["K"]) * q[k] + -(c["g"] * (d[k] if k < 2 else 0.0)) for k in range(3)])
    return en, Dq, FL


def force_rows(charge, typeid, L_typeid, photon: int, Dq, FL, c: dict) -> np.ndarray:
    """The force array (force_of): (-g c_i) Dq for molecules, F_L for the photon, zero for other 'L' particles."""
    f = np.zeros((len(charge), 4))
    s = (-c["g"]) * charge
    f[:, 0] = s * Dq[0]
    f[:, 1] = s * Dq[1]
    f[typeid == L_typeid] = 0.0
    if photon >= 0:
        f[photon, :3] = FL
    return f


def propagated(D, tol, q, charge, c: dict) -> dict:
    """Bounds on |x(d) - x(D)| for every quantity x after d, given |d_k - D_k| <= tol_k: the first-order change plus
    4 u times the magnitudes the two roundings of x work on."""
    en, Dq, FL = finalize(D, q, c)
    t2 = np.asarray(tol, dtype=np.float64)[:2]
    d2 = np.abs(np.asarray(D, dtype=np.float64)[:2])
    q3 = np.abs(np.asarray(q, dtype=np.float64))
    g = abs(c["g"])
    dq = c["gk"] * t2 + 4 * U * (np.abs(Dq) + c["gk"] * d2)
    return dict(
        energies=np.array([0.0,
                           g * float(q3[:2] @ t2) + 4 * U * g * float(q3[:2] @ d2),
                           c["half_g2K"] * float((2 * d2 + t2) @ t2) + 4 * U * c["half_g2K"] * float(d2 @ d2)]),
        Dq=dq,
        FL=np.append(g * t2 + 4 * U * (c["K"] * q3[:2] + g * d2), 0.0),
        force=np.abs(c["g"] * charge)[:, None] * dq[None, :])


# ---- a model of the kernels' reduction order, for the CPU tests -------------------------------------------------------
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def model_sum(t: np.ndarray, threads: int, mode: str = "kernel") -> float:
    """Each of `threads` threads sums its grid-stride subset of t, then the threads' pairs are merged in a pairwise tree
    (lanes l and l + P/2, as the butterflies pair them).  mode "kernel": two_sum_acc / pair_add as written
    (cavb200_internal.cuh); "no_lo": plain sums, no low word anywhere; "drop_fold": the per-thread low words are kept
    but pair_add drops the incoming one (lo + 0.0 instead of lo + lo2)."""
    n = len(t)
    steps = max(-(-n // threads), 1)
    x = np.zeros(steps * threads)
    x[:n] = t
    x = x.reshape(steps, threads)
    hi = np.zeros(threads)
    lo = np.zeros(threads)
    for row in x:
        if mode == "no_lo":
            hi = hi + row
        else:
            hi, e = _two_sum(hi, row)
            lo = lo + e
    P = 1 << max(threads - 1, 0).bit_length()
    hi = np.concatenate([hi, np.zeros(P - threads)])
    lo = np.concatenate([lo, np.zeros(P - threads)])
    while len(hi) > 1:
        h = len(hi) // 2
        if mode == "no_lo":
            hi = hi[:h] + hi[h:]
            lo = lo[:h]
            continue
        s, e = _two_sum(hi[:h], hi[h:])
        lo = (lo[:h] + e) + lo[h:] if mode == "kernel" else lo[:h] + e
        hi = s
    return float(hi[0] + lo[0])
