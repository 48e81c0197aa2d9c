"""Exact references, launch geometry and error bounds for the density field rho[t][k] = sum_j exp(i k.r_j(t))
(cavb200_rhok, cavb200_rhok_f32) and its autocorrelation F[o][l] = mean_k Re(rho[o][k] conj rho[o+l][k])
(cavb200_fkt) -- csrc/rhok.cu.  CPU only; the GPU side is tests/test_fkt_exact_gpu.py.

The argument.  k_rhok forms kr = fma(z, kz, fma(y, ky, x kx)) (rhok.cu, rhok_walk).  NumPy has no FMA, so `fma`
emulates it exactly: the product a b = ph + pl by TwoProduct (Veltkamp/Dekker split), then the correctly rounded
ph + pl + c by TwoSum and a round-to-odd of the low part (Boldo & Melquiond, "Emulation of FMA and correctly rounded
sums: proved algorithms using rounding to odd", IEEE TC 2008).  Valid for |a b| and |c| in the normal range with
no overflow, which every input here is.

The exact reference R.  Each term is (cos, sin) of that double argument in np.longdouble (x86 80-bit cosl / sinl:
exact argument reduction at every magnitude), split into hi + lo doubles and summed by math.fsum.  The long double
value is within 2^-64 |term| <= 5.5e-20 of the true cosine, and fsum rounds the exact sum of the pieces once, so
|R - sum_j exp(i kr_j)| <= N 5.5e-20 + 1/2 ulp(R) (`ref_slack`).

The kernel's summation order (`model_sum`).  Per wave vector k, of slab s (K is cut into slabs of threads*4), with
KQ = ceil(Ks / 4) k-quads and groups = threads // KQ particle groups:
  * CTA (p, t) walks tiles [p tiles_per, (p + 1) tiles_per) of frame t; thread pg walks local particles
    pg, pg + groups, ... of each tile, its chain carried across the CTA's tiles;
  * the chains of a CTA are folded in group order 0, 1, ..., groups - 1;
  * with P > 1 slices, k_rhok_fold: lane L adds slices L, L + 32, ... in order, then the xor tree 16, 8, 4, 2, 1.

The bound.  One pair (particle j, k) on the table path does re = fma(-s, S, fma(c, C, re)): the rotated term has
error eps_j <= 2.4e-16 against the exact exp(i kr_j) (DESIGN.md 3.4, which counts both fused roundings at magnitude 1),
and the two roundings into the accumulator add at most u |acc1| + u |acc2| <= u (2 |S_new| + 1) with S_new the partial
sum after the pair (|acc1| <= |S_new| + 1).  Taking the "+1" into eps_j, a pair costs eps_j + 2 u |S_new|.  A particle
with |kr| >= 2^20 takes CUDA's sincos (2 ulp of 1 each: eps_j = 2^-51) and one rounding re += cs, u |S_new|.  Every
fold addition costs u |result|.  Summing, the kernel's error is at most
    sum_j eps_j + u (2 sum_chains |S| + sum_folds |S|) + (second order),
and the tolerance is sum_j eps_j + c u sum |partial sums of the model| + ref_slack with c = 3: 1.5x the chain
coefficient, 3x the fold coefficient.  The margin covers the difference between the model's partial sums (plain
float64 additions of the rounded terms) and the kernel's, which is itself of order u sum |S| relative to |S|, i.e.
second order.  This a-posteriori bound grows like the random-walk size of the partial sums (~sqrt of a chain's
length per step), where the older 1e-13 N grew like N: at 1M particles and the bench shape it is roughly 10-100x
tighter (an estimate from the geometry).

F*.  For one (o, l): math.fsum of the exact products a_r b_r, a_i b_i (TwoProduct: four doubles per k), divided by K
and rounded once (`fkt_exact`).  k_fkt sums K contracted terms in order, so its error is at most
gamma_{K+1} sum_k (|a_r b_r| + |a_i b_i|) / K plus the rounding of the division (`fkt_bound`).
"""
import functools
import math
import os
from fractions import Fraction

import numpy as np

U = 2.0 ** -53
EPS_TABLE = 2.4e-16          # per component, table path (DESIGN.md 3.4)
EPS_LIBRARY = 2.0 * 2.0 ** -52  # per component, CUDA sincos for |kr| >= 2^20: 2 ulp of 1
HUGE = 2.0 ** 20
C_BOUND = 3.0

TILE = 512
KB = 4
CTA = 256
GRID_PER_SM = 24
TCHUNK = 65535

# -------------------------------------------------------------------------------------------------------------------
# exact FMA
# -------------------------------------------------------------------------------------------------------------------
_SPLIT = 134217729.0  # 2^27 + 1


def two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def two_product(a, b):
    """a b = p + e exactly (Dekker), for |a|, |b| < 2^996."""
    p = a * b
    t = _SPLIT * a
    ah = t - (t - a)
    al = a - ah
    t = _SPLIT * b
    bh = t - (t - b)
    bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def _round_to_odd_sum(a, b):
    """a + b rounded to odd (the neighbour with an odd last significand bit when a + b is not representable)."""
    s, e = two_sum(a, b)
    even = (s.view(np.int64) & 1) == 0
    move = (e != 0) & even
    return np.where(move, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)


def fma(a, b, c):
    """Correctly rounded a b + c, elementwise on float64 arrays (Boldo & Melquiond)."""
    a, b, c = (np.asarray(v, dtype=np.float64) for v in (a, b, c))
    uh, ul = two_product(a, b)
    th, tl = two_sum(c, uh)
    v = _round_to_odd_sum(tl, ul)
    return th + v


def kernel_argument(pos, kvec):
    """kr[k, j] = fma(z, kz, fma(y, ky, x kx)) for positions [N, 3] and wave vectors [K, 3]."""
    x, y, z = (pos[:, c][None, :] for c in range(3))
    kx, ky, kz = (kvec[:, c][:, None] for c in range(3))
    return fma(z, kz, fma(y, ky, x * kx))


def fraction_fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


# -------------------------------------------------------------------------------------------------------------------
# launch geometry (rhok.cu: rhok_slices, rhok_launch)
# -------------------------------------------------------------------------------------------------------------------
def rhok_slices(tiles, T, slots):
    pmax = (GRID_PER_SM * slots + T - 1) // T
    pmax = max(1, min(pmax, tiles))
    best, best_cost = 1, 0.0
    for P in range(1, pmax + 1):
        waves = (P * T + slots - 1) // slots
        per = (tiles + P - 1) // P
        cost = float(waves) * (float(per) + 0.25)
        if P == 1 or cost < best_cost:
            best, best_cost = P, cost
    return best


def geometry(N, T, K, num_sms, threads=CTA):
    """The schedule of one cavb200_rhok call: chunks of frames (P, tiles_per each), slabs of wave vectors
    (k0, Ks, KQ, groups) and the kernel launches it makes."""
    threads = threads if threads in (128, 256) else CTA
    if N == 0 or T == 0 or K == 0:
        return {"chunks": [], "slabs": [], "launches": 0, "threads": threads, "tiles": 0}
    tiles = (N + TILE - 1) // TILE
    slots = 2 * num_sms
    chunks = []
    for t0 in range(0, T, TCHUNK):
        Tc = min(TCHUNK, T - t0)
        P = rhok_slices(tiles, Tc, slots)
        chunks.append({"t0": t0, "T": Tc, "P": P, "tiles_per": (tiles + P - 1) // P})
    slabs = []
    for k0 in range(0, K, threads * KB):
        Ks = min(K - k0, threads * KB)
        KQ = (Ks + KB - 1) // KB
        slabs.append({"k0": k0, "Ks": Ks, "KQ": KQ, "groups": threads // KQ})
    launches = sum(len(slabs) + (c["P"] > 1) for c in chunks)
    return {"chunks": chunks, "slabs": slabs, "launches": launches, "threads": threads, "tiles": tiles}


def chunk_of(geo, t):
    return geo["chunks"][t // TCHUNK]


def groups_of(geo, k):
    return geo["slabs"][k // (geo["threads"] * KB)]["groups"]


# -------------------------------------------------------------------------------------------------------------------
# exact reference and the summation model
# -------------------------------------------------------------------------------------------------------------------
def exact_terms(pos, kvec):
    """(kr [K, N], cos and sin in long double [K, N])."""
    kr = kernel_argument(pos, kvec)
    la = kr.astype(np.longdouble)
    return kr, np.cos(la), np.sin(la)


def _fsum_rows(ld):
    """Row sums of a long-double [K, N] array: hi + lo doubles through math.fsum."""
    hi = ld.astype(np.float64)
    lo = (ld - hi.astype(np.longdouble)).astype(np.float64)
    return np.array([math.fsum(np.concatenate([hi[k], lo[k]]).tolist()) for k in range(ld.shape[0])])


def ref_slack(N, R):
    return N * 5.5e-20 + 0.5 * np.spacing(np.abs(R))


@functools.lru_cache(maxsize=16)
def _chain_layout(N, tiles_per, groups):
    """Index (slice, group, position in chain) of every particle of a frame, and the chain length."""
    j = np.arange(N)
    tile = j // TILE
    p = tile // tiles_per
    local = j % TILE
    pg = local % groups
    cnt = (TILE - pg + groups - 1) // groups  # particles of group pg in a full tile (only a frame's last tile is ragged)
    pos = (tile - p * tiles_per) * cnt + local // groups
    L = tiles_per * ((TILE + groups - 1) // groups)
    return p, pg, pos, L


def model_sum(terms, P, tiles_per, groups):
    """The kernel's order applied to one component's float64 terms [N] of one k: (result, sum of |partial sums| of
    the chains, sum of |partial sums| of the folds).  Additions that are exact whatever the rounding -- the first
    term of a chain (its own roundings are in eps_j), a fold step with a zero operand (empty particle groups, lanes
    without a slice) -- are not counted."""
    N = terms.shape[0]
    p, pg, pos, L = _chain_layout(N, tiles_per, groups)
    grid = np.zeros((P, groups, L))
    mask = np.zeros((P, groups, L), dtype=bool)
    grid[p, pg, pos] = terms
    mask[p, pg, pos] = True
    mask[:, :, 0] = False
    cs = np.cumsum(grid, axis=2)       # sequential float64 additions along each chain (zeros are exact)
    s_chain = float(np.abs(cs)[mask].sum())
    tot = cs[:, :, -1]                  # [P, groups]
    gf = np.cumsum(tot, axis=1)         # group fold in order
    s_fold = float(np.abs(gf[:, 1:])[(tot[:, 1:] != 0) & (gf[:, :-1] != 0)].sum())
    slices = gf[:, -1]
    if P == 1:
        return float(slices[0]), s_chain, s_fold
    lanes = np.zeros((32, (P + 31) // 32))
    lanes[np.arange(P) % 32, np.arange(P) // 32] = slices
    lc = np.cumsum(lanes, axis=1)
    s_fold += float(np.abs(lc[:, 1:])[(lanes[:, 1:] != 0) & (lc[:, :-1] != 0)].sum())
    v = lc[:, -1]
    for m in (16, 8, 4, 2, 1):
        a, b = v[:m], v[m:2 * m]
        v = a + b
        s_fold += float(np.abs(v)[(a != 0) & (b != 0)].sum())
    return float(v[0]), s_chain, s_fold


def library_branch(kr):
    """[K, N] bool: the pair goes through CUDA's sincos.  The kernel tests the KB = 4 arguments of a thread's k-quad
    (k // 4; slabs start at multiples of 4) together: if any is >= 2^20 (or not finite), all four take the library."""
    K, N = kr.shape
    big = ~(np.abs(kr) < HUGE)
    pad = np.zeros(((K + KB - 1) // KB * KB, N), dtype=bool)
    pad[:K] = big
    quad = pad.reshape(-1, KB, N).any(axis=1)
    return np.repeat(quad, KB, axis=0)[:K]


def _reference_block(pos, kv, P, tiles_per, groups):
    """R, tolerance and library-pair count of one frame for a block of whole k-quads."""
    N = pos.shape[0]
    kr, c, s = exact_terms(pos, kv)
    lib = library_branch(kr)
    eps = np.where(lib, EPS_LIBRARY, EPS_TABLE).sum(axis=1)
    R = np.empty((2, len(kv)))
    tol = np.empty((2, len(kv)))
    for comp, terms in ((0, c), (1, s)):
        R[comp] = _fsum_rows(terms)
        t64 = terms.astype(np.float64)
        for i in range(len(kv)):
            _, sc, sf = model_sum(t64[i], P, tiles_per, groups[i])
            tol[comp, i] = eps[i] + C_BOUND * U * (sc + sf) + ref_slack(N, R[comp, i])
    return R, tol, int(lib.sum())


def reference(frames, kvec, geo, check_frames=None, kblock=8, workers=None):
    """Exact R and the tolerance on the frames checked: {t: (R complex[K], tol_re[K], tol_im[K], library pairs)}.
    `frames` [T, N, 3] float64 (float32 inputs widened: the kernel widens exactly).  Frames and k-blocks are
    independent and go to `workers` threads (default: up to 16 CPUs; NumPy's loops run without the GIL)."""
    T, N = frames.shape[0], frames.shape[1]
    check_frames = list(range(T) if check_frames is None else check_frames)
    K = kvec.shape[0]
    tasks = []
    for t in check_frames:
        if N == 0:
            continue
        ch = chunk_of(geo, t)
        for kb in range(0, K, kblock):  # kblock a multiple of 4: whole k-quads
            kv = kvec[kb:kb + kblock]
            groups = [groups_of(geo, kb + i) for i in range(len(kv))]
            tasks.append(((t, kb), (frames[t], kv, ch["P"], ch["tiles_per"], groups)))
    workers = min(os.cpu_count() or 1, 16) if workers is None else workers
    if workers > 1 and len(tasks) > 1 and N * K * len(check_frames) >= 4_000_000:
        import concurrent.futures as cf
        with cf.ThreadPoolExecutor(max_workers=min(workers, len(tasks))) as ex:
            results = list(ex.map(lambda a: _reference_block(*a), [a for _, a in tasks]))
    else:
        results = [_reference_block(*a) for _, a in tasks]
    out = {t: [np.zeros(K), np.zeros(K), np.zeros(K), np.zeros(K), 0] for t in check_frames}
    for ((t, kb), _), (R, tol, n_lib) in zip(tasks, results):
        o = out[t]
        n = R.shape[1]
        o[0][kb:kb + n], o[1][kb:kb + n] = R[0], R[1]
        o[2][kb:kb + n], o[3][kb:kb + n] = tol[0], tol[1]
        o[4] += n_lib
    return {t: (o[0] + 1j * o[1], o[2], o[3], o[4]) for t, o in out.items()}


def reference_small(frames, kvec, geo):
    """`reference` for every frame of a call in which each particle is a chain of its own (one tile per frame, one slice,
    N <= groups): the kernel's order is then the plain sequential sum over j, vectorised here over all frames."""
    T, N = frames.shape[0], frames.shape[1]
    K = kvec.shape[0]
    assert all(c["P"] == 1 for c in geo["chunks"]) and geo["tiles"] == 1
    assert all(N <= sl["groups"] for sl in geo["slabs"])
    x, y, z = (frames[:, None, :, c] for c in range(3))          # [T, 1, N]
    kx, ky, kz = (kvec[None, :, c, None] for c in range(3))      # [1, K, 1]
    kr = fma(z, kz, fma(y, ky, x * kx))                          # [T, K, N]
    lib = np.stack([library_branch(kr[t]) for t in range(T)])
    eps = np.where(lib, EPS_LIBRARY, EPS_TABLE).sum(axis=2)
    la = kr.astype(np.longdouble)
    R, tol = [], []
    for terms in (np.cos(la), np.sin(la)):
        hi = terms.astype(np.float64)
        lo = (terms - hi.astype(np.longdouble)).astype(np.float64)
        pieces = np.concatenate([hi, lo], axis=2).reshape(T * K, 2 * N).tolist()
        r = np.array([math.fsum(row) for row in pieces]).reshape(T, K)
        cs = np.cumsum(hi, axis=2)  # the group fold; chains of one particle are exact
        partial = (np.abs(cs[:, :, 1:]) * ((hi[:, :, 1:] != 0) & (cs[:, :, :-1] != 0))).sum(axis=2)
        R.append(r)
        tol.append(eps + C_BOUND * U * partial + ref_slack(N, r))
    return R[0] + 1j * R[1], tol[0], tol[1]


# -------------------------------------------------------------------------------------------------------------------
# F(k, t)
# -------------------------------------------------------------------------------------------------------------------
def fkt_exact(rho, o, l):
    """F*[o][l] for rho complex [T, K]: the exact sum of the products, divided by K, rounded once; and the bound."""
    a, b = rho[o], rho[o + l]
    K = a.shape[0]
    p1, e1 = two_product(a.real, b.real)
    p2, e2 = two_product(a.imag, b.imag)
    parts = np.concatenate([p1, e1, p2, e2])
    S = math.fsum(parts)
    r = math.fsum(np.concatenate([parts, [-S]]))  # S + r is the exact sum to ~2^-106 relative
    F = float((Fraction(S) + Fraction(r)) / K)
    mag = float(np.sum(np.abs(a.real * b.real) + np.abs(a.imag * b.imag)))
    n = K + 1
    acc = n * U / (1.0 - n * U) * mag / K
    return F, acc + 0.5 * float(np.spacing(abs(F) + acc))


def fkt_fraction(rho, o, l):
    """The same from Fractions (small tables only)."""
    a, b = rho[o], rho[o + l]
    s = sum((Fraction(x.real) * Fraction(y.real) + Fraction(x.imag) * Fraction(y.imag) for x, y in zip(a, b)),
            Fraction(0))
    return float(s / len(a))


# -------------------------------------------------------------------------------------------------------------------
# inputs (every position is float32-representable, so the xyz, Scalar4 and float32 layouts share one reference)
# -------------------------------------------------------------------------------------------------------------------
def _box(N):
    return (max(N, 1) / 0.1) ** (1.0 / 3.0)  # number density of synth.make_system's boxes


def walk_frames(N, T, seed=0, sigma=0.05):
    """MD-like: a wrapped random walk from uniform positions (synth.random_walk_frames), rounded to float32."""
    from cav_hoomd_b200 import synth
    rng = np.random.default_rng(seed)
    L = _box(N)
    pos = np.zeros((N, 4))
    pos[:, :3] = rng.uniform(-L / 2, L / 2, size=(N, 3))
    s = type("S", (), {"pos": pos, "box": (L, L, L)})()
    return synth.random_walk_frames(s, T, sigma=sigma, seed=seed + 1).astype(np.float32).astype(np.float64)


def decorrelated_frames(N, T, seed=0):
    """Independent uniform positions per frame: F at lag >= 1 is a small remainder of terms ~N."""
    L = _box(N)
    rng = np.random.default_rng(seed)
    return rng.uniform(-L / 2, L / 2, size=(T, N, 3)).astype(np.float32).astype(np.float64)


def dyadic_frames(N, T, seed=0):
    """Positions m / 2^10, |m| < 2^20: with dyadic_kvec every k.r is exact in double."""
    rng = np.random.default_rng(seed)
    return rng.integers(-(2 ** 20) + 1, 2 ** 20, size=(T, N, 3)).astype(np.float64) / 1024.0


def dyadic_kvec(K, seed=0):
    """k components n / 2^10, |n| < 2^12."""
    rng = np.random.default_rng(seed + 99)
    return rng.integers(-(2 ** 12) + 1, 2 ** 12, size=(K, 3)).astype(np.float64) / 1024.0


def push_huge(frames, kvec, tiles, seed=0):
    """One particle in each of the chosen tiles of every frame moved out to |r| = 8 2^20 / max |k|, in a random
    direction: most of its |k.r| exceed 2^20, so those tiles mix the table and the library branch."""
    f = frames.copy()
    rng = np.random.default_rng(seed)
    kmax = np.sqrt((kvec ** 2).sum(axis=1)).max()
    for tile in tiles:
        j = min(tile * TILE + int(rng.integers(0, TILE)), f.shape[1] - 1)
        d = rng.standard_normal((f.shape[0], 3))
        d /= np.sqrt((d ** 2).sum(axis=1, keepdims=True))
        f[:, j, :] = (d * (8.0 * HUGE / kmax)).astype(np.float32)
    return f


def zero_frames(T, N):
    return np.zeros((T, N, 3))


def kvectors(K, mag=1.0, seed=0):
    from cav_hoomd_b200 import synth
    if K == 1:
        return np.array([[0.6, -0.48, 0.64]]) * mag
    return synth.fibonacci_sphere(K) * mag
