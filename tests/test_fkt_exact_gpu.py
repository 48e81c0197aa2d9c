"""cavb200_rhok, cavb200_rhok_f32 and cavb200_fkt under every launch schedule, against exact sums
(tests/fkt_inputs.py; the CPU side of the argument is tests/test_fkt_exact.py).

For every case and layout (xyz, Scalar4 with NaN in the fourth word, float32; padded frames whose padding is NaN):
  1. the launch count is the restated schedule's (slabs + one fold launch per chunk of frames with P > 1);
  2. |rho - R| <= the a-posteriori bound of the kernel's summation order, per component, on the checked frames, and
     every frame is written;
  3. the layouts agree bit for bit (every position is float32-representable);
  4. all-zero frames of the same shape give exactly (N, 0) in every frame: every term is (1, 0), so any dropped,
     doubled or misplaced particle, tile, slice, slab or frame is an integer error.
cavb200_fkt is held to F* (the exact sum of the products over K, rounded once) within gamma_{K+1} sum |products| / K
plus the rounding of the division.  At the end of the module the largest error / bound per schedule is printed.
"""
import functools

import numpy as np
import pytest

import fkt_inputs as fi
from cav_hoomd_b200 import capi

pytestmark = pytest.mark.gpu

MISALIGNED = 716  # cudaErrorMisalignedAddress
WORST = {}        # schedule -> largest |rho - R| / bound
FKT_NOTES = {}


@pytest.fixture(scope="module", autouse=True)
def worst_per_schedule(pytestconfig):
    yield
    if not WORST and not FKT_NOTES:
        return
    lines = ["", "largest |error| / bound per schedule and layout"]
    lines += [f"  {k:48s} {v:8.4f}" for k, v in sorted(WORST.items())]
    lines += [f"  {k}: {v}" for k, v in sorted(FKT_NOTES.items())]
    capman = pytestconfig.pluginmanager.getplugin("capturemanager")
    with capman.global_and_fixture_disabled():
        print("\n".join(lines))


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def h():
    handle = capi.Handle(0)
    yield handle
    handle.close()


# name: (N, T, K, threads, builder, checked frames (None = all), P / tiles per CTA / slabs / launches on 148 SMs)
CASES = {
    "tiny": (1, 1, 1, 256, "walk", None, (1, 1, 1, 1)),
    "ragged_kq_one_tile": (512, 1, 7, 256, "decorrelated", None, (1, 1, 1, 1)),
    "two_slices": (513, 1, 63, 256, "walk", None, (2, 1, 1, 2)),
    "ragged_groups": (100001, 3, 65, 256, "walk", None, (98, 2, 1, 2)),
    "live_tracker": (1000001, 1, 64, 256, "walk", None, (280, 7, 1, 2)),
    "bench_shape": (1000001, 32, 64, 256, "walk", (0, 15, 31), (37, 53, 1, 2)),
    "direct_multi_tile": (1537, 8000, 5, 256, "decorrelated", (0, 1, 2, 3999, 7998, 7999), (1, 4, 1, 1)),
    "two_slabs": (20001, 2, 1025, 256, "walk", None, (40, 1, 2, 3)),
    "three_slabs": (5000, 2, 2051, 256, "dyadic", None, (10, 1, 3, 4)),
    "t128_two_slabs": (20001, 2, 513, 128, "decorrelated", None, (40, 1, 2, 3)),
    "t128_f32_sync": (100001, 3, 64, 128, "walk", None, (98, 2, 1, 2)),
    "t128_f32_sync_direct": (1537, 8000, 5, 128, "walk", (0, 1, 4000, 7999), (1, 4, 1, 1)),
    # |k| = 3e4 on the 100 001-particle walk: |k.r| up to ~2.6e6, so tiles mix the table and the library branch
    "huge_arguments": (100001, 2, 64, 256, "walk_k3e4", None, None),
    # one particle per chosen tile far out: those tiles take the range-tested walk, the others the plain one
    "pushed_tiles": (5000, 2, 64, 256, "pushed", None, None),
}
PADDED = {"two_slabs", "three_slabs", "t128_two_slabs", "t128_f32_sync", "t128_f32_sync_direct", "direct_multi_tile",
          "ragged_groups"}


@functools.lru_cache(maxsize=2)
def case_inputs(name, num_sms):
    N, T, K, threads, kind, check, _ = CASES[name]
    mag = 3.0e4 if kind == "walk_k3e4" else 1.0
    kvec = fi.dyadic_kvec(K) if kind == "dyadic" else fi.kvectors(K, mag)
    if kind in ("walk", "walk_k3e4"):
        frames = fi.walk_frames(N, T, seed=N + T)
    elif kind == "decorrelated":
        frames = fi.decorrelated_frames(N, T, seed=N + T)
    elif kind == "dyadic":
        frames = fi.dyadic_frames(N, T, seed=N + T)
    else:
        frames = fi.push_huge(fi.walk_frames(N, T, seed=N), kvec, tiles=(0, 3, 9))
    geo = fi.geometry(N, T, K, num_sms, threads)
    ref = fi.reference(frames, kvec, geo, check_frames=check)
    return frames, kvec, geo, ref


def pack(frames, layout, padded):
    """Device array and frame stride (in elements of the layout) of frames [T, N, 3]."""
    T, N = frames.shape[0], frames.shape[1]
    if layout == "xyz":
        fs, dt, w = 3 * N + (5 if padded else 0), np.float64, 3
    elif layout == "scalar4":
        fs, dt, w = 4 * N + (8 if padded else 0), np.float64, 4
    else:
        fs, dt, w = 3 * N + (1 if padded else 0), np.float32, 3
    a = np.full((T, max(fs, 1)), np.nan, dtype=dt)
    v = a[:, :w * N].reshape(T, N, w)
    v[:, :, :3] = frames
    return a, fs


def run_rhok(h, frames, kvec, layout, padded, threads=256):
    T, N, K = frames.shape[0], frames.shape[1], kvec.shape[0]
    a, fs = pack(frames, layout, padded)
    d_pos = capi.DeviceArray.from_numpy(a)
    d_k = capi.DeviceArray.from_numpy(kvec)
    d_rho = capi.DeviceArray((T, K, 2), np.float64)
    d_rho.fill_bytes(0xFF)
    h.set_tuning(rhok_threads=threads)
    before = h.launch_count
    if layout == "f32":
        h.rhok_f32(d_pos, fs, N, T, d_k, K, d_rho)
    else:
        h.rhok(d_pos, 4 if layout == "scalar4" else 3, fs, N, T, d_k, K, d_rho)
    r = d_rho.numpy()
    if a.nbytes <= 64 << 20:  # positions and padding are read-only (tests/test_guards_gpu.py checks every size)
        assert np.array_equal(d_pos.numpy().view(np.uint8), a.view(np.uint8))
    return r, h.launch_count - before


def check_rho(key, rho, ref, N):
    worst = 0.0
    for t, (R, tol_re, tol_im, _) in ref.items():
        er = np.abs(rho[t, :, 0] - R.real)
        ei = np.abs(rho[t, :, 1] - R.imag)
        worst = max(worst, float((er / tol_re).max()), float((ei / tol_im).max()))
        assert np.all(er <= tol_re) and np.all(ei <= tol_im), (key, t, (er / tol_re).max(), (ei / tol_im).max())
    WORST[key] = max(WORST.get(key, 0.0), worst)


def check_zero(rho, N):
    want = np.array([float(N), 0.0]).view(np.uint64)
    assert np.all(rho.view(np.uint64) == want), np.argwhere(rho.view(np.uint64) != want)[:5]


LAYOUTS = ["xyz", "scalar4", "f32"]


@pytest.mark.parametrize("name", list(CASES))
def test_rhok_schedules(h, num_sms, name):
    N, T, K, threads, kind, check, expect = CASES[name]
    frames, kvec, geo, ref = case_inputs(name, num_sms)
    ch = geo["chunks"][0]
    if expect is not None and num_sms == 148:
        assert (ch["P"], ch["tiles_per"], len(geo["slabs"]), geo["launches"]) == expect
    if kind == "walk_k3e4":
        lib = sum(r[3] for r in ref.values())
        assert 0 < lib < N * K * len(ref), "the case must mix both branches"
    if kind == "pushed":
        assert all(r[3] > 0 for r in ref.values())
    runs = [(lay, False) for lay in LAYOUTS] + ([(lay, True) for lay in LAYOUTS] if name in PADDED else [])
    first = None
    for layout, padded in runs:
        rho, launches = run_rhok(h, frames, kvec, layout, padded, threads)
        assert launches == geo["launches"], (layout, padded, launches, geo["launches"])
        assert np.isfinite(rho).all(), (layout, padded)
        sched = f"P{ch['P']}x{ch['tiles_per']} slabs{len(geo['slabs'])} t{geo['threads']}"
        check_rho(f"{name} [{sched}] {layout}{' padded' if padded else ''}", rho, ref, N)
        if first is None:
            first = rho
        else:
            assert np.array_equal(rho.view(np.uint64), first.view(np.uint64)), (layout, padded)
        zero, launches = run_rhok(h, fi.zero_frames(T, N), kvec, layout, padded, threads)
        assert launches == geo["launches"]
        check_zero(zero, N)
    h.set_tuning(rhok_threads=0)


@pytest.mark.parametrize("T", [65535, 65536, 70000])
def test_rhok_any_frame_count(h, num_sms, T):
    """grid y holds at most 65535 frames: longer calls are launched in chunks (every frame checked)."""
    N, K = 8, 3
    frames = fi.walk_frames(N, T, seed=T, sigma=0.5)
    kvec = fi.kvectors(K)
    geo = fi.geometry(N, T, K, num_sms)
    assert geo["launches"] == (T + 65534) // 65535
    R, tol_re, tol_im = fi.reference_small(frames, kvec, geo)
    ref = {t: (R[t], tol_re[t], tol_im[t], 0) for t in range(T)}
    for layout in LAYOUTS:
        rho, launches = run_rhok(h, frames, kvec, layout, layout == "f32")
        assert launches == geo["launches"]
        check_rho(f"frames T={T} [direct, {len(geo['chunks'])} chunk(s)] {layout}", rho, ref, N)
        zero, _ = run_rhok(h, fi.zero_frames(T, N), kvec, layout, False)
        check_zero(zero, N)


def test_rhok_empty_calls(h):
    kvec = capi.DeviceArray.from_numpy(fi.kvectors(4))
    pos = capi.DeviceArray.from_numpy(np.zeros((2, 10, 4)))
    pos32 = capi.DeviceArray.from_numpy(np.zeros((2, 10, 3), np.float32))
    rho = capi.DeviceArray((2, 4, 2), np.float64)
    for stride in (3, 4, None):
        rho.fill_bytes(0xFF)
        n0 = h.launch_count
        if stride is None:
            h.rhok_f32(pos32, 30, 0, 2, kvec, 4, rho)
        else:
            h.rhok(pos, stride, 40, 0, 2, kvec, 4, rho)
        assert h.launch_count == n0 and np.all(rho.numpy() == 0.0)  # N = 0: rho = 0, no kernel
        rho.fill_bytes(0xFF)
        for T, K in ((0, 4), (2, 0)):
            if stride is None:
                h.rhok_f32(pos32, 30, 10, T, kvec, K, rho)
            else:
                h.rhok(pos, stride, 40, 10, T, kvec, K, rho)
        assert h.launch_count == n0
        assert np.all(rho.numpy().view(np.uint64) == np.uint64(0xFFFFFFFFFFFFFFFF))  # nothing written


def test_rhok_misaligned_arguments(h):
    kvec = capi.DeviceArray.from_numpy(fi.kvectors(4))
    pos = capi.DeviceArray.from_numpy(np.zeros((2, 12, 4)))  # room for a frame stride of 44
    rho = capi.DeviceArray((2, 4, 2), np.float64)
    n0 = h.launch_count
    for fs in (41, 42, 43):
        with pytest.raises(capi.CavbError) as e:
            h.rhok(pos, 4, fs, 10, 2, kvec, 4, rho)
        assert e.value.code == MISALIGNED
    h.rhok(pos, 4, 44, 10, 2, kvec, 4, rho)   # padded Scalar4 frames, stride a multiple of 4
    h.rhok(pos, 4, 40, 10, 2, kvec, 4, rho)
    n1 = h.launch_count
    assert n1 > n0
    with pytest.raises(capi.CavbError) as e:
        h.rhok_f32(pos.offset(2), 30, 10, 2, kvec, 4, rho)
    assert e.value.code == MISALIGNED
    assert h.launch_count == n1


# ---------------------------------------------------------------------------------------------------------------------
# cavb200_fkt
# ---------------------------------------------------------------------------------------------------------------------
def synthetic_rho(T, K, correlated, seed):
    """|rho| ~ 1e3 (a frame of ~1e6 particles); correlated: a slow drift, decorrelated: independent per frame."""
    rng = np.random.default_rng(seed)
    z = (rng.standard_normal((T, K)) + 1j * rng.standard_normal((T, K))) * 700.0
    if correlated:
        z = z[0][None, :] + np.cumsum(z * 0.02, axis=0)
    return z


def run_fkt(h, rho, n_or, n_lag):
    T, K = rho.shape
    d_rho = capi.DeviceArray.from_numpy(np.stack([rho.real, rho.imag], axis=-1))
    d_out = capi.DeviceArray((n_or, n_lag), np.float64)
    d_out.fill_bytes(0x00)
    n0 = h.launch_count
    h.fkt(d_rho, T, K, n_or, n_lag, d_out)
    F = d_out.numpy()
    assert h.launch_count == n0 + 1
    o, l = np.meshgrid(np.arange(n_or), np.arange(n_lag), indexing="ij")
    assert np.array_equal(np.isnan(F), o + l >= T)  # NaN exactly where the lag runs past the last frame
    return F


def check_fkt(key, rho, F, cells):
    worst = 0.0
    for o, l in cells:
        Fs, b = fi.fkt_exact(rho, o, l)
        err = abs(F[o, l] - Fs)
        worst = max(worst, err / b)
        assert err <= b, (key, o, l, F[o, l], Fs, b)
    WORST[key] = max(WORST.get(key, 0.0), worst)


@pytest.mark.parametrize("K", [1, 64, 4096])
@pytest.mark.parametrize("correlated", [True, False])
def test_fkt_small_tables(h, K, correlated):
    T, n_or, n_lag = 12, 8, 10
    rho = synthetic_rho(T, K, correlated, seed=K)
    F = run_fkt(h, rho, n_or, n_lag)
    check_fkt(f"fkt K={K} {'correlated' if correlated else 'decorrelated'}", rho, F,
              [(o, l) for o in range(n_or) for l in range(n_lag) if o + l < T])


@pytest.mark.parametrize("correlated", [True, False])
def test_fkt_full_size_table(h, correlated):
    T, K = 1200, 64
    rho = synthetic_rho(T, K, correlated, seed=7)
    F = run_fkt(h, rho, 1000, 1000)
    cells = [(o, l) for o in range(200) for l in range(200)]
    rng = np.random.default_rng(11)
    o = rng.integers(0, 1000, 10000)
    l = rng.integers(0, 1000, 10000)
    cells += [(int(a), int(b)) for a, b in zip(o, l) if a + b < T]
    check_fkt(f"fkt 1000x1000 T=1200 {'correlated' if correlated else 'decorrelated'}", rho, F, cells)


def test_fkt_more_origins_than_frames(h):
    T, K = 5, 16
    rho = synthetic_rho(T, K, True, seed=3)
    F = run_fkt(h, rho, 9, 3)
    check_fkt("fkt n_origins > T", rho, F, [(o, l) for o in range(9) for l in range(3) if o + l < T])


def test_fkt_orthogonal_pair(h):
    """b = i a: Re(a conj b) = a_r (-a_i) + a_i a_r = 0 exactly.  With the products contracted to an FMA the kernel
    returns the rounding residual of one product there, not 0; the bound still holds."""
    K = 64
    rho = synthetic_rho(2, K, False, seed=5)
    rho[1] = 1j * rho[0]
    F = run_fkt(h, rho, 1, 2)
    Fs, b = fi.fkt_exact(rho, 0, 1)
    assert Fs == 0.0
    assert abs(F[0, 1]) <= b
    FKT_NOTES["fkt b = i a, K=64: F[0][1] (exact 0)"] = f"{F[0, 1]!r} (bound {b:.3e})"
