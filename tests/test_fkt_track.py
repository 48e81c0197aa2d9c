"""cavb200_extras.FieldAutocorrelation on the CPU: its schedule against the host mirror's
(analysis.FieldAutocorrelationTracker.act, the reference's act restated) and the conversion of device records
(layout: include/cavb200.h) into rows, on a stub of the C++ force's fktOpen / fktStep / fktRead that keeps the ring in
NumPy.  The device side is tests/test_fkt_track_gpu.py."""
import importlib.util
import os

import numpy as np
import pytest

from cav_hoomd_b200 import analysis, synth
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def extras():
    spec = importlib.util.spec_from_file_location("cavb200_extras", os.path.join(ROOT, "plugin", "python",
                                                                                  "cavb200_extras.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class StubForce:
    """fktOpen / fktStep / fktRead with the device tracker's semantics, rho from the NumPy restatement of
    compute_density_field and F from compute_field_autocorr."""

    def __init__(self, positions):
        self.positions = positions  # callable -> current [N, 3]
        self.steps = []

    def fktOpen(self, kvectors, max_references, capacity):
        self.k = np.array(kvectors, dtype=np.float64)
        self.M, self.cap = max_references, capacity
        self.refs, self.ring, self.count = [], [None] * capacity, 0

    def fktStep(self, timestep, record, add_reference):
        assert record or add_reference
        assert not add_reference or len(self.refs) < self.M
        self.steps.append((timestep, record, add_reference))
        rho = O.numpy_density_field(self.positions(), self.k)
        if record:
            F = [np.nan] * self.M
            for r, ref in enumerate(self.refs):
                F[r] = analysis.FieldAutocorrelationTracker.compute_field_autocorr(ref, rho)
            rec = np.concatenate([[timestep, len(self.refs)], F, np.stack([rho.real, rho.imag], axis=1).ravel()])
            self.ring[self.count % self.cap] = rec
            self.count += 1
        if add_reference:
            self.refs.append(rho)

    def fktRead(self, max_records):
        have = min(self.count, self.cap, max_records)
        recs = [self.ring[i % self.cap] for i in range(self.count - have, self.count)]
        words = 2 + self.M + 2 * len(self.k)
        return (np.array(recs) if recs else np.zeros((0, words))), self.count


class MirrorOnHost(analysis.FieldAutocorrelationTracker):
    """The mirror's act() with its density field on the host (its own needs a device)."""

    def __init__(self, positions, wavevectors, reference_interval_steps, max_references):
        self.positions, self.wavevectors = positions, wavevectors
        self.reference_interval_steps, self.max_references = reference_interval_steps, max_references
        self.references, self.last_reference_step, self.current_autocorr_value = [], 0, 0.0
        self._add_reference(0)

    def _current_field(self):
        return O.numpy_density_field(self.positions(), self.wavevectors)


@pytest.mark.parametrize("interval,M,steps", [(2, 3, 12), (1, 10, 6), (5, 2, 20), (10000, 10, 8)])
def test_schedule_and_rows_match_the_mirror(interval, M, steps):
    X = extras()
    frames = np.random.default_rng(interval + M).uniform(-5, 5, size=(steps + 1, 40, 3))
    cur = {"t": 0}
    positions = lambda: frames[cur["t"]]  # noqa: E731
    k = synth.fibonacci_sphere(7) * 1.3
    mirror = MirrorOnHost(positions, k, interval, M)
    stub = StubForce(positions)
    dev = X.FieldAutocorrelation(stub, k, reference_interval_steps=interval, max_references=M, capacity=64)
    assert stub.steps == [(0, False, True)]
    want = []
    for t in range(steps + 1):
        cur["t"] = t
        want += [(r, t, lag, v) for r, lag, v in mirror.act(t)]
        assert dev.act(t) is None
    assert dev.reference_timesteps == [r["timestep"] for r in mirror.references]
    assert len(stub.steps) == steps + 1 and all(rec for _, rec, _ in stub.steps[1:])
    rows, rho = dev.read()
    assert rows == want
    assert rho.shape == (steps, 7, 2)
    for t in range(1, steps + 1):
        f = O.numpy_density_field(frames[t], k)
        assert np.array_equal(rho[t - 1, :, 0], f.real) and np.array_equal(rho[t - 1, :, 1], f.imag)
    assert dev.read()[0] == []


def test_read_returns_the_records_since_the_last_read_and_at_most_the_ring():
    X = extras()
    frames = np.random.default_rng(1).uniform(-5, 5, size=(30, 10, 3))
    cur = {"t": 0}
    stub = StubForce(lambda: frames[cur["t"]])
    k = synth.fibonacci_sphere(3)
    dev = X.FieldAutocorrelation(stub, k, reference_interval_steps=4, max_references=2, capacity=5)
    for t in range(1, 4):
        cur["t"] = t
        dev.act(t)
    rows, rho = dev.read()
    assert [(r, t) for r, t, _, _ in rows] == [(0, 1), (0, 2), (0, 3)] and rho.shape == (3, 3, 2)
    for t in range(4, 30):
        cur["t"] = t
        dev.act(t)
    rows, rho = dev.read()  # 26 new records, the ring keeps the newest 5
    assert sorted({t for _, t, _, _ in rows}) == list(range(25, 30)) and rho.shape == (5, 3, 2)
    assert [(r, t, lag) for r, t, lag, _ in rows if t == 29] == [(0, 29, 29), (1, 29, 25)]


def test_records_to_rows():
    X = extras()
    M, K = 3, 2
    nan = np.nan
    recs = np.array([[7, 1, 0.5, nan, nan, 1, 2, 3, 4],
                     [9, 3, 0.25, 0.125, -1.0, 5, 6, 7, 8]])
    assert recs.shape[1] == 2 + M + 2 * K
    rows = X.records_to_rows(recs, [0, 4, 8], M)
    assert rows == [(0, 7, 7, 0.5), (0, 9, 9, 0.25), (1, 9, 5, 0.125), (2, 9, 1, -1.0)]
    assert X.records_to_rows(np.zeros((0, 9)), [0], M) == []


def test_accepts_the_wrapper_or_its_cpp_object():
    X = extras()
    stub = StubForce(lambda: np.zeros((2, 3)))
    wrapper = type("W", (), {"_cpp_obj": stub})()
    X.FieldAutocorrelation(wrapper, [[1.0, 0.0, 0.0]])
    assert stub.steps == [(0, False, True)]
    with pytest.raises(RuntimeError):
        X.FieldAutocorrelation(type("W", (), {"_cpp_obj": None})(), [[1.0, 0.0, 0.0]])
