#!/usr/bin/env python
"""tools/bench_fkt_track.py -- what the F(k,t) tracker without snapshots (cavb200_fkt_track_step) costs per MD step on a
B200, CUDA events, against the snapshot path it replaces.

Per MD step at N particles, rotating over systems that together exceed L2 (as tools/bench_photon_bath.py), in one
process and on one handle, alternating between the arms (the order reversed every other repetition):
  fused       cavb200_md_step_fused_wrap alone
  fused_fkt   the same, then cavb200_fkt_track_step(RECORD) on the positions it wrote, against `--refs` stored references
  rhok        cavb200_rhok of one Scalar4 frame (T = 1) alone: the density field the tracker's record is built on
for each K of `--k`.  The tracker's cost is fused_fkt - fused.
The tracker and rhok arms read a copy of each system's initial positions (one per system, rotated with it), not the
positions the fused step keeps writing: these synthetic boxes are not equilibrated, their photon is thrown out within a
few dozen steps (|v| ~ 1e19 after 8 steps at 1M particles, g = 1e-3), and a non-finite or huge coordinate would send the
density field down the library sincos branch, which is not what a production run pays.  The density field is FP64
bound, so reading a frame that was not just written (and is not in L2) costs it little.
The snapshot path (the reference's FieldAutocorrelationTracker.act: a full device -> host copy of the positions, K NumPy
passes over them, the correlation with every reference) is timed with a host clock over `--snapshot-steps` steps, at the
sizes in `--snapshot-n-mol` only (16M particles take tens of seconds per step)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cav_hoomd_b200 import capi, synth  # noqa: E402
from oracle import oracle as O  # noqa: E402

ARMS = ("fused", "fused_fkt", "rhok")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in out.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-mol", type=int, nargs="+", default=[1_000_000, 16_000_000])
    ap.add_argument("--k", type=int, nargs="+", default=[50, 64])
    ap.add_argument("--refs", type=int, default=10)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--snapshot-n-mol", type=int, nargs="*", default=[1_000_000])
    ap.add_argument("--snapshot-steps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    st = capi.Stream()
    p = capi.Params.make(0.01, 1e-3)
    dt = synth.DT_1FS
    rows = []
    for n_mol in args.n_mol:
        N = n_mol + 1
        n_sys = max(2, min(8, int(2e9 // (148 * N))))
        dof = 3.0 * n_mol - 3
        a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, dt, dof, 0.1, (dof - 1) / 2)
        base = synth.make_system(n_mol, photon="last")
        h = capi.Handle(0)
        systems = [{f: capi.DeviceArray.from_numpy(getattr(base, f)) for f in ("pos", "charge", "image", "vel")}
                   for _ in range(n_sys)]
        for d in systems:
            h.bussi_ke(d["vel"], None, 0, n_mol, st.ptr)
        frames = [capi.DeviceArray.from_numpy(base.pos) for _ in range(n_sys)]
        d0 = systems[0]
        h.force_rank1(d0["pos"], d0["charge"], d0["image"], N, base.box, base.L_typeid, p, st.ptr)
        print(f"N={N} systems={n_sys} ({n_sys * 148 * N / 1e6:.0f} MB of step traffic per rotation)", flush=True)
        for K in args.k:
            kvec = synth.fibonacci_sphere(K) * 1.0
            d_k = capi.DeviceArray.from_numpy(kvec)
            d_rho = capi.DeviceArray((K, 2), np.float64)
            h.fkt_track_open(kvec, args.refs, 4096, N)
            for r in range(args.refs):
                h.fkt_track_step(frames[r % n_sys], N, r, capi.Handle.FKT_ADD_REFERENCE, st.ptr)
            t_step = [args.refs]

            def step(arm, k):
                d, frame = systems[k % n_sys], frames[k % n_sys]
                if arm == "rhok":
                    h.rhok(frame, 4, 4 * N, N, 1, d_k, K, d_rho, st.ptr)
                    return
                h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, dt, base.box, base.L_typeid, p,
                                0, n_mol, a, st.ptr, wrap=True)
                if arm == "fused_fkt":
                    h.fkt_track_step(frame, N, t_step[0], capi.Handle.FKT_RECORD, st.ptr)
                    t_step[0] += 1

            def run(arm, steps):
                e0, e1 = capi.Event(), capi.Event()
                capi.sync()
                e0.record(st.ptr)
                for k in range(steps):
                    step(arm, k)
                e1.record(st.ptr)
                ms = e1.elapsed_ms_since(e0) / steps
                if arm == "rhok":
                    assert np.isfinite(d_rho.numpy(st.ptr)).all()
                elif arm == "fused_fkt":
                    rec, _ = h.fkt_track_read(1, st.ptr)
                    assert np.isfinite(rec).all()
                return ms

            times = {arm: [] for arm in ARMS}
            for arm in ARMS:
                run(arm, 5)
            for r in range(args.reps):
                for arm in (ARMS if r % 2 == 0 else ARMS[::-1]):
                    times[arm].append(run(arm, args.steps) * 1e3)
            med = {arm: float(np.median(times[arm])) for arm in ARMS}
            rec, total = h.fkt_track_read(1, st.ptr)
            assert total == 5 + args.reps * args.steps and rec[0, 1] == args.refs
            for arm in ARMS:
                row = dict(N=N, K=K, refs=args.refs, arm=arm, us_per_step_median=med[arm],
                           us_per_step_min=float(min(times[arm])), us_per_step_max=float(max(times[arm])),
                           reps=args.reps, steps=args.steps, **info)
                if arm == "fused_fkt":
                    row["tracker_us_per_step"] = med["fused_fkt"] - med["fused"]
                rows.append(row)
                extra = f"  tracker {row['tracker_us_per_step']:8.2f} us" if arm == "fused_fkt" else ""
                print(f"  K={K:3d} {arm:9s}: median {med[arm]:9.2f} us/step  (min {min(times[arm]):9.2f}, "
                      f"max {max(times[arm]):9.2f}){extra}", flush=True)

            if n_mol in args.snapshot_n_mol:
                # the snapshot path: positions to the host, K NumPy passes, F against every reference on the host
                refs = [O.numpy_density_field(base.pos[:, :3], kvec)] * args.refs
                ts = []
                for s in range(args.snapshot_steps):
                    capi.sync()
                    t0 = time.perf_counter()
                    pos = frames[s % n_sys].numpy(st.ptr)
                    rho = O.numpy_density_field(pos[:, :3], kvec)
                    F = [float(np.mean(np.real(f0 * np.conj(rho)))) for f0 in refs]
                    ts.append((time.perf_counter() - t0) * 1e6)
                    assert np.isfinite(F).all()
                row = dict(N=N, K=K, refs=args.refs, arm="snapshot", us_per_step_median=float(np.median(ts)),
                           us_per_step_min=float(min(ts)), us_per_step_max=float(max(ts)), steps=args.snapshot_steps,
                           clock="host perf_counter", **info)
                rows.append(row)
                print(f"  K={K:3d} snapshot : median {row['us_per_step_median']:9.0f} us/step  "
                      f"(min {min(ts):9.0f}, max {max(ts):9.0f}, {args.snapshot_steps} steps, host clock)", flush=True)
        assert h.fault_count == 0
        for d in systems:
            for x in d.values():
                x.free()
        for x in frames:
            x.free()
        h.close()
    if args.out:
        json.dump(rows, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
