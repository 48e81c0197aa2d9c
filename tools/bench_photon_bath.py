#!/usr/bin/env python
"""tools/bench_photon_bath.py -- what the cavity mode's Langevin bath (the *_bath entry points) costs on a B200, CUDA
events.

Per MD step at N particles, rotating over systems that together exceed L2 (as tools/bench_group_list.py), in one process
and on one handle, alternating between the arms of the same work (the order reversed every other repetition):
  fused        cavb200_md_step_fused_wrap (one launch per step, 148 B/particle)
  fused_bath   cavb200_md_step_fused_wrap_bath
  rank1        cavb200_nvt_step_one_rank1_wrap ; cavb200_force_rank1 ; cavb200_nvt_step_two_rank1 (three launches)
  rank1_bath   cavb200_nvt_step_one_rank1_wrap_bath ; cavb200_force_rank1 ; cavb200_nvt_step_two_rank1_bath
The group is the window of all molecules, the photon last; the bath is the reference's (gamma = 1 / 5 ps at 100 K).
The bath adds no bytes per particle: only the photon's thread reads gamma, coeff r and the 24-byte slot."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cav_hoomd_b200 import capi, synth  # noqa: E402

ARMS = ("fused", "fused_bath", "rank1", "rank1_bath")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in out.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-mol", type=int, nargs="+", default=[1_000_000, 16_000_000])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    st = capi.Stream()
    p = capi.Params.make(0.01, 1e-3)
    dt = synth.DT_1FS
    bath = capi.LangevinArgs.make(1.0 / synth.TAU_5PS, synth.KT_100K, (0.3, -0.7, 0.5))
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
        d0 = systems[0]
        h.force_rank1(d0["pos"], d0["charge"], d0["image"], N, base.box, base.L_typeid, p, st.ptr)

        def step(arm, d):
            with_bath = arm.endswith("_bath")
            if arm.startswith("fused"):
                h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, dt, base.box, base.L_typeid, p, 0,
                                n_mol, a, st.ptr, wrap=True, bath=bath if with_bath else None)
            else:
                h.nvt_step_one_rank1(d["pos"], d["vel"], None, d["charge"], N, dt, base.L_typeid, 1e-3, 0, n_mol, a,
                                     st.ptr, image=d["image"], box=base.box, bath=with_bath)
                h.force_rank1(d["pos"], d["charge"], d["image"], N, base.box, base.L_typeid, p, st.ptr)
                h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], N, dt, base.L_typeid, 1e-3, 0, n_mol, st.ptr,
                                     bath=bath if with_bath else None)

        def run(arm, steps):
            e0, e1 = capi.Event(), capi.Event()
            capi.sync()
            e0.record(st.ptr)
            for k in range(steps):
                step(arm, systems[k % n_sys])
            e1.record(st.ptr)
            return e1.elapsed_ms_since(e0) / steps

        print(f"N={N} systems={n_sys} ({n_sys * 148 * N / 1e6:.0f} MB of step traffic per rotation)", flush=True)
        times = {arm: [] for arm in ARMS}
        for arm in ARMS:
            run(arm, 5)
        for r in range(args.reps):
            for arm in (ARMS if r % 2 == 0 else ARMS[::-1]):
                times[arm].append(run(arm, args.steps) * 1e3)
        med = {arm: float(np.median(times[arm])) for arm in ARMS}
        for arm in ARMS:
            ref = arm.replace("_bath", "")
            row = dict(N=N, arm=arm, us_per_step_median=med[arm], us_per_step_min=float(min(times[arm])),
                       us_per_step_max=float(max(times[arm])), vs=ref, overhead=med[arm] / med[ref] - 1.0,
                       reps=args.reps, steps=args.steps, **info)
            rows.append(row)
            print(f"  {arm:10s}: median {med[arm]:9.2f} us/step  (min {min(times[arm]):9.2f}, max {max(times[arm]):9.2f})"
                  f"  vs {ref:6s} {100 * row['overhead']:+6.2f} %", flush=True)
        assert h.bussi_read(st.ptr)["err"] == 0.0
        assert h.fault_count == 0
        for d in systems:
            for x in d.values():
                x.free()
        h.close()
    if args.out:
        json.dump(rows, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
