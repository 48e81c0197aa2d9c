#!/usr/bin/env python
"""tools/bench_group_list.py -- what the group mask (cavb200_group_set, CAVB200_GROUP_MASK) costs on a B200, CUDA events.

Per MD step at N particles, rotating over systems that together exceed L2 (as tools/bench_nvt.py), in one process,
alternating between four arms of the same work (the order reversed every other repetition).  Two handles, each with its
own systems, so that each mask arm is compared with a window arm on the same memory and handle:
  window    handle A, photon last: group_first = 0, the window [0, n) of all molecules
  range     handle A: the same group as a mask built from the index list 0 .. n-1
  window_b  handle B, photon in the middle: the window [0, n) (same amount of work; the photon is in it)
  middle    handle B: all molecules as a mask (the index list has a hole where the photon sits)
for two steps:
  fused    cavb200_md_step_fused_wrap (one launch per step, 148 B/particle)
  rank1    cavb200_nvt_step_one_rank1_wrap ; cavb200_force_rank1 ; cavb200_nvt_step_two_rank1 (three launches)
The mask adds one 4-byte word per 32 particles and pass (0.125 B/particle).  Also timed: what a particle sort costs
once, cavb200_group_set + cavb200_rank1_reindex (both blocking), host clock around the pair."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cav_hoomd_b200 import capi, synth  # noqa: E402

ARMS = ("window", "range", "window_b", "middle")
BASE = {"window": "window", "range": "window", "window_b": "window_b", "middle": "window_b"}


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
    rows = []
    for n_mol in args.n_mol:
        N = n_mol + 1
        n_sys = max(2, min(8, int(2e9 // (148 * N))))
        dof = 3.0 * n_mol - 3
        a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, dt, dof, 0.1, (dof - 1) / 2)
        arms = {}
        for photon, (w_arm, m_arm) in (("last", ("window", "range")), ("middle", ("window_b", "middle"))):
            base = synth.make_system(n_mol, photon=photon)
            h = capi.Handle(0)
            idx = capi.DeviceArray.from_numpy(np.flatnonzero(base.typeid != base.L_typeid).astype(np.uint32))
            h.group_set(idx, n_mol, N, st.ptr)
            systems = [{f: capi.DeviceArray.from_numpy(getattr(base, f)) for f in ("pos", "charge", "image", "vel")}
                       for _ in range(n_sys)]
            for d in systems:
                h.bussi_ke(d["vel"], idx, 0, n_mol, st.ptr)
            d0 = systems[0]
            h.force_rank1(d0["pos"], d0["charge"], d0["image"], N, base.box, base.L_typeid, p, st.ptr)
            arms[w_arm] = dict(h=h, base=base, first=0, systems=systems, idx=idx)
            arms[m_arm] = dict(h=h, base=base, first=capi.Handle.GROUP_MASK, systems=systems, idx=idx)

        def step(kind, arm, d):
            h, base, first = arm["h"], arm["base"], arm["first"]
            if kind == "fused":
                h.md_step_fused(d["pos"], d["vel"], None, d["charge"], d["image"], N, dt, base.box, base.L_typeid, p, first,
                                n_mol, a, st.ptr, wrap=True)
            else:
                h.nvt_step_one_rank1(d["pos"], d["vel"], None, d["charge"], N, dt, base.L_typeid, 1e-3, first, n_mol, a,
                                     st.ptr, image=d["image"], box=base.box)
                h.force_rank1(d["pos"], d["charge"], d["image"], N, base.box, base.L_typeid, p, st.ptr)
                h.nvt_step_two_rank1(d["vel"], None, d["charge"], d["pos"], N, dt, base.L_typeid, 1e-3, first, n_mol, st.ptr)

        def run(kind, arm, steps):
            e0, e1 = capi.Event(), capi.Event()
            capi.sync()
            e0.record(st.ptr)
            for k in range(steps):
                step(kind, arm, arm["systems"][k % n_sys])
            e1.record(st.ptr)
            return e1.elapsed_ms_since(e0) / steps

        print(f"N={N} systems per arm={n_sys}", flush=True)
        for kind in ("fused", "rank1"):
            times = {arm: [] for arm in ARMS}
            for arm in ARMS:
                run(kind, arms[arm], 5)
            for r in range(args.reps):
                for arm in (ARMS if r % 2 == 0 else ARMS[::-1]):
                    times[arm].append(run(kind, arms[arm], args.steps) * 1e3)
            med = {arm: float(np.median(times[arm])) for arm in ARMS}
            for arm in ARMS:
                row = dict(N=N, step=kind, arm=arm, us_per_step_median=med[arm], us_per_step_min=float(min(times[arm])),
                           us_per_step_max=float(max(times[arm])), vs=BASE[arm],
                           overhead=med[arm] / med[BASE[arm]] - 1.0, **info)
                rows.append(row)
                print(f"  {kind:5s} {arm:8s}: median {med[arm]:9.2f} us/step  (min {min(times[arm]):9.2f}, max "
                      f"{max(times[arm]):9.2f})  vs {BASE[arm]:8s} {100 * row['overhead']:+6.2f} %", flush=True)
        for arm in ARMS:
            assert arms[arm]["h"].bussi_read(st.ptr)["err"] == 0.0
            assert arms[arm]["h"].fault_count == 0

        if N <= 2_000_000:
            arm = arms["middle"]
            d = arm["systems"][0]
            t_sort = []
            for k in range(12):
                capi.sync()
                t0 = time.perf_counter()
                arm["h"].group_set(arm["idx"], n_mol, N, st.ptr)
                arm["h"].rank1_reindex(d["pos"], N, arm["base"].L_typeid, st.ptr)
                t_sort.append((time.perf_counter() - t0) * 1e6)
            t_sort = t_sort[2:]
            rows.append(dict(N=N, step="group_set+rank1_reindex", us_median=float(np.median(t_sort)),
                             us_min=float(min(t_sort)), us_max=float(max(t_sort)), **info))
            print(f"  group_set + rank1_reindex (once per sort, host clock): median {np.median(t_sort):.1f} us "
                  f"(min {min(t_sort):.1f}, max {max(t_sort):.1f})", flush=True)
        for arm in ("window", "window_b"):
            for d in arms[arm]["systems"]:
                for x in d.values():
                    x.free()
            arms[arm]["h"].close()
    if args.out:
        json.dump(rows, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
