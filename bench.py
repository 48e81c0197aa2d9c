#!/usr/bin/env python
"""bench.py -- cavity-force + Bussi step throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one 1M-particle (+1 photon) synthetic charged box:
the cavity force (dipole reduce + per-particle force + photon force + energies) and the
BussiReservoir thermostat (KE reduce + alpha + velocity rescale).  Prints ONE JSON line (rank 0).

  value      M particle-steps/s of cavb200_step -- force + thermostat in ONE launch, the north-star
             "one HBM round trip per particle per step" path -- whole job, inputs resident in HBM,
             CUDA-event timed on the launching stream, max over ranks.
  roofline   the dominant kernel (k_split_folder, the only kernel of a step): algorithmic 148 B/particle over
             its average launch duration (event span / K), against MEASURED_PEAKS.json hbm_gbs; next to it the
             kernel's own globaltimer stamps (kernel_ms_device) and the isolated figure (events around every launch)
  separate_calls / separate_calls_index_list   the same work as the two calls HOOMD's integrator makes
             (cavb200_force, then cavb200_bussi), with the group as a window and as HOOMD's index list
  e2e        same metric through the host-buffer C-ABI calls (pinned host arrays in, host arrays out,
             H2D / D2H inside the timed region); three byte budgets, all declared
  fkt        BASELINE configs[4]: F(k,t) field sum, 1M particles x 64 wave vectors, with an FP64 roofline
             against a DFMA microbenchmark run in the same process
  sharded    (N > 1) BASELINE configs[3]: the 16M-particle box particle-sharded over the N GPUs, one
             160-byte record per rank per step over NVLink, with in-run parity against the CPU oracle
  small_n    (N = 1) BASELINE configs[0] size (501 particles) and a short sweep: GPU vs one CPU core
  cpu_baseline  (N = 1) the reference's own CPU code (oracle/_ref: src/CavityForceCompute.cc +
             src/BussiReservoirThermostat.h compiled verbatim) on the host cores, bounded sample

L2 hygiene: the timed loops rotate over `--systems` distinct systems (default 8 x 116 MB = 928 MB,
larger than the 126 MB L2), so no step finds its inputs in L2.

N > 1 (torchrun, one process per GPU): every rank runs an independent replica (BASELINE configs[2],
no data-path collective; "scaling": "weak"); rank 0 reports the aggregate; the sharded and F(k,t)
legs then use all N GPUs for ONE problem.

--dump-outputs DIR writes what the last timed cavb200_step of rank 0 returned to its caller as float64
.npy files (see dump_outputs), so that two builds run with the same arguments can be compared output
for output: every input is generated from fixed seeds.  The velocities and the reservoir's cumulative
energy carry every earlier step on the same handle and system, warm-up included, so two dumps are
comparable only when --n-mol, --systems, --warmup and --steps all match.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cav_hoomd_b200 import synth  # noqa: E402

METRIC = "cavity-force+Bussi M particle-steps/s"
UNIT = "M particle-steps/s"
OMEGAC, COUPLSTR, PHMASS = 0.01, 1e-3, 1.0
FORCE_BYTES, BUSSI_BYTES = 84, 64  # algorithmic bytes per particle (SURVEY.md 8d, DESIGN.md)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# NUMA placement of the pinned host buffers of the e2e path
# ---------------------------------------------------------------------------------------------
class NumaLocal:
    """Context manager: while the pinned host buffers of the e2e leg are allocated, bind this thread to the CPUs of
    the GPU's NUMA node so that the pinned pages land next to the GPU's PCIe root (the kernel allocates on the node
    of the calling thread) on a multi-socket host.  Affinity is restored on exit.  A no-op when sysfs reports no node
    for the device -- the case on this pool's boxes (one node, numa_node = -1), where the e2e step is 1.73-1.75 ms on
    boxes whose duplex PCIe rate measures ~97 GB/s and 2.5 ms on the occasional box that measures ~58 GB/s; the rates
    are reported next to the number (e2e.pcie)."""

    def __init__(self, gpu_index: int):
        self.info = {"numa_node": None, "bound": False}
        self._old = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = gpu_index
            if vis:
                try:
                    idx = int(vis.split(",")[gpu_index])
                except (ValueError, IndexError):
                    pass
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            bus = bus.lower()
            if len(bus.split(":")[0]) == 8:  # NVML pads the domain to 8 hex digits, sysfs uses 4
                bus = bus[4:]
            node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
            self.info["numa_node"] = node
            if node >= 0:
                cpus = set()
                for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
                self._cpus = cpus & os.sched_getaffinity(0)
            else:
                # sysfs reports no node (the case in this pool's containers): ask NVML for the CPUs closest to the GPU
                self._cpus = set()
                try:
                    ncpu = os.cpu_count() or 1
                    words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(idx), (ncpu + 63) // 64)
                    near = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
                    near &= os.sched_getaffinity(0)
                    if near and len(near) < len(os.sched_getaffinity(0)):
                        self._cpus = near
                        self.info["nvml_cpu_affinity"] = f"{len(near)} of {len(os.sched_getaffinity(0))} cpus"
                except Exception:
                    pass
        except Exception:
            self._cpus = set()

    def __enter__(self):
        if self._cpus and not os.environ.get("CAVB_BENCH_NO_NUMA"):
            try:
                self._old = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self._cpus)
                self.info["bound"] = True
            except OSError:
                self._old = None
        return self

    def __exit__(self, *a):
        if self._old is not None:
            os.sched_setaffinity(0, self._old)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML in a thread of this process
    (a sample every ~2 ms); nvidia-smi -lms as the fallback when pynvml is missing."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.nvml = None
        self.samples = []  # (sm_mhz, reasons bitmask)
        self.sm_max = None
        self._stop = threading.Event()
        self._thread = None

    def _visible_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self._visible_index()), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self._stop.is_set():
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.dev, n.NVML_CLOCK_SM))
                try:
                    rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.dev))
                except Exception:
                    rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev))
                self.samples.append((sm, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """Number of samples so far (to report how many fell inside a region)."""
        return len(self.samples) if self.nvml else len(self.rows)

    def stop(self, first=0, last=None):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if self.nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            n = self.nvml
            bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
            sel = self.samples[first:last] or self.samples
            sm = [x[0] for x in sel]
            reasons = sorted(k for k, b in bits.items() if any(x[1] & b for x in sel))
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.sm_max, "reasons": reasons,
                    "samples": len(sm), "source": "nvml, sampled during the timed regions"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU code on the host cores
# ---------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """One replica, one thread: `steps` x (reference cavity force + reference Bussi step)."""
    n_mol, replica, steps, kind, warm = args
    from oracle import oracle as O
    s = synth.make_system(n_mol, replica=replica)
    rng = np.random.default_rng(replica)
    dof = 3.0 * n_mol - 3.0
    draws = [(rng.standard_normal(), rng.gamma((dof - 1) / 2)) for _ in range(steps)]
    if kind == "reference":
        ro = O.RefOracle()
        hc = ro.cavity_open(s.N, s.box, s.L_typeid, OMEGAC, COUPLSTR, PHMASS)
        ro.lib.ref_cavity_load(hc, O._d(s.pos), O._d(s.charge), O._i(s.image))
        hb = ro.bussi_open(s.vel, np.arange(n_mol, dtype=np.uint32), dof, synth.KT_100K, synth.TAU_5PS)
        for k in range(max(warm, 1)):  # warm-up (page faults)
            ro.lib.ref_cavity_compute(hc, 1)
            if warm > 1:
                ro.bussi_step(hb, 10**6 + k, synth.DT_1FS, 0.0, (dof - 1) / 2)
        t0 = time.perf_counter()
        for k in range(steps):
            ro.lib.ref_cavity_compute(hc, 1)
            ro.bussi_step(hb, k, synth.DT_1FS, draws[k][0], draws[k][1])
        dt = time.perf_counter() - t0
    else:
        co = O.COracle()
        idx = np.arange(n_mol, dtype=np.uint32)
        res = np.zeros(2)
        co.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, OMEGAC, COUPLSTR, PHMASS)
        t0 = time.perf_counter()
        for k in range(steps):
            co.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, OMEGAC, COUPLSTR, PHMASS)
            co.bussi_step(s.vel, idx, dof, synth.DT_1FS, synth.KT_100K, synth.TAU_5PS, draws[k][0], draws[k][1], res)
        dt = time.perf_counter() - t0
    return s.N * steps, dt


def cpu_reference_throughput(n_mol: int, steps: int, cores: int, warm: int = 1):
    """Aggregate M particle-steps/s of `cores` concurrent single-threaded replicas (the reference CPU
    path is single-threaded; its authors run one core per replica, reference submit.sh:7)."""
    import multiprocessing as mp
    from oracle import oracle as O
    O.build()
    kind = "reference" if O.have_ref() else "port"
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(n_mol, r, steps, kind, warm) for r in range(cores)])
    wall = time.perf_counter() - t0
    # every worker times only its own compute loop; the job rate is the sum of per-replica rates
    rate = sum(n / dt for n, dt in res) / 1e6
    # one replica alone on the machine (SURVEY.md 8d asks for both): the per-core rate without the others
    # competing for memory bandwidth
    with ctx.Pool(1) as pool:
        n1, dt1 = pool.map(_cpu_worker, [(n_mol, 0, max(3, min(steps, 60) // 3), kind, 1)])[0]
    return dict(value=rate, unit=UNIT, cores=cores, kind=kind,
                sample=f"{cores} concurrent 1-thread replicas x {steps} steps of the {n_mol + 1}-particle box "
                       f"(cavity force + Bussi), wall {wall:.1f} s incl. setup",
                single_process={"value": n1 / dt1 / 1e6, "unit": UNIT, "cores": 1,
                                "sample": f"1 replica x {max(3, min(steps, 60) // 3)} steps, alone on the host"})


WORKLOAD = ("synthetic {n}-particle charged box + 1 photon, CavityForce g=1e-3 omegac=0.01 + BussiReservoir kT=100K "
            "tau=5ps (BASELINE configs[1])")
L2_NOTE = ("inputs larger than the last-level cache: no step works on the system of the previous step (B200 arm: rotation "
           "over 8 systems x 116 MB = 928 MB > 126 MB L2; reference arm: one 116 MB system per host core)")


def bench_config(n_mol, world):
    """The SAME dictionary on both arms (the driver compares them): what is computed, on which data."""
    w = WORKLOAD.format(n=n_mol)
    if world > 1:
        w += f"; {world} independent replicas, one per GPU (configs[2])"
    return {"workload": w, "l2": L2_NOTE}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    cores = min(cores, 128)
    # a reference step of the 1M box is ~45 ms on one core: K timed steps after W warm-up steps per replica, K bounded
    # so that the run ends within minutes (every step is the full 1M-particle workload)
    steps = max(1, min(args.steps, 400))
    warm = max(1, min(args.warmup, 10))
    t0 = time.perf_counter()
    out = cpu_reference_throughput(args.n_mol, steps, cores, warm)
    ms = 1e3 * (args.n_mol + 1) * cores / (out["value"] * 1e6)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {
        "impl": "reference", "metric": METRIC, "value": out["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.n_mol, world),
        "details": {"arm": "the reference's own CPU classes (oracle/_ref: src/CavityForceCompute.cc + "
                           "src/BussiReservoirThermostat.h compiled verbatim) on the host cores, one single-threaded "
                           "replica per core (how the authors run it, reference submit.sh:7)"},
        "cpu_baseline": out,
        "e2e": {"value": out["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    _LINES.append(json.dumps(line))
    return 0


def ncu_traffic(n_mol):
    """dram__bytes_read.sum + dram__bytes_write.sum of the step kernel, per launch, from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json; a number measured under the profiler, so it is
    read from the committed summary, never taken live).  None when the capture is for another size."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            t = json.load(fh)
        if int(t.get("n_mol", -1)) != int(n_mol):
            return None, None
        return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"]), t.get("source")
    except Exception:
        return None, None


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
class DeviceSystem:
    """One particle system resident in HBM, HOOMD layouts."""

    def __init__(self, capi, s):
        self.N = s.N
        self.box = s.box
        self.L_typeid = s.L_typeid
        self.pos = capi.DeviceArray.from_numpy(s.pos)
        self.charge = capi.DeviceArray.from_numpy(s.charge)
        self.image = capi.DeviceArray.from_numpy(s.image)
        self.vel = capi.DeviceArray.from_numpy(s.vel)
        self.force = capi.DeviceArray((s.N, 4), np.float64)


DUMP_ROWS = 1 << 19  # per-particle arrays of larger systems are dumped as this many rows: 2 x 16 MB


def dump_outputs(out_dir, h, d, st):
    """What the last cavb200_step handed its caller: the force array and the rescaled velocities of the system it ran
    on, the energies, dipole and photon index (cavb200_force_read) and the thermostat record ke, alpha, instantaneous,
    cumulative, err (cavb200_bussi_read).  A system of more than DUMP_ROWS particles contributes a fixed, seeded sample
    of rows that always holds the last one (the photon of the bench's systems)."""
    os.makedirs(out_dir, exist_ok=True)
    force, vel = d.force.numpy(st), d.vel.numpy(st)
    if d.N > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(d.N - 1, DUMP_ROWS - 1, replace=False))
        rows = np.append(rows, d.N - 1)
        force, vel = force[rows], vel[rows]
    en, dip, ph = h.force_read(st)
    bo = h.bussi_read(st)
    out = {"force": force, "vel": vel, "energies": en, "dipole": dip, "photon_idx": [ph],
           "bussi": [bo[k] for k in ("ke", "alpha", "instantaneous", "cumulative", "err")]}
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


class Ctx:
    """What every leg of the B200 arm needs."""

    def __init__(self, args):
        from cav_hoomd_b200 import capi
        self.capi = capi
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist  # plumbing only: barrier + max over ranks (+ bootstrap blobs of the sharded leg)
            import datetime
            dist.init_process_group(backend="gloo", timeout=datetime.timedelta(seconds=600))
            self.dist = dist
        if capi.device_count() < 1:
            raise RuntimeError("bench.py: no CUDA device; the product has no CPU fallback")
        self.h = capi.Handle(self.local_rank)
        self.stream = capi.Stream()
        self.st = self.stream.ptr
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        self.capi.sync()
        if self.dist is not None:
            self.dist.barrier()

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return vals if len(vals) > 1 else vals[0]
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        out = tuple(float(x) for x in t)
        return out if len(out) > 1 else out[0]

    def timed(self, fn, steps, k0=0, gate=True, handle=None):
        """CUDA-event time (ms, max over ranks) of fn(k0) ... fn(k0 + steps - 1) on the launching stream, and the
        handle's launch count over the region.  gate: a one-thread delay kernel holds the stream while the host
        enqueues the launches, and the start event is recorded BEHIND it, so the region measures the device working
        through a non-empty queue -- the steady state of an MD loop, where the host runs ahead -- instead of the
        host's launch latency at the head of a short region (with 20 steps that head was 2.6 us per step)."""
        capi, h = self.capi, handle or self.h
        e0, e1 = capi.Event(), capi.Event()
        self.barrier()
        l0 = h.launch_count
        if gate:
            h.debug_delay(min(100_000_000, 100_000 + 12_000 * min(steps, 4000)), self.st)
        e0.record(self.st)
        for k in range(steps):
            fn(k0 + k)
        e1.record(self.st)
        ms = e1.elapsed_ms_since(e0)
        capi.sync()
        launches = h.launch_count - l0
        ms = self.max_over_ranks(ms)
        self.barrier()
        return ms, launches


def leg_fkt(cx, n_mol):
    """BASELINE configs[4]: F(k,t) on a 1M-particle trajectory, 64 wave vectors, 1000 time origins.
    rho[t][k] = sum_j exp(i k.r_j(t)) for T frames per launch (two rotating frame buffers, larger than L2), then the
    1000 x 1000 origin/lag table.  Roofline: the kernel is FP64-pipe bound (DESIGN.md 3.4) -- 17 FP64 instructions per
    (particle, k) pair (3 for k.r, 4 for the reduction to |r| <= pi/512, 6 for sin r and cos r, 4 FMAs that rotate by the
    table entry and accumulate; 13 of them fused multiply-adds = 30 flops) -- against the DFMA rate of this device measured
    by cavb200_debug_fp64_peak in this run."""
    capi, h, st = cx.capi, cx.h, cx.st
    N, K, T, ORIGINS = n_mol + 1, 64, 32, 1000
    FP64_PER_PAIR, FLOPS_PER_PAIR = 17, 30
    base = synth.make_system(n_mol, replica=cx.rank)
    rng = np.random.default_rng(7 + cx.rank)
    kvec = synth.fibonacci_sphere(K) * 1.0
    d_k = capi.DeviceArray.from_numpy(kvec)
    frames = np.empty((T, N, 4))
    cur = base.pos.copy()
    for t in range(T):
        cur[:, :3] += 0.05 * rng.standard_normal((N, 3))  # random walk, sigma 0.05 Bohr (SURVEY.md Appendix D)
        frames[t] = cur
    bufs = [capi.DeviceArray.from_numpy(frames) for _ in range(2)]  # 2 x 1 GB
    d_rho = capi.DeviceArray((T, K, 2), np.float64)

    # one GPU: 4 launches of T frames (128 frames); N GPUs: the 1000 frames in equal contiguous ranges per rank
    # (replicas.frames_for_rank, balanced), launches of at most T frames, no data-path collective, time = max over ranks
    from cav_hoomd_b200 import replicas
    blocks = [(0, T)] * 4 if cx.world == 1 else replicas.frames_for_rank(ORIGINS, cx.rank, cx.world, block=T, balanced=True)

    def launch(k):
        h.rhok(bufs[k & 1], 4, N * 4, N, blocks[k % len(blocks)][1], d_k, K, d_rho, st)

    for k in range(3):
        launch(k)
    capi.sync()
    n_launch = len(blocks)
    ms, launches = cx.timed(launch, n_launch, gate=True)
    frames_done = n_launch * T if cx.world == 1 else ORIGINS
    ms_per_frame = ms / frames_done
    pairs_per_s = N * K / (ms_per_frame * 1e-3)
    rho = d_rho.numpy(st)
    # the tracker's live use (reference analysis.py:34-47 called once per sampling period inside a run): one frame per
    # call, each call on a different frame of the rotating buffers
    d_rho1 = capi.DeviceArray((1, K, 2), np.float64)

    def launch_one(k):
        h.rhok(bufs[k & 1].ptr + (k % T) * N * 32, 4, N * 4, N, 1, d_k, K, d_rho1, st)

    live = None
    if cx.world == 1:
        for k in range(3):
            launch_one(k)
        ms_live, _ = cx.timed(launch_one, 16, gate=True)
        live = {"ms_per_call": ms_live / 16, "note": "T = 1: one 1M-particle frame x 64 wave vectors per call (k_rhok + k_rhok_fold), 16 calls back to back"}
    big = np.ascontiguousarray(np.tile(rho, (ORIGINS // T + 1, 1, 1))[:ORIGINS])
    d_big = capi.DeviceArray.from_numpy(big)
    d_F = capi.DeviceArray((ORIGINS, ORIGINS), np.float64)
    h.fkt(d_big, ORIGINS, K, ORIGINS, ORIGINS, d_F, st)
    ms_corr, _ = cx.timed(lambda k: h.fkt(d_big, ORIGINS, K, ORIGINS, ORIGINS, d_F, st), 3, gate=False)
    ms_corr /= 3
    dfma = h.debug_fp64_peak()
    peak_tflops = 2.0 * dfma / 1e12
    achieved = 2.0 * FP64_PER_PAIR * pairs_per_s / cx.world / 1e12  # per GPU, FMA-equivalent flops
    out = {
        "workload": f"F(k,t): {N} particles x {K} wave vectors per frame, {ORIGINS} time origins (BASELINE configs[4]); "
                    f"{T} frames per launch, float64 Scalar4 positions resident in HBM (2 rotating buffers x {frames.nbytes >> 20} MB)",
        "ms_per_frame": ms_per_frame, "pairs_per_s": pairs_per_s, "frames_timed": frames_done, "gpu_launches": launches,
        "live_single_frame": live,
        "seconds_for_1000_origins": ms_per_frame * 1e-3 * ORIGINS * (1 if cx.world == 1 else 1) + ms_corr * 1e-3,
        "ms_origin_lag_table_1000x1000": ms_corr,
        "position_GBs": 32 * N / (ms_per_frame * 1e-3) / 1e9,
        "roofline": {"bound": "fp64", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
                     "frac": achieved / peak_tflops, "traffic": None, "kernel": "k_rhok<4, false>",
                     "convention": f"FP64-pipe issue slots, counted as fused multiply-adds (2 flops each): {FP64_PER_PAIR} "
                                   f"FP64 instructions per (particle, k) pair (3 for k.r, 4 reduction to |r| <= pi/512, 6 for sin r and cos r, 4 rotate-by-table-entry-and-accumulate; round 1 and early round 2 needed 26); arithmetic flops are {FLOPS_PER_PAIR} per pair",
                     "arithmetic_TFLOPs": FLOPS_PER_PAIR * pairs_per_s / cx.world / 1e12,
                     "peak_source": "measured in this run: cavb200_debug_fp64_peak (DFMA microbenchmark, "
                                    "cav_hoomd_b200/csrc/debug.cu), best of 4"},
    }
    if cx.world > 1:
        out["multi_gpu"] = {"n_gpus": cx.world, "partition": f"equal contiguous ranges of frames per rank in launches of at most {T}, no collective in the data path",
                            "seconds_for_1000_frame_field_sum": ms * 1e-3, "pairs_per_s": N * K * ORIGINS / (ms * 1e-3)}
    for b in bufs:
        b.free()
    return out


def leg_small_n(cx, params):
    """BASELINE configs[0] runs 500 molecular particles + 1 photon (SURVEY.md section 0).  At that size a step is launch
    bound on the GPU and cache resident on the CPU: report both, a short N sweep and the crossover."""
    capi, h, st = cx.capi, cx.h, cx.st
    from oracle import oracle as O  # cpu_baseline leg: the reference's CPU classes as the comparison
    rows = []
    ref = O.RefOracle() if O.have_ref() else None
    co = O.COracle()
    for n_mol in (500, 2000, 8000, 32000, 131072):
        s = synth.make_system(n_mol, replica=3)
        d = DeviceSystem(capi, s)
        dof = 3.0 * n_mol - 3.0
        a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof, 0.1, (dof - 1) / 2)

        def both(k):
            h.force(d.pos, d.charge, d.image, d.force, s.N, s.box, s.L_typeid, params, st)
            h.bussi(d.vel, None, 0, n_mol, a, st)

        def fused(k):
            h.step(d.pos, d.charge, d.image, d.force, d.vel, s.N, s.box, s.L_typeid, params, 0, n_mol, a, st)

        for k in range(5):
            both(k)
            fused(k)
        K = 400
        ms_both, _ = cx.timed(both, K)
        ms_fused, _ = cx.timed(fused, K)
        # the same 100 steps as ONE CUDA graph launch (what a launch-bound inner loop should do)
        g = h.graph_capture(st, lambda: [both(k) for k in range(100)])
        h.graph_launch(g, st)
        ms_graph, _ = cx.timed(lambda k: h.graph_launch(g, st), 4, gate=False)
        h.graph_destroy(g)
        # the reference's CPU classes, one core, same system
        idx = np.arange(n_mol, dtype=np.uint32)
        reps = max(20, min(4000, int(2e6 // max(n_mol, 1))))
        if ref is not None:
            hc = ref.cavity_open(s.N, s.box, s.L_typeid, OMEGAC, COUPLSTR, PHMASS)
            ref.lib.ref_cavity_load(hc, O._d(s.pos), O._d(s.charge), O._i(s.image))
            hb = ref.bussi_open(s.vel, idx, dof, synth.KT_100K, synth.TAU_5PS)
            ref.lib.ref_cavity_compute(hc, 1)
            t0 = time.perf_counter()
            for k in range(reps):
                ref.lib.ref_cavity_compute(hc, 1)
                ref.bussi_step(hb, k, synth.DT_1FS, 0.1, (dof - 1) / 2)
            cpu_us = 1e6 * (time.perf_counter() - t0) / reps
            kind = "reference"
        else:
            v = s.vel.copy()
            res = np.zeros(2)
            t0 = time.perf_counter()
            for k in range(reps):
                co.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, OMEGAC, COUPLSTR, PHMASS)
                co.bussi_step(v, idx, dof, synth.DT_1FS, synth.KT_100K, synth.TAU_5PS, 0.1, (dof - 1) / 2, res)
            cpu_us = 1e6 * (time.perf_counter() - t0) / reps
            kind = "port"
        rows.append({"n_particles": s.N, "gpu_two_calls_us": 1e3 * ms_both / K, "gpu_one_launch_us": 1e3 * ms_fused / K,
                     "gpu_two_calls_graph_us": 1e3 * ms_graph / 400, "cpu_one_core_us": cpu_us, "cpu_kind": kind})
    # crossover: the particle count above which the GPU step (two calls, stream launches) is faster than one CPU core
    cross = None
    for lo, hi in zip(rows, rows[1:]):
        dl, dh = lo["cpu_one_core_us"] - lo["gpu_two_calls_us"], hi["cpu_one_core_us"] - hi["gpu_two_calls_us"]
        if dl < 0 <= dh:
            cross = lo["n_particles"] + (hi["n_particles"] - lo["n_particles"]) * (-dl) / (dh - dl)
    if cross is None and rows[0]["cpu_one_core_us"] >= rows[0]["gpu_two_calls_us"]:
        cross = f"below {rows[0]['n_particles']}"
    return {"note": "cavity force + Bussi step at the reference authors' own system size (configs[0]: 500 particles + photon) "
                    "and up: calls over at most 768 particles run as ONE CTA (k_small, no inter-CTA hand-off), calls with the force "
                    "in them up to 8192 particles as ONE thread-block cluster (k_cluster, records through distributed shared "
                    "memory); both are bound by launch latency (python/ctypes host loop; the CUDA-graph column replays 100 steps per launch); the CPU "
                    "reference runs out of cache",
            "sweep": rows, "gpu_faster_than_one_core_above_n_particles": cross}


def leg_sharded(cx, params):
    """BASELINE configs[3]: the 16M-particle box sharded over the ranks' GPUs.  Every rank owns a contiguous block; per
    step ONE 160-byte record per rank crosses NVLink, stored straight into every peer's mailbox from inside the
    persistent kernel (csrc/shard.cu, mode nvlink) -- or an ncclAllGather of the same records (mode nccl).  In-run parity:
    a 200k-particle system sharded the same way against the UNSHARDED CPU oracle, and all ranks bitwise identical."""
    capi, dist, rank, world = cx.capi, cx.dist, cx.rank, cx.world
    from cav_hoomd_b200 import shard
    import torch
    N_TOTAL, CHECK_N, STEPS = 16_000_000, 200_000, 50
    out = {"n_particles": N_TOTAL + 1, "n_gpus": world, "steps": STEPS}
    for mode in ("nvlink", "nccl"):
        res = {}
        try:
            h = capi.Handle(cx.local_rank)
            shard.bootstrap(h, dist, mode)
            st = capi.Stream()
            # ---- parity ----
            s = synth.make_system(CHECK_N)
            sub, off, (first, n) = shard.shard_system(s, rank, world)
            dof = 3.0 * CHECK_N - 3.0
            a = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof, 0.3, (dof - 1) / 2)
            dev = {k: capi.DeviceArray.from_numpy(getattr(sub, k)) for k in ("pos", "charge", "image", "vel")}
            d_f = capi.DeviceArray((max(sub.N, 1), 4), np.float64)
            h.bussi_reset(st.ptr)
            h.shard_step(dev["pos"], dev["charge"], dev["image"], d_f, dev["vel"], sub.N, off, s.box, s.L_typeid, params,
                         first, n, a, st.ptr)
            en, dip, ph = h.force_read(st.ptr)
            bo = h.bussi_read(st.ptr)
            f, v = d_f.numpy(st.ptr)[:sub.N], dev["vel"].numpy(st.ptr)
            if rank == 0:
                from oracle import oracle as O  # the checker
                co = O.COracle()
                ref = co.cavity_force(s.pos, s.charge, s.image, s.box, s.L_typeid, OMEGAC, COUPLSTR)
                vref = s.vel.copy()
                alpha, ke = co.bussi_step(vref, np.arange(CHECK_N, dtype=np.uint32), dof, synth.DT_1FS, synth.KT_100K,
                                          synth.TAU_5PS, a.r_normal, a.gamma_draw, np.zeros(2))
                blob = [[ref["force"], vref, ref["energies"], alpha, ref["photon_idx"]]]
            else:
                blob = [None]
            dist.broadcast_object_list(blob, src=0)
            rf, rv, ren, ralpha, rph = blob[0]
            ok = bool(ph == rph and np.abs(f - rf[off:off + sub.N]).max() <= 1e-10 * np.abs(rf).max()
                      and np.allclose(en, ren, rtol=1e-10) and abs(bo["alpha"] - ralpha) <= 1e-12 * abs(ralpha)
                      and np.allclose(v, rv[off:off + sub.N], rtol=1e-12, atol=0))
            oks, scal = [None] * world, [None] * world
            dist.all_gather_object(oks, ok)
            dist.all_gather_object(scal, (en.tobytes(), dip.tobytes(), bo["alpha"], ph))
            res["parity_all_ranks"] = all(oks)
            res["ranks_bitwise_identical"] = all(x == scal[0] for x in scal)
            res["parity_check"] = f"{CHECK_N + 1} particles sharded over {world} ranks vs the unsharded CPU oracle (forces 1e-10, alpha / velocities 1e-12)"
            # ---- timing: this rank's block of the 16M box (synthetic; only the last rank holds the photon) ----
            lo, hi = shard.shard_bounds(N_TOTAL + 1, world)[rank]
            last = rank == world - 1
            n_loc_mol = (hi - lo) - (1 if last else 0)
            big = synth.make_system(n_loc_mol, replica=500 + rank, photon="last" if last else "absent")
            L = (N_TOTAL / synth.NUMBER_DENSITY) ** (1.0 / 3.0)
            dofb = 3.0 * N_TOTAL - 3.0
            ab = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dofb, 0.3, (dofb - 1) / 2)
            devb = {k: capi.DeviceArray.from_numpy(getattr(big, k)) for k in ("pos", "charge", "image", "vel")}
            d_fb = capi.DeviceArray((big.N, 4), np.float64)

            def one(k):
                h.shard_step(devb["pos"], devb["charge"], devb["image"], d_fb, devb["vel"], big.N, lo, (L, L, L),
                             big.L_typeid, params, 0, n_loc_mol, ab, st.ptr)

            for k in range(5):
                one(k)
            st.sync()
            dist.barrier()
            e0, e1 = capi.Event(), capi.Event()
            e0.record(st.ptr)
            for k in range(STEPS):
                one(k)
            e1.record(st.ptr)
            ms = e1.elapsed_ms_since(e0)
            bo = h.bussi_read(st.ptr)
            t = torch.tensor([ms], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item()) / STEPS
            res.update({"ms_per_step": ms, "value": (N_TOTAL + 1) / (ms * 1e-3) / 1e6, "unit": UNIT,
                        "frac_per_gpu": 148 * (N_TOTAL + 1) / world / (ms * 1e-3) / 1e9 / cx.peak,
                        "err": bo["err"], "l2": f"{116 * (hi - lo) / 1e6:.0f} MB per rank (larger than L2)"})
            h.close()
            for x in list(dev.values()) + list(devb.values()) + [d_f, d_fb]:
                x.free()
        except Exception as e:  # a mode that cannot run on this box (e.g. no libnccl) is reported, not fatal
            res["unavailable"] = f"{type(e).__name__}: {e}"[:300]
        dist.barrier()
        out[mode] = res
    best = min((m for m in ("nvlink", "nccl") if "ms_per_step" in out[m]), key=lambda m: out[m]["ms_per_step"], default=None)
    if best:
        out.update({"mode": best, **{k: out[best][k] for k in ("ms_per_step", "value", "unit", "frac_per_gpu",
                                                                 "parity_all_ranks", "ranks_bitwise_identical")}})
    return out


def run_b200(args):
    cx = Ctx(args)
    capi, h, st, rank, world, local_rank = cx.capi, cx.h, cx.st, cx.rank, cx.world, cx.local_rank
    if args.variant is not None:
        h.set_tuning(variant=args.variant)
    if args.threads:
        h.set_tuning(threads=args.threads)
    if args.ctas_per_sm:
        h.set_tuning(ctas_per_sm=args.ctas_per_sm)
    if args.unroll:
        h.set_tuning(unroll=args.unroll)

    n_mol = args.n_mol
    base = synth.make_system(n_mol, replica=rank)
    N = base.N
    systems, host_pv = [], []
    for k in range(args.systems):
        s = base if k == 0 else synth.make_system(n_mol, replica=rank + 1000 * k)
        systems.append(DeviceSystem(capi, s))
        host_pv.append((s.pos, s.vel))
    params = capi.Params.make(OMEGAC, COUPLSTR, PHMASS)
    dof = 3.0 * n_mol - 3.0
    rng = np.random.default_rng(1234 + rank)
    bargs = [capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof, rng.standard_normal(),
                            rng.gamma((dof - 1) / 2)) for _ in range(64)]
    # the thermostatted group as HOOMD hands it out: an index list (ParticleGroup::getIndexArray) -- the whole range, and
    # the range with one particle missing in the middle (where the photon sits once HOOMD's SFC sorter has run)
    gidx_range = capi.DeviceArray.from_numpy(np.arange(n_mol, dtype=np.uint32))
    hole = np.delete(np.arange(n_mol, dtype=np.uint32), n_mol // 2)
    gidx_hole = capi.DeviceArray.from_numpy(hole)
    dof_hole = 3.0 * (n_mol - 1) - 3.0
    bargs_hole = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof_hole, 0.1, (dof_hole - 1) / 2)

    def step(k):
        d = systems[k % len(systems)]
        h.step(d.pos, d.charge, d.image, d.force, d.vel, N, d.box, d.L_typeid, params, 0, n_mol, bargs[k % 64], st)

    def two_calls(k, gidx=None, n=None, a=None):
        d = systems[k % len(systems)]
        h.force(d.pos, d.charge, d.image, d.force, N, d.box, d.L_typeid, params, st)
        h.bussi(d.vel, gidx, 0, n_mol if n is None else n, a or bargs[k % 64], st)

    # warm-up (>= 3), every path
    W = max(args.warmup, 3)
    for k in range(W):
        two_calls(k)
        two_calls(k, gidx_range)
        step(k)
    capi.sync()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)
    m0 = sampler.mark()
    K = args.steps
    ms_fused, launches_fused = cx.timed(step, K, k0=W)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h, systems[(W + K - 1) % len(systems)], st)
    ms_fused_hostpaced, _ = cx.timed(step, K, k0=W + K, gate=False)
    ms_sep, launches_sep = cx.timed(two_calls, K, k0=W)
    ms_sep_list, _ = cx.timed(lambda k: two_calls(k, gidx_range), K, k0=W)
    ms_sep_hole, _ = cx.timed(lambda k: two_calls(k, gidx_hole, n_mol - 1, bargs_hole), K, k0=W)

    # per-launch device timestamps of the step kernel (first CTA start -> last CTA end, globaltimer), taken in a
    # second pass of min(K, 1000) launches with the two atomics per CTA switched on (tuning stamps = 2)
    KR = min(K, 1000)
    h.set_tuning(stamps=2)
    h.debug_launch_ring(reset=True, read=False)
    cx.timed(step, KR, k0=W)
    ring, ep = h.debug_launch_ring()
    h.set_tuning(stamps=0)
    slots = [(ep - i) & 2047 for i in range(KR)][::-1]
    t_start = ring[slots, 0].astype(np.float64)
    t_end = ring[slots, 1].astype(np.float64)
    ring_ok = bool(np.all(ring[slots, 1] > 0) and np.all(ring[slots, 0] != np.uint64(0xFFFFFFFFFFFFFFFF)))
    dev_ms = (t_end - t_start) * 1e-6 if ring_ok else np.array([float("nan")])
    period_ms = np.diff(t_start) * 1e-6 if (ring_ok and KR > 1) else dev_ms

    # per-kernel durations with CUDA events around every launch (breaks the launch overlap: "isolated")
    evs = [(capi.Event(), capi.Event()) for _ in range(min(K, 200))]
    capi.sync()
    for k, (a, b) in enumerate(evs):
        a.record(st)
        step(k)
        b.record(st)
    capi.sync()
    t_step = float(np.mean([b.elapsed_ms_since(a) for a, b in evs]))
    # what the same two events measure around a kernel that does nothing (one CTA, returns at once): the part of every
    # "isolated" figure that is the launch and the two event records, not the kernel
    for k, (a, b) in enumerate(evs):
        a.record(st)
        h.debug_delay(0, st)
        b.record(st)
    capi.sync()
    t_empty = float(np.mean([b.elapsed_ms_since(a) for a, b in evs]))
    evs = [(capi.Event(), capi.Event(), capi.Event()) for _ in range(min(K, 200))]
    for k, (a, b, c) in enumerate(evs):
        d = systems[k % len(systems)]
        a.record(st)
        h.force(d.pos, d.charge, d.image, d.force, N, d.box, d.L_typeid, params, st)
        b.record(st)
        h.bussi(d.vel, None, 0, n_mol, bargs[k % 64], st)
        c.record(st)
    capi.sync()
    t_force = float(np.mean([b.elapsed_ms_since(a) for a, b, c in evs]))
    t_bussi = float(np.mean([c.elapsed_ms_since(b) for a, b, c in evs]))
    # the two calls alone, back to back (launch overlap intact): cavb200_force only, cavb200_bussi only
    ms_force_only, _ = cx.timed(lambda k: h.force(systems[k % 8].pos, systems[k % 8].charge, systems[k % 8].image,
                                                  systems[k % 8].force, N, base.box, base.L_typeid, params, st), K, k0=W)
    ms_bussi_only, _ = cx.timed(lambda k: h.bussi(systems[k % 8].vel, None, 0, n_mol, bargs[k % 64], st), K, k0=W)

    # whole MD step of the repo's velocity-Verlet harness (SURVEY.md 8f.1 / 8f.2; not the headline metric):
    #   folded  nvt_step_one ; force ; nvt_step_two          thermostat inside the kicks, 340 B/particle
    #   rank1   nvt_step_one_rank1 ; force_rank1 ; nvt_step_two_rank1   cavity force never stored, 260 B/particle
    #   rank1_reduce_in_step_one   md_step_one ; nvt_step_two_rank1       next dipole reduce inside step one, 220 B/particle
    #   one_launch                 md_step_fused                          step two of t-1 + step one of t, 148 B/particle
    # sanity first: the timed regions above must have produced finite forces and a sane alpha (not a timing of nothing)
    step(0)
    en, dip, ph = h.force_read(st)
    bo = h.bussi_read(st)
    assert ph == n_mol and np.isfinite(en).all() and bo["err"] == 0.0 and 0.5 < bo["alpha"] < 1.5, (ph, en, bo)
    assert h.fault_count == 0
    md = {}
    md_steps = max(20, min(K, 100))
    for kind, nbytes in (("folded", 340), ("rank1", 260), ("rank1_reduce_in_step_one", 220), ("one_launch", 148)):
        def md_step(k):
            d = systems[k % len(systems)]
            a = bargs[k % len(bargs)]
            if kind == "folded":
                h.nvt_step_one(d.pos, d.vel, d.force, N, synth.DT_1FS, 0, n_mol, a, st)
                h.force(d.pos, d.charge, d.image, d.force, N, d.box, d.L_typeid, params, st)
                h.nvt_step_two(d.vel, d.force, N, synth.DT_1FS, 0, n_mol, st)
            elif kind == "rank1":
                h.nvt_step_one_rank1(d.pos, d.vel, None, d.charge, N, synth.DT_1FS, d.L_typeid, COUPLSTR, 0, n_mol, a, st)
                h.force_rank1(d.pos, d.charge, d.image, N, d.box, d.L_typeid, params, st)
                h.nvt_step_two_rank1(d.vel, None, d.charge, d.pos, N, synth.DT_1FS, d.L_typeid, COUPLSTR, 0, n_mol, st)
            elif kind == "rank1_reduce_in_step_one":
                h.md_step_one(d.pos, d.vel, None, d.charge, d.image, N, synth.DT_1FS, d.box, d.L_typeid, params, 0, n_mol, a, st)
                h.nvt_step_two_rank1(d.vel, None, d.charge, d.pos, N, synth.DT_1FS, d.L_typeid, COUPLSTR, 0, n_mol, st)
            else:
                h.md_step_fused(d.pos, d.vel, None, d.charge, d.image, N, synth.DT_1FS, d.box, d.L_typeid, params, 0, n_mol, a, st)
        # (the harness integrates: every variant starts from the same fresh positions and velocities)
        for d, (hp, hv) in zip(systems, host_pv):
            d.pos.upload(hp, st)
            d.vel.upload(hv, st)
            h.bussi_ke(d.vel, None, 0, n_mol, st)
        h.force_rank1(systems[0].pos, systems[0].charge, systems[0].image, N, base.box, base.L_typeid, params, st)
        for k in range(5):
            md_step(k)
        ms, _ = cx.timed(md_step, md_steps)
        ms /= md_steps
        md[kind] = {"ms_per_step": ms, "algorithmic_bytes_per_particle": nbytes,
                    "achieved_GBs": nbytes * N / (ms * 1e-3) / 1e9, "value": world * N / (ms * 1e-3) / 1e6, "unit": UNIT}
    clocks = sampler.stop(first=m0) if rank == 0 else None  # samples from the start of the first timed region to here

    # e2e: host-buffer C-ABI calls, pinned host arrays, copies inside the timed region.  The driver holds E2E_SLOTS
    # independent systems on the host (replicas) and submits system k+1 before waiting for system k
    # (cavb200_step_host_submit_ex / _wait_ex), so the next upload runs under this download.  Three byte budgets:
    #   full_copy     every array every step: pos, charge, image, vel in; force, vel out       (84 B in, 64 B out / particle)
    #   (headline)    charge and image flagged "unchanged since the slot's last submit" (charges never change in an MD
    #                 run, images only when a particle crosses the box): pos, vel in; force, vel out    (64 B in, 64 B out)
    #   rank1_result  additionally the rank-1 result {Dq, F_L, energies} instead of the force array       (64 B in, 32 B out)
    e2e_steps = max(6, min(K, 24))
    E2E_SLOTS = 3
    pins = []
    numa = NumaLocal(local_rank)
    with numa:
        for r in range(E2E_SLOTS):
            pin = {k: capi.PinnedArray.from_numpy(getattr(base, k)) for k in ("pos", "charge", "image", "vel")}
            pin["force"] = capi.PinnedArray((N, 4), np.float64)
            pin["force"].array[:] = 0.0  # touch the pages while bound
            pins.append(pin)
    pin, pin_force = pins[0], pins[0]["force"]
    KEEP = capi.Handle.HOST_KEEP_CHARGE | capi.Handle.HOST_KEEP_IMAGE

    def run_pipelined(steps, flags):
        def submit(k):
            q = pins[k % E2E_SLOTS]
            h.step_host_submit_ex(k % E2E_SLOTS, q["pos"], q["charge"], q["image"], q["force"], q["vel"], N, base.box,
                                  base.L_typeid, params, 0, n_mol, bargs[k % len(bargs)], flags)
        results = []
        for k in range(min(E2E_SLOTS - 1, steps)):
            submit(k)
        for k in range(steps):
            if k + E2E_SLOTS - 1 < steps:
                submit(k + E2E_SLOTS - 1)
            results.append(h.step_host_wait_ex(k % E2E_SLOTS))
        return results

    def e2e_rounds(flags):
        # three rounds of e2e_steps steps, the median round is reported (one host-side hiccup in a 40 ms region moves
        # a single round by 20 %; all three are in the JSON line)
        run_pipelined(E2E_SLOTS, flags)
        rounds = []
        for _ in range(3):
            cx.barrier()
            t0 = time.perf_counter()
            res = run_pipelined(e2e_steps, flags)
            capi.sync()
            rounds.append(time.perf_counter() - t0)
        assert all(np.isfinite(en).all() and bo["err"] == 0.0 and 0.5 < bo["alpha"] < 1.5 and r1["photon_idx"] == n_mol
                   for en, bo, r1 in res), res[-1]
        return cx.max_over_ranks(sorted(rounds)[1]), rounds

    e2e_full_s, rounds_full = e2e_rounds(0)        # also fills every slot's device copy of charge / image
    e2e_keep_s, rounds_keep = e2e_rounds(KEEP)
    e2e_rank1_s, rounds_rank1 = e2e_rounds(KEEP | capi.Handle.HOST_RANK1_RESULT)
    for k in range(2):
        h.step_host(pin["pos"], pin["charge"], pin["image"], pin_force, pin["vel"], N, base.box, base.L_typeid, params, 0,
                    n_mol, bargs[k])
    cx.barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        en, bo = h.step_host(pin["pos"], pin["charge"], pin["image"], pin_force, pin["vel"], N, base.box, base.L_typeid,
                             params, 0, n_mol, bargs[k % len(bargs)])
    capi.sync()
    e2e_sync_s = cx.max_over_ranks(time.perf_counter() - t0)

    def e2e_val(sec):
        return world * N * e2e_steps / sec / 1e6

    # raw PCIe rates of this box (pinned, 32 MB copies, one direction at a time and both together).  With N > 1 every
    # rank measures AT THE SAME TIME (barrier before each measurement), so the figures are what a rank gets while the
    # other ranks' copies load the same host memory and PCIe root complexes: the host-side limit of the e2e leg.
    lib = capi.load()
    nb = 32 * N
    s2 = capi.Stream()

    def rate(fn, reps=6):
        fn()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        capi.sync()
        return nb * reps / (time.perf_counter() - t0) / 1e9

    h2d = rate(lambda: lib.cavb200_memcpy_h2d(systems[0].pos.ptr, pin["pos"].ptr, nb, st))
    d2h = rate(lambda: lib.cavb200_memcpy_d2h(pin_force.ptr, systems[0].force.ptr, nb, st))

    def both():
        lib.cavb200_memcpy_h2d(systems[0].pos.ptr, pin["pos"].ptr, nb, st)
        lib.cavb200_memcpy_d2h(pin_force.ptr, systems[1].force.ptr, nb, s2.ptr)
    duplex = 2 * rate(both)
    rates = [(h2d, d2h, duplex)]
    if cx.dist is not None:
        rates = [None] * world
        cx.dist.all_gather_object(rates, (h2d, d2h, duplex))
    pcie = None
    if rank == 0:
        a = np.array(rates)
        h2d_r, d2h_r = float(a[:, 0].min()), float(a[:, 1].min())
        pcie = {"h2d_GBs": h2d_r, "d2h_GBs": d2h_r, "duplex_GBs": float(a[:, 2].min()),
                "floor_ms_per_step": {"full_copy": max((52 * N + 32 * n_mol) / (h2d_r * 1e6), (32 * N + 32 * n_mol) / (d2h_r * 1e6)),
                                      "headline": max((32 * N + 32 * n_mol) / (h2d_r * 1e6), (32 * N + 32 * n_mol) / (d2h_r * 1e6)),
                                      "rank1_result": max((32 * N + 32 * n_mol) / (h2d_r * 1e6), 32 * n_mol / (d2h_r * 1e6))},
                "note": "floor = the busier PCIe direction at the measured one-direction rate"
                        + (f"; {world} ranks copying concurrently: per-rank minimum shown, aggregate h2d {a[:, 0].sum():.0f} / d2h "
                           f"{a[:, 1].sum():.0f} / duplex {a[:, 2].sum():.0f} GB/s over the host's memory and PCIe roots -- the "
                           f"limiter of the e2e leg at this N (not a kernel or a collective)" if world > 1 else "")}
        if world > 1:
            pcie["per_rank_concurrent"] = {"h2d_GBs": [float(x) for x in a[:, 0]], "d2h_GBs": [float(x) for x in a[:, 1]],
                                           "duplex_GBs": [float(x) for x in a[:, 2]]}

    assert h.fault_count == 0

    # the other BASELINE configurations, measured in this same run
    for d in systems[2:]:
        for x in (d.pos, d.charge, d.image, d.vel, d.force):
            x.free()
    fkt = leg_fkt(cx, n_mol) if not args.no_fkt else None
    sharded = leg_sharded(cx, params) if world > 1 and not args.no_sharded else None
    small = leg_small_n(cx, params) if world == 1 and not args.no_small_n else None

    if rank != 0:
        return 0

    peak, peak_src = cx.peak, cx.peak_src
    STEP_BYTES = FORCE_BYTES + BUSSI_BYTES
    value = world * N * K / (ms_fused * 1e-3) / 1e6
    # the timed region holds nothing but K launches of the step kernel, so its CUDA-event span / K is that kernel's
    # average launch duration
    t_launch = ms_fused / K
    achieved = STEP_BYTES * N / (t_launch * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(n_mol)

    def frac_of(ms_total, nbytes, steps=K):
        return nbytes * steps / (ms_total * 1e-3) / 1e9 / peak

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": t_launch, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(n_mol, world),
        "details": {
            "path": "cavb200_step: cavity force + Bussi thermostat in one launch (split-phase kernel with a folder CTA), device-resident arrays",
            "timing": "CUDA events on the launching stream around K launches enqueued behind a one-thread gate kernel (the "
                      "device works through a non-empty queue, as in an MD loop where the host runs ahead); "
                      "host_paced_ms_per_step is the same region without the gate",
            "tuning": {k: h.get_tuning(k) for k in ("variant", "threads", "auto_threads", "ctas_per_sm", "unroll", "pdl")},
            "host_paced_ms_per_step": ms_fused_hostpaced / K,
        },
        "roofline": {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_split_folder (cavb200_step)",
            "algorithmic_bytes_per_particle": STEP_BYTES, "kernel_ms": t_launch, "peak_source": peak_src,
            "kernel_ms_device": {"mean": float(dev_ms.mean()), "median": float(np.median(dev_ms)),
                                 "launch_period_median": float(np.median(period_ms)), "launches": int(KR),
                                 "frac_at_period": STEP_BYTES * N / (float(np.median(period_ms)) * 1e-3) / 1e9 / peak,
                                 "note": "globaltimer stamps written by the kernel itself: first CTA start -> last CTA end "
                                         "(consecutive launches overlap by their programmatic-dependent-launch tail, so "
                                         "the start-to-start period is the throughput figure)"},
            "isolated": {"kernel_ms": t_step, "achieved": STEP_BYTES * N / (t_step * 1e-3) / 1e9,
                         "frac": STEP_BYTES * N / (t_step * 1e-3) / 1e9 / peak,
                         "empty_kernel_ms": t_empty,
                         "note": "CUDA events around every single launch (no launch overlap); empty_kernel_ms is the same "
                                 "pair of events around a kernel that returns at once"},
        },
        "separate_calls": {
            "value": world * N * K / (ms_sep * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_sep / K,
            "frac": frac_of(ms_sep, STEP_BYTES * N),
            "path": "cavb200_force + cavb200_bussi (the two calls HOOMD's integrator makes), contiguous group", "gpu_launches": launches_sep,
            "force_call": {"ms": ms_force_only / K, "frac": frac_of(ms_force_only, FORCE_BYTES * N)},
            "bussi_call": {"ms": ms_bussi_only / K, "frac": frac_of(ms_bussi_only, BUSSI_BYTES * n_mol)},
            "force_kernel": {"kernel_ms": t_force, "achieved": FORCE_BYTES * N / (t_force * 1e-3) / 1e9,
                             "frac": FORCE_BYTES * N / (t_force * 1e-3) / 1e9 / peak, "note": "isolated (events around every launch)"},
            "bussi_kernel": {"kernel_ms": t_bussi, "achieved": BUSSI_BYTES * n_mol / (t_bussi * 1e-3) / 1e9,
                             "frac": BUSSI_BYTES * n_mol / (t_bussi * 1e-3) / 1e9 / peak, "note": "isolated (events around every launch)"},
        },
        "separate_calls_index_list": {
            "path": "the same two calls with the thermostatted group passed as an index list (ParticleGroup::getIndexArray, what "
                    "the plugin class passes): 152 algorithmic B/particle, indices fetched one iteration ahead",
            "whole_range": {"ms_per_step": ms_sep_list / K, "frac": frac_of(ms_sep_list, (STEP_BYTES + 4) * N),
                            "vs_contiguous": ms_sep_list / ms_sep},
            "range_with_a_hole": {"ms_per_step": ms_sep_hole / K, "frac": frac_of(ms_sep_hole, (STEP_BYTES + 4) * N),
                                  "vs_contiguous": ms_sep_hole / ms_sep,
                                  "note": "one particle missing in the middle of the range (the photon after HOOMD's particle sort)"},
        },
        "harness_md_step": {"note": "kick+drift, cavity force, kick with the Bussi thermostat folded in (repo's own "
                                    "velocity-Verlet harness, not HOOMD's integrator); 3 launches per step, 2 for rank1_reduce_in_step_one, 1 for one_launch", **md},
        "e2e": {"value": e2e_val(e2e_keep_s), "unit": UNIT, "h2d_bytes_per_step": 32 * N + 32 * n_mol,
                "d2h_bytes_per_step": 32 * N + 32 * n_mol + 192, "steps": e2e_steps,
                "path": f"cavb200_step_host_submit_ex/_wait_ex over {E2E_SLOTS} host-resident systems (next upload under this "
                        "download), pinned host buffers; positions and velocities in, forces and velocities out every step; "
                        "charges and images flagged unchanged since the slot's last submit (uploaded once, before the timed region)",
                "ms_per_step": 1e3 * e2e_keep_s / e2e_steps,
                "rounds_ms_per_step": [1e3 * x / e2e_steps for x in rounds_keep],
                "full_copy": {"value": e2e_val(e2e_full_s), "ms_per_step": 1e3 * e2e_full_s / e2e_steps,
                              "h2d_bytes_per_step": 52 * N + 32 * n_mol, "d2h_bytes_per_step": 32 * N + 32 * n_mol + 192,
                              "path": "every array every step (charge and image too)"},
                "rank1_result": {"value": e2e_val(e2e_rank1_s), "ms_per_step": 1e3 * e2e_rank1_s / e2e_steps,
                                 "h2d_bytes_per_step": 32 * N + 32 * n_mol, "d2h_bytes_per_step": 32 * n_mol + 192,
                                 "path": "as the headline, and the rank-1 result {Dq, F_L, energies} instead of the force array "
                                         "(F_i = -g c_i Dq, formed by the consumer from the charges it holds)"},
                "host_buffers": numa.info,
                "synchronous": {"value": e2e_val(e2e_sync_s), "ms_per_step": 1e3 * e2e_sync_s / e2e_steps,
                                "path": "one blocking cavb200_step_host call per step, one system, every array"},
                "pcie": pcie},
        "gpu_launches": launches_fused, "clocks": clocks,
    }
    if fkt is not None:
        line["fkt"] = fkt
    if sharded is not None:
        line["sharded"] = sharded
    if small is not None:
        line["small_n"] = small
    if world == 1 and not args.no_cpu_baseline:
        cores = min(os.cpu_count() or 1, 32)
        line["cpu_baseline"] = cpu_reference_throughput(n_mol, args.cpu_steps, cores)
    _LINES.append(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-mol", type=int, default=1_000_000)
    ap.add_argument("--systems", type=int, default=8)
    ap.add_argument("--variant", type=int, default=None)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--unroll", type=int, default=0)
    ap.add_argument("--cpu-steps", type=int, default=30)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fkt", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-small-n", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the B200 path (--impl b200)")
    # stdout carries the ONE JSON line and nothing else: native libraries write there too (NCCL prints its version
    # banner to fd 1 when the sharded leg creates its communicator), so fd 1 points at stderr while the run lasts and
    # the line goes to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        return (run_reference if args.impl == "reference" else run_b200)(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
        for text in _LINES:
            print(text)
        sys.stdout.flush()


_LINES = []  # what main() prints on the real stdout


if __name__ == "__main__":
    sys.exit(main())
