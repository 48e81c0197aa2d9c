"""Argument checks of the sixteen C entry points of the velocity-Verlet harness (csrc/nve.cu), table-driven: a valid call
returns 0 and launches one kernel; each single bad argument returns its cudaError_t and launches nothing; N == 0 returns
0 and launches nothing wherever that rule applies (everywhere but cavb200_group_set, whose N sizes the mask)."""
import ctypes as C

import numpy as np
import pytest

from cav_hoomd_b200 import capi, synth

pytestmark = pytest.mark.gpu
INVALID_VALUE, MISALIGNED = 1, 716  # cudaError_t
ALIGN = {"pos": 32, "vel": 32, "force": 32, "force_other": 32, "net_force": 32, "charge": 8, "image": 4, "group_idx": 4}
MD = "pos vel force_other charge image N dt Lx Ly Lz L_typeid params group_first n_group bussi stream"
MD_REQ = "pos vel charge image params"
# entry point, its arguments after the handle, the pointers that may not be NULL
ENTRIES = [
    ("cavb200_nve_kick_drift", "pos vel force N dt stream", "pos vel force"),
    ("cavb200_nve_kick_drift_wrap", "pos vel force image N dt Lx Ly Lz stream", "pos vel force image"),
    ("cavb200_nve_half_kick", "vel force N dt stream", "vel force"),
    ("cavb200_nvt_step_one", "pos vel force N dt group_first n_group bussi stream", "pos vel force"),
    ("cavb200_nvt_step_one_wrap", "pos vel force image N dt Lx Ly Lz group_first n_group bussi stream",
     "pos vel force image"),
    ("cavb200_nvt_step_two", "vel force N dt group_first n_group stream", "vel force"),
    ("cavb200_nvt_step_one_rank1", "pos vel force_other charge N dt L_typeid couplstr group_first n_group bussi stream",
     "pos vel charge"),
    ("cavb200_nvt_step_one_rank1_wrap",
     "pos vel force_other charge image N dt Lx Ly Lz L_typeid couplstr group_first n_group bussi stream",
     "pos vel charge image"),
    ("cavb200_nvt_step_two_rank1", "vel force_other charge pos N dt L_typeid couplstr group_first n_group stream",
     "vel charge pos"),
    ("cavb200_md_step_one", MD, MD_REQ),
    ("cavb200_md_step_one_wrap", MD, MD_REQ),
    ("cavb200_md_step_fused", MD, MD_REQ),
    ("cavb200_md_step_fused_wrap", MD, MD_REQ),
    ("cavb200_net_force_add_rank1", "net_force charge pos N L_typeid couplstr stream", "net_force charge pos"),
    ("cavb200_group_set", "group_idx n N stream", "group_idx"),
    ("cavb200_rank1_reindex", "pos N L_typeid stream", "pos"),
]


def bad_arguments(name, args, required, N, n_group):
    """(what, {argument: value}, expected code) for every single bad argument of one entry point."""
    args = args.split()
    yield "handle NULL", {"h": None}, INVALID_VALUE
    for k in required.split():
        yield f"{k} NULL", {k: None}, INVALID_VALUE
    for k in args:
        if k in ALIGN:  # 8 bytes off a 32-byte alignment, half of a smaller one
            yield f"{k} misaligned", {k: ("+", 8 if ALIGN[k] == 32 else ALIGN[k] // 2)}, MISALIGNED
    if "group_first" in args:
        yield "window past N", {"group_first": 1, "n_group": N}, INVALID_VALUE
        yield "mask of another n_group", {"group_first": capi.Handle.GROUP_MASK, "n_group": n_group + 1}, INVALID_VALUE
        yield "mask of another N", {"group_first": capi.Handle.GROUP_MASK, "N": N - 1}, INVALID_VALUE
    if name.endswith("_wrap"):
        for k in ("Lx", "Ly", "Lz"):
            yield f"{k} = 0", {k: 0.0}, INVALID_VALUE
            yield f"{k} < 0", {k: -1.0}, INVALID_VALUE


@pytest.mark.parametrize("name,args,required", ENTRIES, ids=[e[0] for e in ENTRIES])
def test_harness_entry_point_arguments(name, args, required):
    s = synth.make_system(999, photon="middle")
    N = s.N
    h = capi.Handle(0)
    p = capi.Params.make(0.01, 1e-3)
    dof = 3.0 * (N - 1) - 3.0
    b = capi.BussiArgs(synth.KT_100K, synth.TAU_5PS, synth.DT_1FS, dof, 0.3, (dof - 1) / 2)
    mol = np.flatnonzero(s.typeid != s.L_typeid).astype(np.uint32)
    d = {k: capi.DeviceArray.from_numpy(getattr(s, k)) for k in ("pos", "vel", "charge", "image")}
    d["force"] = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    d["force_other"] = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    d["net_force"] = capi.DeviceArray.from_numpy(np.zeros((N, 4)))
    d["group_idx"] = capi.DeviceArray.from_numpy(mol)
    h.force_rank1(d["pos"], d["charge"], d["image"], N, s.box, s.L_typeid, p)
    h.group_set(d["group_idx"], len(mol), N)  # the mask of the GROUP_MASK calls: the molecules
    h.bussi_ke(d["vel"], None, 0, N, None)
    env = {k: v.ptr for k, v in d.items()}
    env.update(h=h.h, N=N, n=len(mol), dt=synth.DT_1FS, Lx=s.box[0], Ly=s.box[1], Lz=s.box[2],
               L_typeid=s.L_typeid & 0xFFFFFFFF, couplstr=1e-3, params=C.byref(p), group_first=0, n_group=N,
               bussi=C.byref(b), stream=None)
    fn = getattr(capi.load(), name)

    def call(**over):
        vals = {k: (env[k] + v[1] if isinstance(v, tuple) else v) for k, v in over.items()}
        before = h.launch_count
        rc = fn(*[vals.get(k, env[k]) for k in ["h"] + args.split()])
        return rc, h.launch_count - before

    assert call() == (0, 1)
    if "group_first" in args:
        assert call(group_first=capi.Handle.GROUP_MASK, n_group=len(mol)) == (0, 1)
    for what, over, code in bad_arguments(name, args, required, N, len(mol)):
        assert call(**over) == (code, 0), what
    if name != "cavb200_group_set":
        assert call(N=0) == (0, 0)
    capi.sync()
    assert h.fault_count == 0
    h.close()
