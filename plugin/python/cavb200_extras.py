"""hoomd.cavitymd.cavb200_extras -- the B200 build's additions, reached THROUGH the reference's own wrapper objects.

The Python layer of a B200 deployment is the reference's, file for file and unmodified: plugin/CMakeLists.txt installs
src/cavitymd/*.py and src/bussi_reservoir/*.py from a cav-hoomd checkout (CAV_HOOMD_SOURCE_DIR) next to the B200 builds
of _cavitymd / _bussi_reservoir.  hoomd.cavitymd.CavityForce(kvector, couplstr, omegac, phmass) then finds
_cavitymd.CavityForceComputeGPU on a GPU device (reference src/cavitymd/forces.py:103-119) and
hoomd.bussi_reservoir.BussiReservoir(kT, tau) constructs _bussi_reservoir.BussiReservoirThermostat
(reference src/bussi_reservoir/thermostats.py:87-93) exactly as before.

What the B200 classes offer beyond the reference's API is switched on the attached C++ object (`_cpp_obj`), so no wrapper
needs a new constructor argument.  (Needs a HOOMD install; the pybind classes underneath are tested against hoomd_shim
in tests/test_plugin_gpu.py.)"""


def _cpp(obj):
    cpp = getattr(obj, "_cpp_obj", None)
    if cpp is None:
        raise RuntimeError("attach the object to a simulation first (run(0))")
    return cpp


def set_fused_rescale(bussi, on=True):
    """BussiReservoir: KE reduce, alpha, reservoir bookkeeping AND v <- alpha v in one launch; the thermostat then
    reports {1, 1} to HOOMD's integration method (plugin/src/BussiReservoirThermostat.h, "Two modes")."""
    _cpp(bussi).fused_rescale = bool(on)


def set_cooperative_launch(obj, on=True):
    """CavityForce or BussiReservoir: launch the persistent kernels cooperatively (use when the GPU is shared with other
    streams or processes; include/cavb200.h, conventions)."""
    _cpp(obj).cooperative_launch = bool(on)


def fault_count(obj):
    return _cpp(obj).getFaultCount()


def total_dipole(cavity_force):
    """Total molecular dipole of the last step (free with the force's reduction)."""
    return _cpp(cavity_force).getDipole()


def set_photon_bath(simulation, method, filter, kT, gamma):
    """Give the cavity mode (the one particle of type 'L' that `filter` selects) its own Langevin bath inside the fused
    method of make_fused_method ("rank1" or "one_launch" mode): HOOMD's TwoStepLangevin on the photon, in the method's
    own launches.  Use it INSTEAD of hoomd.md.methods.Langevin(filter=photon), which would integrate the photon a second
    time.  kT: a number or a hoomd.variant.Variant; gamma >= 0 (the reference's run: tau = 5 ps, gamma = 1 / tau).  The
    photon must not be in the method's thermostatted group.  method.clearPhotonBath() removes the bath."""
    if isinstance(kT, (int, float)):
        import hoomd
        kT = hoomd.variant.Constant(float(kT))
    method.setPhotonBath(simulation.state._get_group(filter), kT, float(gamma))


def make_fused_method(simulation, filter, bussi, cavity_force, mode="rank1"):
    """The fused integration method (plugin/src/TwoStepConstantVolumeCavity.h) as a C++ object, built from attached
    wrapper objects: thermostat folded into the kicks, cavity force rank-1 ("rank1"), or one launch per MD step
    ("one_launch").  Returns the C++ method; add it to the integrator's C++ object the way HOOMD's
    ConstantVolume._attach_hook does."""
    from . import _cavitymd
    group = simulation.state._get_group(filter)
    return _cavitymd.TwoStepConstantVolumeCavity(simulation.state._cpp_sys_def, group, _cpp(bussi) if bussi is not None else None,
                                                 _cpp(cavity_force), mode)
