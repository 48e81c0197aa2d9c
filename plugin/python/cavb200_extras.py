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


class FieldAutocorrelation:
    """F(k,t) without snapshots, on the schedule of the reference's FieldAutocorrelationTracker.act
    (src/cavitymd/analysis.py:380-414): reference 0 at construction, nothing at timestep 0, then every step a record of F
    against every stored reference, and a new reference once `reference_interval_steps` have passed since the last one
    while fewer than `max_references` are stored.  The density field rho(t) and F are formed on the device by the cavity
    force's C++ object (fktOpen / fktStep / fktRead, include/cavb200.h); act() issues one asynchronous step and returns
    nothing, read() brings back what was recorded since the previous read.

    wavevectors: K x 3, e.g. the reference's hoomd.cavitymd.analysis.generate_fibonacci_sphere(n) * kmag.  cavity_force:
    the attached CavityForce wrapper or its C++ object.  In the fused method's "one_launch" mode the positions are
    complete after every launch (only the velocities lag half a kick), so act() needs no flush() of the method.
    Constructing another tracker on the same force re-opens the device tracker and drops this one's references."""

    def __init__(self, cavity_force, wavevectors, reference_interval_steps=10000, max_references=10, capacity=16384):
        self._cpp_force = cavity_force if hasattr(cavity_force, "fktOpen") else _cpp(cavity_force)
        self.wavevectors = [tuple(float(c) for c in k) for k in wavevectors]
        self.K = len(self.wavevectors)
        self.reference_interval_steps = reference_interval_steps
        self.max_references = max_references
        self.capacity = capacity
        self._cpp_force.fktOpen(self.wavevectors, max_references, capacity)
        self.reference_timesteps = []  # timestep of reference r
        self.last_reference_step = 0
        self._seen = 0
        self._cpp_force.fktStep(0, False, True)
        self.reference_timesteps.append(0)

    def act(self, timestep):
        if timestep == 0:
            return
        add = (len(self.reference_timesteps) < self.max_references
               and timestep - self.last_reference_step >= self.reference_interval_steps)
        self._cpp_force.fktStep(timestep, True, add)
        if add:
            self.reference_timesteps.append(timestep)
            self.last_reference_step = timestep

    def read(self):
        """-> (rows, rho) of the records appended since the previous read (at most `capacity`, the newest): rows are
        (reference number, timestep, lag in steps, F), record by record and reference by reference as act() of the
        reference produces them; rho is float64[n_records, K, 2] ({re, im} of rho(t) per record)."""
        _, total = self._cpp_force.fktRead(0)
        records, total = self._cpp_force.fktRead(min(total - self._seen, self.capacity))
        self._seen = total
        return records_to_rows(records, self.reference_timesteps, self.max_references), \
            records[:, 2 + self.max_references:].reshape(len(records), self.K, 2)


def records_to_rows(records, reference_timesteps, max_references):
    """Rows (reference number, timestep, lag, F) of F(k,t) tracker records (layout: include/cavb200.h)."""
    rows = []
    for rec in records:
        t = int(rec[0])
        for r in range(int(rec[1])):
            rows.append((r, t, t - reference_timesteps[r], float(rec[2 + r])))
    return rows
