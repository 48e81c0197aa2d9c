// CavityForceComputeGPU.h -- B200 host class of the cavity force.
//
// Drop-in for the reference's class of the same name (reference src/CavityForceComputeGPU.h:30-56):
// same constructor (sysdef, omegac, couplstr, phmass = 1), same pybind name, same methods
// (setParams, getParams, getHarmonicEnergy, getCouplingEnergy, getDipoleSelfEnergy), still a
// hoomd::ForceCompute whose computeForces(timestep) HOOMD's integrator calls once per step.
// What changed is everything below that boundary: instead of four GPUArray workspaces, per-step
// memsets, a C++ kernel driver, two blocking D2H copies, a device synchronize and two full-array
// host read-backs (reference src/CavityForceComputeGPU.cc:102-253), computeForces borrows HOOMD's
// device pointers and makes ONE asynchronous call into the C ABI (include/cavb200.h).  Energies stay
// on the device until a getter asks for them.
#ifndef CAVB200_CAVITY_FORCE_COMPUTE_GPU_H
#define CAVB200_CAVITY_FORCE_COMPUTE_GPU_H

#include "hoomd/ForceCompute.h"
#include "hoomd/HOOMDMath.h"

#include <cavb200.h>
#include <memory>
#include <pybind11/pybind11.h>

namespace hoomd
    {
namespace cavitymd
    {
class PYBIND11_EXPORT CavityForceComputeGPU : public ForceCompute
    {
    public:
    CavityForceComputeGPU(std::shared_ptr<SystemDefinition> sysdef, Scalar omegac, Scalar couplstr,
                          Scalar phmass = Scalar(1.0));
    virtual ~CavityForceComputeGPU();

    //! K = phmass * omegac * omegac, as the reference's cavity_force_params constructor forms it
    void setParams(Scalar omegac, Scalar couplstr, Scalar phmass = Scalar(1.0));
    pybind11::dict getParams();
    Scalar getHarmonicEnergy();
    Scalar getCouplingEnergy();
    Scalar getDipoleSelfEnergy();
    //! total molecular dipole of the last step (not in the reference API; free with the reduction)
    pybind11::tuple getDipole();
    //! true: cooperative launches (safe when the GPU is shared with other streams / processes); false (default):
    //! programmatic dependent launches.  The library switches to cooperative by itself after a hand-off timeout.
    bool getCooperativeLaunch() const;
    void setCooperativeLaunch(bool c);
    unsigned long long getFaultCount() const;
    //! CUDA stream the force kernel is issued on, as an integer (cudaStream_t); 0 = the legacy default stream HOOMD's
    //! own kernels run on (the default, and what a HOOMD run uses).  For harnesses that drive several objects at once.
    void setStream(size_t stream) { m_stream = reinterpret_cast<void*>(stream); }
    size_t getStream() const { return reinterpret_cast<size_t>(m_stream); }

    //! Device-side trackers (SURVEY.md 8f.4): what DipoleAutocorrelation / CavityModeTracker / EnergyTracker of the
    //! reference get from a full cpu_local_snapshot every step (src/cavitymd/analysis.py:188,234,535,578,1327) is
    //! appended on the device, one 128-byte record per call, and read back once per output period.
    //! The ring lives on this object's own handle, so attaching or detaching an integration method keeps a run's records.
    //! A record reads the dipole, q, energies and photon index of the handle that computes the force (the method's in the
    //! rank-1 modes) and [12..14] of the handle that ran the thermostat (the method's; NaN with no method attached, since
    //! this object cannot know a thermostat of its own).  While the method's one_launch mode holds a second half kick
    //! back, [11] and [12] are NaN: they need the velocities of the full step (flush() first).
    void trackOpen(unsigned int capacity);
    void trackSetReference();
    void trackRecord(uint64_t timestep);
    //! newest min(max_records, stored) records, oldest first: list of 16-tuples (layout: include/cavb200.h)
    pybind11::list trackRead(unsigned int max_records);

    //! F(k,t) without snapshots: what FieldAutocorrelationTracker.act of the reference gets from a cpu_local_snapshot and
    //! K NumPy passes every step (src/cavitymd/analysis.py:260-418) is formed on the device on this object's handle and
    //! stream, one record per step {timestep, n_refs, F per reference, rho(t)} (layout: include/cavb200.h).
    //! kvectors: K rows of 3 numbers.  fktOpen blocks and drops every stored reference; fktStep is asynchronous and reads
    //! the current positions; fktRead returns (records float64[n, 2 + max_references + 2K] oldest first, total appended).
    void fktOpen(pybind11::object kvectors, unsigned int max_references, unsigned int capacity);
    void fktStep(uint64_t timestep, bool record, bool add_reference);
    pybind11::tuple fktRead(unsigned int max_records);

    //! Used by TwoStepConstantVolumeCavity (SURVEY.md 8f.1/8f.2).  mode 0: back to normal (own handle, forces stored).
    //! mode 1: rank-1 -- the dipole reduce runs on the integration method's handle `h` and NOTHING is written per
    //! particle: m_force stays zero, the method's kicks form F_i = (-g c_i) Dq from the charge
    //! (reference src/CavityForceCompute.cc:183,188-200).  mode 2: as 1, and the method's own step-one kernel reduces the
    //! dipole of the new positions, so computeForces only runs the reduce until the method has taken over.
    void useHandle(cavb200_handle* h, int mode);
    void integratorHasReduced() { m_integrator_reduced = true; m_fresh = false; }
    //! Used by TwoStepConstantVolumeCavity in every mode: the handle whose step kernels publish KE / alpha / reservoir
    //! (nullptr: none), and whether the velocities are half a kick short of the step (one_launch between flushes).
    void useThermostatHandle(cavb200_handle* h) { m_bussi_handle = h; }
    cavb200_handle* thermostatHandle() const { return m_bussi_handle; }
    void setVelocitiesPending(bool pending) { m_vel_pending = pending; }
    const cavb200_params& params() const { return m_params; }

    protected:
    virtual void computeForces(uint64_t timestep);

    private:
    void readBack();
    cavb200_handle* m_handle;
    cavb200_params m_params;
    double m_energies[3];
    double m_dipole[3];
    bool m_fresh; //!< host copies are current
    void* m_stream = nullptr;
    cavb200_handle* m_ext_handle = nullptr; //!< the integration method's handle (rank-1 modes), not owned
    cavb200_handle* m_bussi_handle = nullptr; //!< the handle the thermostat runs on (the method's), not owned
    bool m_vel_pending = false;             //!< one_launch: the velocities lack the deferred second half kick
    int m_mode = 0;
    bool m_integrator_reduced = false;
    bool m_zeroed = false;
    unsigned int m_fkt_words = 0; //!< doubles per F(k,t) record (0: fktOpen not called)
    };

namespace detail
    {
void export_CavityForceComputeGPU(pybind11::module& m);
    }
    } // namespace cavitymd
    } // namespace hoomd
#endif
