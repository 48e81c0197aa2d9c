// TwoStepConstantVolumeCavity.h -- a HOOMD two-step integration method with the Bussi thermostat and the cavity force
// folded into its kernels (SURVEY.md 8f rows 1 and 2).
//
// HOOMD's own TwoStepConstantVolume [upstream, not in the reference tree] does, per step,
//     integrateStepOne:  alpha = thermostat->getRescalingFactorsOne(t, dt) (reference src/Thermostat.h:50-73; for the
//                        Bussi thermostat a full ComputeThermo pass);  v <- alpha v + a dt/2;  r <- r + v dt;  wrap
//     (net force)        every ForceCompute writes its Scalar4 array, the integrator sums them
//     integrateStepTwo:  v <- v + a dt/2
// and is entered from hoomd.md.methods.ConstantVolume(filter, thermostat) (reference examples/05_advanced_run.py:652).
// This class keeps that interface -- IntegrationMethodTwoStep, (sysdef, group, thermostat) plus the cavity force -- and
// issues the library's fused kernels instead:
//   mode "stored"      step one = cavb200_nvt_step_one_wrap (alpha from the kinetic energy the previous step two left on
//                      the device -- no thermo pass), step two = cavb200_nvt_step_two (sums the next KE on the way out)
//   mode "rank1"       the cavity force is never stored: CavityForceComputeGPU only reduces the dipole (its force array
//                      stays zero in HOOMD's net-force sum) and the kicks form F_i = (-g c_i) Dq from the charge
//                      (cavb200_nvt_step_one_rank1_wrap / cavb200_nvt_step_two_rank1)
//   mode "one_launch"  step two of step t is deferred into step one of step t+1: ONE persistent launch per MD step
//                      (cavb200_md_step_fused_wrap: second half kick, KE -> alpha, rescale, first half kick, drift, wrap,
//                      dipole reduce of the new positions).  Between steps the velocities are half a kick behind;
//                      flush() completes them (call it before anything reads velocities, and at the end of a run).
// Thermostatted group: with index_list_group = false (default) it must be a contiguous index range [first, first + n)
// -- e.g. all molecular particles with the photon first or last -- and the kernels take that window.  With
// index_list_group = true any group is accepted: a contiguous list still takes the window, any other list becomes the
// handle's bit mask (cavb200_group_set, CAVB200_GROUP_MASK), rebuilt when HOOMD's particle sorter has reordered the
// particles or the group / particle count changed.  In either case a sort (getParticleSortSignal) also moves the photon
// index of the last rank-1 result (cavb200_rank1_reindex) in the rank1 and one_launch modes, before the next launch.
// Photon bath (setPhotonBath, rank1 and one_launch modes): the cavity mode gets its own Langevin bath, HOOMD's
// TwoStepLangevin on the one particle of type 'L' [HOOMD-upstream: restated], in the same launches (the *_bath entry
// points of include/cavb200.h).  integrateStepTwo draws r with RandomGenerator(Seed(RNGIdentifier::TwoStepLangevin, t,
// seed), Counter(photon tag)) and evaluates kT(t); the photon kicks with f + bd, bd = coeff r - gamma v.  This replaces
// hoomd.md.methods.Langevin(filter=photon) next to the method, which would integrate the photon twice.
// Restrictions (checked, stated in INTEGRATION.md): every particle of the system is integrated by this method; point
// particles only; single rank; with the sorter on, one particle of type 'L' in the rank-1 modes; the photon bath acts on
// a group of exactly that one particle, outside the thermostatted group, not in the stored mode.
#ifndef CAVB200_TWO_STEP_CONSTANT_VOLUME_CAVITY_H
#define CAVB200_TWO_STEP_CONSTANT_VOLUME_CAVITY_H

#include "CavbHooks.h"
#include "CavityForceComputeGPU.h"

#include <hoomd/RNGIdentifiers.h>
#include <hoomd/RandomNumbers.h>
#include <hoomd/Variant.h>
#include <hoomd/md/IntegrationMethodTwoStep.h>
#include <hoomd/md/Thermostat.h>

#include <cavb200.h>
#include <memory>
#include <string>

namespace hoomd::md
    {
class PYBIND11_EXPORT TwoStepConstantVolumeCavity : public IntegrationMethodTwoStep
    {
    public:
    TwoStepConstantVolumeCavity(std::shared_ptr<SystemDefinition> sysdef, std::shared_ptr<ParticleGroup> group,
                                std::shared_ptr<Thermostat> thermostat,
                                std::shared_ptr<cavitymd::CavityForceComputeGPU> cavity, const std::string& mode);
    ~TwoStepConstantVolumeCavity() override;

    void integrateStepOne(uint64_t timestep) override;
    void integrateStepTwo(uint64_t timestep) override;
    //! one_launch mode: the deferred second half kick of the last step (no-op otherwise or when nothing is pending)
    void flush();
    std::string getMode() const;
    unsigned long long getLaunchCount() const { return cavb200_launch_count(m_handle); }
    bool getIndexListGroup() const { return m_index_list; }
    void setIndexListGroup(bool on);
    //! HOOMD's particle sort signal: the mask and the photon index are rebuilt before the next launch
    void slotParticleSort();
    //! the cavity mode's Langevin bath on photon_group (one particle of type 'L', not thermostatted): kT(t), gamma >= 0
    void setPhotonBath(std::shared_ptr<ParticleGroup> photon_group, std::shared_ptr<Variant> kT, Scalar gamma);
    void clearPhotonBath();
    bool hasPhotonBath() const { return (bool)m_bath_group; }

    private:
    void window(unsigned int& first, unsigned int& n);
    void group(unsigned int& first, unsigned int& n);
    void reindexPhoton(uint32_t L_typeid);
    uint32_t photonTypeId() const;
    void check(int err, const char* what) const;
    enum Mode { STORED = 0, RANK1 = 1, ONE_LAUNCH = 2 };
    std::shared_ptr<Thermostat> m_thermostat;
    CavbBussiSource* m_source; //!< the thermostat's hook (nullptr: no thermostat, plain velocity Verlet)
    std::shared_ptr<cavitymd::CavityForceComputeGPU> m_cavity;
    cavb200_handle* m_handle;
    Mode m_mode;
    bool m_started;   //!< the kinetic energy of the initial velocities has been put on the device
    bool m_pending;   //!< one_launch: a second half kick is outstanding
    bool m_index_list;     //!< index_list_group: any group, as a mask when it is not a contiguous range
    bool m_group_stale;    //!< index_list_group: the window / mask must be rebuilt before the next launch
    bool m_use_mask;       //!< index_list_group: the group is the handle's mask (else the window at m_first)
    unsigned int m_first;  //!< index_list_group: first index of a contiguous group
    unsigned int m_group_n, m_group_N; //!< members and particle count the window / mask was built for
    bool m_photon_stale;   //!< particles were sorted since the last rank-1 result was formed
    std::shared_ptr<ParticleGroup> m_bath_group; //!< photon bath: its group (nullptr: no bath)
    std::shared_ptr<Variant> m_bath_kT;
    Scalar m_bath_gamma;
    bool m_bath_primed;    //!< photon bath: a step two with the bath has stored bd in the handle's slot
    bool m_pending_bath;   //!< one_launch: the outstanding second half kick takes m_pending_args
    cavb200_langevin_args m_pending_args;
    cavb200_langevin_args drawBath(uint64_t timestep);
    };

namespace detail
    {
void export_TwoStepConstantVolumeCavity(pybind11::module& m);
    }
    } // namespace hoomd::md
#endif
