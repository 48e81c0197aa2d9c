/*
 * cavb200.h -- C ABI of libcavb200.so, the B200 (sm_100a) implementation of cav-hoomd's
 * data-parallel hot path: the cavity force, the BussiReservoir kinetic-energy reduce + velocity
 * rescale, and the F(k,t) density-field sum.
 *
 * This is the drop-in boundary.  The reference's plugin layer calls ONE C++ driver,
 *     hipError_t hoomd::cavitymd::kernel::gpu_compute_cavity_force(Scalar4* d_force,
 *         const Scalar4* d_pos, const Scalar* d_charge, const int3* d_image, const BoxDim* box,
 *         unsigned N, const cavity_force_params&, Scalar* d_temp_energy, int* d_photon_idx,
 *         Scalar3* d_temp_dipole, Scalar3* d_dipole_global, unsigned L_typeid, unsigned& block_size)
 *     (reference src/CavityForceComputeGPU.cuh:28-40, called from src/CavityForceComputeGPU.cc:172-184)
 * and gets the kinetic energy / velocity rescale from HOOMD itself
 *     (reference src/BussiReservoirThermostat.h:50-55 and :78-98).
 * Each entry point below names the reference interface it replaces.  plugin/ holds the
 * pybind11/HOOMD host classes that bind to this header; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - plain C types only.  Particle arrays use HOOMD's device layouts and are BORROWED for the
 *     duration of the call (the library never frees or retains them):
 *         pos    double[4*N]  x,y,z,w   w = type id in the LOW 32 bits   (Scalar4, 32-byte aligned)
 *         vel    double[4*N]  vx,vy,vz,mass                              (Scalar4, 32-byte aligned)
 *         force  double[4*N]  fx,fy,fz,pe                                (Scalar4, 32-byte aligned)
 *         charge double[N]                                               (8-byte aligned)
 *         image  int32[3*N]                                              (int3, 4-byte aligned)
 *   - every compute call is ASYNCHRONOUS on `stream` (a cudaStream_t passed as void*; NULL is the
 *     legacy default stream HOOMD runs on) and never synchronises the host.  Scalars (energies,
 *     dipole, KE, alpha) stay on the device until a *_read call copies them back.
 *   - return value: a cudaError_t as int (0 = success).  NULL array arguments with N > 0 return
 *     cudaErrorInvalidValue (1), like the reference driver (CavityForceComputeGPU.cu:522-528);
 *     N == 0 is a successful no-op (:530-532).  There is no CPU fallback anywhere: without a
 *     CUDA device cavb200_create fails.
 *   - a handle owns its workspace and is bound to one device; calls on one handle must be issued
 *     from one host thread at a time (HOOMD's integrator thread).
 *   - the force / Bussi / step / md_step_fused / shard kernels are PERSISTENT: their grids fill the device and the CTAs
 *     hand results to each other while resident.  By default they are launched with programmatic stream serialization
 *     (the next call's CTAs start while this call drains), which relies on the stream having the device to itself --
 *     one stream, as HOOMD does, or streams ordered by events (what cavb200_step_host_submit does internally).  If
 *     something else holds SM slots (another stream, another process under MPS) and a grid is not co-resident, the
 *     hand-off gives up after 50 ms: nothing hangs, that call's outputs are NOT written, the kernel raises a fault word
 *     in pinned host memory, and the NEXT compute call on the handle returns cudaErrorLaunchTimeout once (the plugin
 *     classes throw) and switches the handle to cooperative launches for good -- the driver then guarantees
 *     co-residency, at ~2 us per launch.  cavb200_set_tuning(h, "pdl", 0) selects cooperative launches from the start
 *     (use it when the GPU is shared).  The *_read calls of the failed call also return cudaErrorLaunchTimeout /
 *     err = 2; the status words are rewritten by every call, so one failure does not stick.
 */
#ifndef CAVB200_H
#define CAVB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAVB200_VERSION 100

typedef struct cavb200_handle cavb200_handle;

/* Mirrors struct cavity_force_params {omegac, couplstr, K, phmass}
 * (reference src/CavityForceCompute.h:28-54).  K = phmass*omegac*omegac is filled by the caller
 * exactly as the reference constructor does (:38-42). */
typedef struct
    {
    double omegac;
    double couplstr;
    double K;
    double phmass;
    } cavb200_params;

/* Everything compute_rescale_factor needs that does NOT depend on the kinetic energy
 * (reference src/BussiReservoirThermostat.h:177-225): the two random draws are made by the host
 * class (HOOMD's RandomGenerator in a real build) BEFORE the launch, so the factor can be formed
 * on the device right after the reduction with no host round trip.
 *   r_normal   = normal(rng)                        (:192-193)
 *   gamma_draw = gamma((dof-1)/2, 1)(rng) if dof>1  (:195-200; the library doubles it like :199) */
typedef struct
    {
    double kT;         /* set_T, the temperature set point at this timestep (:69) */
    double tau;        /* thermostat time constant; 0 = instantaneous (:186-190) */
    double deltaT;     /* step size; 0 makes the call a no-op with alpha = 1 (:45-48) */
    double dof;        /* translational degrees of freedom of the group (:52) */
    double r_normal;
    double gamma_draw;
    } cavb200_bussi_args;

/* ---- lifetime ------------------------------------------------------------------------------ */

int cavb200_version(void);
/* Binds to `device` (cudaSetDevice) and allocates the workspace.  Replaces the GPUArray members
 * m_temp_energy / m_temp_dipole / m_photon_idx / m_dipole_global of the reference host class
 * (src/CavityForceComputeGPU.h:50-53, .cc:43-54). */
int cavb200_create(cavb200_handle** out, int device);
int cavb200_destroy(cavb200_handle* h);
const char* cavb200_error_string(int err);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
uint64_t cavb200_launch_count(const cavb200_handle* h);
/* Number of hand-off timeouts this handle has seen (see the conventions above); 0 in a healthy run. */
uint64_t cavb200_fault_count(const cavb200_handle* h);
/* Debug: with tuning "stamps" = 1 the cooperative kernel records, per CTA, globaltimer ns at
 * {start, after reduce, after barrier, after combine, after apply}; out = uint64[8*n_ctas]. */
int cavb200_debug_stamps(cavb200_handle* h, uint64_t* out, uint32_t n_ctas);
/* Measurement helpers (bench.py, tools/; never on the product path):
 *   cavb200_debug_delay        a one-thread kernel that holds `stream` for `ns` nanoseconds (<= 100 ms), so that a timed
 *                              region can be enqueued completely before its first kernel starts
 *   cavb200_debug_fp64_peak    DFMA microbenchmark on the handle's device: FP64 fused multiply-adds per second over all
 *                              SMs (the roofline denominator of the F(k,t) kernel); synchronous, ~50 ms
 *   cavb200_debug_launch_ring  with tuning "stamps" = 2 the persistent kernels record, per launch, {first CTA start,
 *                              last CTA end} in globaltimer ns into a ring of 2048 pairs indexed by the launch's epoch;
 *                              out = uint64[2*n_pairs] (may be NULL), *epoch = epoch of the last launch; reset != 0
 *                              re-arms the ring.  Synchronises the device. */
int cavb200_debug_delay(cavb200_handle* h, uint64_t ns, void* stream);
int cavb200_debug_fp64_peak(cavb200_handle* h, double* dfma_per_s);
int cavb200_debug_launch_ring(cavb200_handle* h, int reset, uint64_t* out, uint32_t n_pairs, uint64_t* epoch);
/* Tuning knobs ("variant", "threads", "ctas_per_sm", "unroll", "pdl", "stamps", ...); unknown key -> 1.
 * By size: calls over at most "small_n" particles (768) run as one CTA; calls that include the force, over at most
 * "cluster_n" particles (8192), as one thread-block cluster of "cluster_ctas" CTAs (16; 8 and half the size if the device
 * refuses the non-portable cluster size); everything else as persistent grids.  0 switches either off. */
int cavb200_set_tuning(cavb200_handle* h, const char* key, int value);
int cavb200_get_tuning(const cavb200_handle* h, const char* key, int* value);

/* ---- cavity force ---------------------------------------------------------------------------
 * Replaces gpu_compute_cavity_force + the per-step memsets and D2H copies of
 * CavityForceComputeGPU::computeForces (src/CavityForceComputeGPU.cc:102-253), with the
 * SEMANTICS of the CPU class CavityForceCompute::computeForces (src/CavityForceCompute.cc:134-208),
 * which is the parity oracle:
 *   photon = first index whose type id == L_typeid; none -> all forces and energies zero;
 *   d = sum_{i != photon} charge_i * (pos_i + image_i * L);   Dq = q_xy + (g/K) d_xy;
 *   type != L:  force = {(-g*charge)*Dq.x, (-g*charge)*Dq.y, 0, 0};   other 'L': zero;
 *   photon:     force = {-K q.x - g d.x, -K q.y - g d.y, -K q.z, 0};
 *   energies {1/2 K q.q, g d_xy.q_xy, 1/2 g^2/K d_xy.d_xy} kept on the device.
 * Every force[i] (all four components) is overwritten; virial is not touched (the reference never
 * writes it).  L_typeid = UINT32_MAX means "no type named 'L'" (zero forces, zero energies). */
int cavb200_force(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image,
                  double* force, uint32_t N, double Lx, double Ly, double Lz, uint32_t L_typeid,
                  const cavb200_params* params, void* stream);

/* Lazy getters: one small D2H copy + stream sync when called, nothing per step.
 * Replace getHarmonicEnergy/getCouplingEnergy/getDipoleSelfEnergy (src/CavityForceCompute.cc:58-71). */
int cavb200_force_read(cavb200_handle* h, double energies[3], double dipole[3], int32_t* photon_idx,
                       void* stream);

/* ---- Bussi reservoir thermostat ---------------------------------------------------------------
 * KE = 1/2 sum_group m |v|^2 (HOOMD ComputeThermo, consumed at BussiReservoirThermostat.h:50-55),
 * alpha = compute_rescale_factor(KE, dof, dt, kT, draws) (:177-225), reservoir bookkeeping
 * delta = KE (1 - alpha^2), cumulative += delta (:86-95) and v <- alpha v, in ONE launch.
 * group_idx == NULL means the contiguous group [group_first, group_first + n).
 * KE == 0 with dof != 0 sets the error flag read back by cavb200_bussi_read (the reference throws
 * "Bussi thermostat requires non-zero initial momenta", :57-61) and leaves velocities untouched. */
int cavb200_bussi(cavb200_handle* h, double* vel, const uint32_t* group_idx, uint32_t group_first,
                  uint32_t n, const cavb200_bussi_args* args, void* stream);
/* KE reduction only (what getRescalingFactorsOne needs when HOOMD itself applies the rescale). */
int cavb200_bussi_ke(cavb200_handle* h, const double* vel, const uint32_t* group_idx,
                     uint32_t group_first, uint32_t n, void* stream);
/* out = {KE before, alpha, instantaneous reservoir, cumulative reservoir, error flag}. */
int cavb200_bussi_read(cavb200_handle* h, double out[5], void* stream);
/* resetReservoirEnergy (src/BussiReservoirThermostat.h:153-159). */
int cavb200_bussi_reset(cavb200_handle* h, void* stream);

/* ---- fused step: cavity force + Bussi in one launch --------------------------------------------
 * The north-star "each particle makes one HBM round trip per step": one persistent kernel reduces
 * the dipole and the kinetic energy together, crosses one grid barrier, then writes forces and
 * rescaled velocities.  Same results as cavb200_force followed by cavb200_bussi.
 * The Bussi group is the contiguous range [group_first, group_first + n_group). */
int cavb200_step(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image,
                 double* force, double* vel, uint32_t N, double Lx, double Ly, double Lz,
                 uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                 uint32_t n_group, const cavb200_bussi_args* bussi, void* stream);

/* ---- minimal NVE harness (velocity Verlet around the cavity force) ------------------------------
 * Not a reference function: the step harness the 10k-step energy-drift comparison of
 * BASELINE.json runs on both arms (oracle: orc_nve_step).  Masses are vel.w; positions are NOT
 * wrapped and images are not touched.
 *   kick_drift:  v += (dt/2) f/m;  r += dt v        half_kick:  v += (dt/2) f/m
 *   kinetic:     writes sum 1/2 m |v|^2 over all N particles to the Bussi KE slot (cavb200_bussi_read) */
int cavb200_nve_kick_drift(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                           void* stream);
int cavb200_nve_half_kick(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt, void* stream);

/* Thermostatted harness step (SURVEY.md 8f.1; not a reference function, not HOOMD's integrator):
 * the Bussi rescale rides on the first half step and the kinetic energy for the NEXT step is taken
 * while the second half step writes the velocities, so the thermostat costs no pass of its own.
 *   step_one:  alpha = compute_rescale_factor(KE, draws) (reference src/BussiReservoirThermostat.h:177-225)
 *              from the KE the previous step_two (or cavb200_bussi_ke) left on the device, reservoir
 *              bookkeeping (:86-95);  group [group_first, +n_group): v <- alpha v;
 *              all N: v += (dt/2) f/m;  r += dt v.      bussi == NULL: alpha = 1 (plain NVE).
 *   step_two:  all N: v += (dt/2) f/m;  KE = 1/2 sum_group m|v|^2 -> device (cavb200_bussi_read()[0]).
 * A step is  step_one ; cavb200_force ; step_two.  Call cavb200_bussi_ke once before the first step. */
int cavb200_nvt_step_one(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                         uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream);
int cavb200_nvt_step_two(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt,
                         uint32_t group_first, uint32_t n_group, void* stream);

/* The same steps with the BOX WRAP of the drift (SURVEY.md 8a row a11: r <- r + v dt, then wrap): after the drift a
 * coordinate at or above L/2 moves down by L and its image flag goes up by one, a coordinate below -L/2 the other way
 * (HOOMD's BoxDim::wrap for an orthorhombic, fully periodic box; upstream code restated from its definition, oracle
 * orc_wrap).  `image` (int32[3*N]) is read and, for particles that cross a face, written.  The unwrapped position
 * pos + image * L that the dipole uses (reference src/CavityForceCompute.cc:107-109) is unchanged by the wrap up to one
 * rounding.  plugin/src/TwoStepConstantVolumeCavity binds these to HOOMD's integrateStepOne / integrateStepTwo. */
int cavb200_nve_kick_drift_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image, uint32_t N,
                                double dt, double Lx, double Ly, double Lz, void* stream);
int cavb200_nvt_step_one_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image, uint32_t N,
                              double dt, double Lx, double Ly, double Lz, uint32_t group_first, uint32_t n_group,
                              const cavb200_bussi_args* bussi, void* stream);

/* ---- rank-1 cavity force (SURVEY.md 8f.2) -------------------------------------------------------
 * Every molecular particle's cavity force is the same 2-vector times its charge,
 *     F_i = (-couplstr * charge_i) * Dq,   Dq = q_xy + (g/K) d_xy
 * (reference src/CavityForceCompute.cc:183,188-200), so it need not be stored at all:
 *   cavb200_force_rank1      cavb200_force without the force array: dipole reduce (52 B/particle read,
 *                            nothing written per particle); energies / dipole / photon index as
 *                            cavb200_force_read; Dq, F_L stay on the device for the consumers below.
 *   cavb200_rank1_read       Dq[2], F_L[3] (photon force, :203-207), photon index, number of 'L' particles
 *                            (a schedule that merges per-CTA records reports any number above one as 2).
 *   cavb200_net_force_add_rank1   net_force[i] += F_i formed from charge_i: what HOOMD's net-force sum
 *                            (Integrator::computeNetForceGPU, upstream) would do with this contribution.
 *                            The photon gets F_L; further 'L' particles get 0 (pos is only read, for the
 *                            type, when more than one 'L' particle exists).
 *   cavb200_nvt_step_one_rank1 / _two_rank1   the harness steps above with the cavity force formed in the
 *                            kick: f = force_other (NULL = none) + F_i.  Bit-identical to the stored-force
 *                            steps when force_other == NULL.
 * All consumers use the result of the LAST cavb200_force_rank1 on this handle. */
int cavb200_force_rank1(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image, uint32_t N,
                        double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params, void* stream);
int cavb200_rank1_read(cavb200_handle* h, double Dq[2], double F_L[3], int32_t* photon_idx, uint32_t* n_L, void* stream);
int cavb200_net_force_add_rank1(cavb200_handle* h, double* net_force, const double* charge, const double* pos,
                                uint32_t N, uint32_t L_typeid, double couplstr, void* stream);
int cavb200_nvt_step_one_rank1(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                               const double* charge, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                               uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream);
/*   cavb200_md_step_one      step one of the harness with the NEXT cavity force's reduce pass inside it: the kick uses
 *                            the rank-1 force of the previous result, the drift produces r_new, and the dipole term
 *                            charge * (r_new + image L) (reference src/CavityForceCompute.cc:107-109,124) is accumulated
 *                            on the spot, so the positions are not read a second time.  Replaces
 *                            cavb200_nvt_step_one_rank1 + cavb200_force_rank1 by ONE launch; a step is
 *                            cavb200_md_step_one ; cavb200_nvt_step_two_rank1  (220 algorithmic B/particle).
 *                            Energies / dipole / photon index afterwards as cavb200_force_read. */
int cavb200_md_step_one(cavb200_handle* h, double* pos, double* vel, const double* force_other, const double* charge,
                        const int32_t* image, uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t L_typeid,
                        const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                        const cavb200_bussi_args* bussi, void* stream);
/*   cavb200_md_step_fused    ONE launch per MD step: cavb200_nvt_step_two_rank1 of the previous step followed by
 *                            cavb200_md_step_one of this step (second half kick, KE, alpha, rescale, first half kick,
 *                            drift, dipole reduce of the new positions), every array moved once: 148 B/particle.
 *                            A run is  cavb200_force_rank1 ; cavb200_bussi_ke ; cavb200_md_step_one ;
 *                            cavb200_md_step_fused x (T-1) ; cavb200_nvt_step_two_rank1.
 *                            `bussi` holds the draws of the step whose first half it performs. */
int cavb200_md_step_fused(cavb200_handle* h, double* pos, double* vel, const double* force_other, const double* charge,
                          const int32_t* image, uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t L_typeid,
                          const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                          const cavb200_bussi_args* bussi, void* stream);
int cavb200_nvt_step_two_rank1(cavb200_handle* h, double* vel, const double* force_other, const double* charge,
                               const double* pos, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                               uint32_t group_first, uint32_t n_group, void* stream);
/* ... and with the box wrap + image update after the drift (see cavb200_nvt_step_one_wrap): */
int cavb200_nvt_step_one_rank1_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                    const double* charge, int32_t* image, uint32_t N, double dt, double Lx, double Ly,
                                    double Lz, uint32_t L_typeid, double couplstr, uint32_t group_first, uint32_t n_group,
                                    const cavb200_bussi_args* bussi, void* stream);
int cavb200_md_step_one_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other, const double* charge,
                             int32_t* image, uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t L_typeid,
                             const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                             const cavb200_bussi_args* bussi, void* stream);
int cavb200_md_step_fused_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other, const double* charge,
                               int32_t* image, uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t L_typeid,
                               const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                               const cavb200_bussi_args* bussi, void* stream);

/* ---- index-list groups and particle sorts -------------------------------------------------------
 * HOOMD hands a group out as an index list, and its particle sorter permutes the particle arrays.
 *   cavb200_group_set      builds the handle's group mask (one bit per particle, ceil(N/32) words) from the device
 *                          index list group_idx[n] of a system of N particles.  Blocking: returns
 *                          cudaErrorInvalidValue for an index >= N or an index listed twice (no mask is then set).
 *                          Call it once per change of the list, not per step.
 *   CAVB200_GROUP_MASK     passed as `group_first` to cavb200_nvt_step_one(_wrap), _two, _one_rank1(_wrap),
 *                          _two_rank1, cavb200_md_step_one(_wrap) and cavb200_md_step_fused(_wrap): the thermostatted
 *                          group is that mask.  `n_group` and `N` must be the n and N of the last cavb200_group_set,
 *                          else (or without one) the call returns cudaErrorInvalidValue.  A mask that holds the range
 *                          [first, first + n) gives bit-identical results to group_first = first.
 *   cavb200_rank1_reindex  after a permutation of the particle arrays: finds the particle of type L_typeid (low 32 bits
 *                          of pos.w) again and moves the photon index of the last rank-1 result there, so that the
 *                          next rank-1 kick gives F_L to the photon.  Dq, F_L and the energies do not depend on the
 *                          order.  Blocking; cudaErrorNotSupported when more than one particle has that type. */
#define CAVB200_GROUP_MASK 0xFFFFFFFFu
int cavb200_group_set(cavb200_handle* h, const uint32_t* group_idx, uint32_t n, uint32_t N, void* stream);
int cavb200_rank1_reindex(cavb200_handle* h, const double* pos, uint32_t N, uint32_t L_typeid, void* stream);

/* ---- device-side trackers (SURVEY.md 8f.4) ------------------------------------------------------
 * Replace the per-step cpu_local_snapshot of the reference's trackers (reference
 * src/cavitymd/analysis.py:188,234 AutocorrelationTracker / DipoleAutocorrelation, :1327
 * CavityModeTracker, :535,578 EnergyTracker) by a 128-byte record per step, appended on the device from
 * the results the last cavb200_force* / cavb200_bussi* / nvt step left there; the host reads the ring
 * once per output period.  Record layout (CAVB200_TRACK_WORDS doubles):
 *   [0] timestep   [1..3] total dipole d = sum_i q_i r~_i (compute_total_dipole_moment, :18-31; the photon
 *   is excluded, which is the same number whenever its charge is 0, examples/05_advanced_run.py:502)
 *   [4..6] photon coordinate q (unwrapped)   [7..9] harmonic, coupling, dipole-self energy
 *   [10] C(t) = d(ref) . d(t) (:222-224)   [11] cavity-mode kinetic energy 1/2 m|v|^2 of the photon (:1352-1354;
 *   0 if vel == NULL or there is no photon)   [12] group kinetic energy   [13] alpha   [14] cumulative
 *   reservoir energy   [15] photon index (-1: none; the cavity force then computes nothing, reference
 *   src/CavityForceCompute.cc:149-156, and [1..11] are 0).
 *   cavb200_track_open(capacity)   allocate / reset the ring (oldest records are overwritten when full)
 *   cavb200_track_set_reference    d(ref) <- current dipole (_initialize_reference / _start_new_reference)
 *   cavb200_track_record           append one record; asynchronous, stream-ordered after the step's kernels
 *   cavb200_track_read             newest min(max_records, stored) records, oldest first; *total = records
 *                                  appended since open.  Synchronises the stream. */
#define CAVB200_TRACK_WORDS 16
int cavb200_track_open(cavb200_handle* h, uint32_t capacity);
int cavb200_track_set_reference(cavb200_handle* h, void* stream);
int cavb200_track_record(cavb200_handle* h, uint64_t timestep, const double* vel, uint32_t N, void* stream);
int cavb200_track_read(cavb200_handle* h, double* out, uint32_t max_records, uint32_t* n_out, uint64_t* total,
                       void* stream);

/* ---- F(k,t): density field --------------------------------------------------------------------
 * rho[t][k] = sum_j exp(i kvec[k] . r_j(t)) over ALL N particles of frame t (wrapped positions),
 * the batched form of compute_density_field (reference src/cavitymd/analysis.py:34-47).
 * pos: T frames of N particles, `stride` doubles per particle (3 = xyz, 4 = HOOMD Scalar4),
 * frame t starts at pos + t*frame_stride doubles.  kvec: double[3*K] (device).
 * rho: double[2*K*T] (device), interleaved {re, im}.  Deterministic (fixed-order) reduction.
 * Each term exp(i x) is accurate to 2.4e-16 absolute per component (about 1 ulp of 1) for |x| < 2^20;
 * larger arguments, inf and nan go through the CUDA library's sincos.  The first call on a handle
 * uploads an 8 KB table with a blocking copy (like a workspace growth), so make it outside a capture. */
int cavb200_rhok(cavb200_handle* h, const double* pos, uint32_t stride, uint64_t frame_stride,
                 uint32_t N, uint32_t T, const double* kvec, uint32_t K, double* rho, void* stream);
/* The same for float32 xyz positions, the way a GSD trajectory stores them (particles/position, Nx3 float32;
 * reference examples/05_advanced_run.py:1231-1246 writes the trajectory the analysis reads): 12 B/particle/frame
 * instead of 24-32 cross PCIe and HBM; the values are widened exactly, as NumPy does in np.dot(float32, float64)
 * (analysis.py:42).  frame t starts at pos_xyz + t*frame_stride FLOATS. */
int cavb200_rhok_f32(cavb200_handle* h, const float* pos_xyz, uint64_t frame_stride, uint32_t N, uint32_t T,
                     const double* kvec, uint32_t K, double* rho, void* stream);
/* F[o][l] = mean_k Re(rho[o][k] * conj(rho[o+l][k])) for origins o < n_origins, lags l < n_lags
 * with o + l < T (compute_field_autocorr, analysis.py:359-364).  out: double[n_origins*n_lags],
 * entries with o + l >= T are set to NaN. */
int cavb200_fkt(cavb200_handle* h, const double* rho, uint32_t T, uint32_t K, uint32_t n_origins,
                uint32_t n_lags, double* out, void* stream);

/* ---- particle-sharded multi-GPU (one process per GPU) -------------------------------------------
 * New functionality (the reference never reduces across ranks, SURVEY.md 2.3): each rank holds a
 * contiguous block of particles; between the reduce pass and the apply pass the ranks combine
 * {d (compensated pairs), first-photon index and position, KE} in rank-ascending order.
 *   mode 0: ncclAllGather of the 160-byte per-rank record (libnccl resolved with dlopen)
 *   mode 1: one-shot NVLink exchange -- the reduce kernel's last block stores the record into
 *           every peer's mailbox (CUDA IPC peer memory) and the apply kernel spins on its own. */
#define CAVB200_SHARD_RECORD_BYTES 160
#define CAVB200_NCCL_UNIQUE_ID_BYTES 128
int cavb200_shard_nccl_unique_id(void* out128);
int cavb200_shard_init_nccl(cavb200_handle* h, const void* unique_id128, int rank, int nranks);
/* IPC mailbox: every rank exports its mailbox handle (64 bytes), gathers all ranks' handles by
 * any host-side means (bench.py uses torch.distributed) and opens them. */
int cavb200_shard_mailbox_export(cavb200_handle* h, void* out64);
int cavb200_shard_mailbox_open(cavb200_handle* h, const void* handles64_x_nranks, int rank, int nranks);
int cavb200_shard_set_mode(cavb200_handle* h, int mode);
/* `index_offset` = global index of this rank's first particle (photon index is global). */
int cavb200_shard_step(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image,
                       double* force, double* vel, uint32_t N_local, uint64_t index_offset,
                       double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params,
                       uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                       void* stream);

/* ---- host-buffer entry points (end-to-end path) ------------------------------------------------
 * Same results as cavb200_force + cavb200_bussi but every array is a HOST pointer: the library stages
 * through device buffers it owns (velocities in -> thermostat -> velocities out, overlapped with
 * positions / charges / images in -> force -> forces out).  This is what bench.py's "e2e" measures.
 * Pinned host memory (cavb200_host_alloc) gives full PCIe speed; pageable memory works but is slower.
 *   cavb200_step_host          synchronous: returns when outputs are on the host.
 *   cavb200_step_host_submit   asynchronous, staging slot 0..3: a driver holding several independent
 *                              systems on the host (the replicas of examples/05_advanced_run.py:1570-1612)
 *                              submits system k+1 before waiting for system k, so the next upload runs
 *                              under this download.  The host arrays must stay valid and untouched
 *                              until cavb200_step_host_wait(slot) returns; a slot is reusable after that.
 *   cavb200_step_host_wait     blocks until the slot's outputs are on the host; its energies
 *                              {harmonic, coupling, dipole self} and {KE, alpha, inst, cumulative, err}.
 * energies[3] and bussi_out[5] may be NULL.  The reservoir's cumulative energy is per HANDLE (it runs
 * over every step submitted, in submission order). */
int cavb200_step_host_submit(cavb200_handle* h, uint32_t slot, const double* pos, const double* charge,
                             const int32_t* image, double* force, double* vel, uint32_t N, double Lx, double Ly,
                             double Lz, uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                             uint32_t n_group, const cavb200_bussi_args* bussi);
int cavb200_step_host_wait(cavb200_handle* h, uint32_t slot, double energies[3], double bussi_out[5]);
/* The same with fewer bytes over PCIe.  flags:
 *   CAVB200_HOST_KEEP_CHARGE   the charges are unchanged since this slot's last submit (they never change in an MD run:
 *                              reference examples/05_advanced_run.py:502 sets them once): not uploaded, `charge` may be NULL
 *   CAVB200_HOST_KEEP_IMAGE    the same for the image flags (they change only when a particle crosses the box)
 *   CAVB200_HOST_RANK1_RESULT  the cavity force is rank-1, F_i = (-couplstr charge_i) Dq (reference
 *                              src/CavityForceCompute.cc:183,188-200): return {Dq[2], F_L[3], photon index} (and the
 *                              energies) through cavb200_step_host_wait_ex instead of the 32 B/particle force array
 *                              (`force` may be NULL; nothing is written per particle on the device either)
 * KEEP_* need an earlier submit of the same N on the slot (else cudaErrorInvalidValue).  Velocities and positions are
 * always moved.  rank1_out = {Dq.x, Dq.y, F_L.x, F_L.y, F_L.z, photon index}; may be NULL. */
#define CAVB200_HOST_KEEP_CHARGE 1u
#define CAVB200_HOST_KEEP_IMAGE 2u
#define CAVB200_HOST_RANK1_RESULT 4u
int cavb200_step_host_submit_ex(cavb200_handle* h, uint32_t slot, const double* pos, const double* charge,
                                const int32_t* image, double* force, double* vel, uint32_t N, double Lx, double Ly,
                                double Lz, uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                                uint32_t n_group, const cavb200_bussi_args* bussi, uint32_t flags);
int cavb200_step_host_wait_ex(cavb200_handle* h, uint32_t slot, double energies[3], double bussi_out[5],
                              double rank1_out[6]);
int cavb200_step_host(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image,
                      double* force, double* vel, uint32_t N, double Lx, double Ly, double Lz,
                      uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                      uint32_t n_group, const cavb200_bussi_args* bussi, double energies[3],
                      double bussi_out[5]);

/* ---- device/host memory helpers for harnesses that have no CUDA runtime of their own ------------
 * (tests/, bench.py and the ctypes host mirror use these; a HOOMD build never needs them). */
int cavb200_device_count(int* n);
int cavb200_dev_alloc(void** ptr, uint64_t bytes);
int cavb200_dev_free(void* ptr);
int cavb200_host_alloc(void** ptr, uint64_t bytes); /* pinned */
int cavb200_host_free(void* ptr);
int cavb200_memcpy_h2d(void* dst, const void* src, uint64_t bytes, void* stream);
int cavb200_memcpy_d2h(void* dst, const void* src, uint64_t bytes, void* stream);
int cavb200_memcpy_d2d(void* dst, const void* src, uint64_t bytes, void* stream);
int cavb200_memset(void* dst, int value, uint64_t bytes, void* stream);
int cavb200_stream_create(void** stream);
int cavb200_stream_destroy(void* stream);
int cavb200_stream_sync(void* stream);
int cavb200_device_sync(void);
/* CUDA-event timing on the launching stream (bench.py): */
int cavb200_event_create(void** ev);
int cavb200_event_destroy(void* ev);
int cavb200_event_record(void* ev, void* stream);
int cavb200_event_elapsed_ms(void* start, void* stop, float* ms); /* syncs on `stop` */
/* CUDA-graph capture of a fixed sequence of calls on `stream` (launch-bound inner loops): */
int cavb200_graph_begin(void* stream);
int cavb200_graph_end(void* stream, void** graph_exec);
int cavb200_graph_launch(void* graph_exec, void* stream);
int cavb200_graph_destroy(void* graph_exec);

#ifdef __cplusplus
}
#endif
#endif /* CAVB200_H */
