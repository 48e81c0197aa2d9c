// cavb200_internal.cuh -- handle, device-resident scalar blocks and small device helpers shared
// by the translation units of libcavb200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cavb200.h"

#define CAVB_CHECK(expr)                       \
    do                                         \
        {                                      \
        cudaError_t _e = (expr);               \
        if (_e != cudaSuccess)                 \
            return (int)_e;                    \
        } while (0)

namespace cavb
    {
constexpr uint32_t NO_INDEX = 0xFFFFFFFFu;
constexpr unsigned long long HANDOFF_TIMEOUT_NS = 50000000ull; // 50 ms: a co-resident grid hands off in microseconds
constexpr unsigned long long PEER_TIMEOUT_NS = 2000000000ull;  // 2 s: peer ranks may start late
constexpr int MAX_PARTIALS = 2048; // upper bound on the grid of a reduce pass
// stamps buffer (8 * MAX_PARTIALS u64): [0, 8192) per-CTA phase stamps, [8192, 12288) their second bank,
// [12288, 16384) the per-launch ring of {start, end} pairs (tuning stamps = 2)
constexpr unsigned long long LAUNCH_RING_OFFSET = 12288ull;
constexpr unsigned long long LAUNCH_RING = 2048ull;

// One reduce-pass record per CTA (and, in sharded mode, per rank): 160 bytes = five 32-byte sectors,
// each written with ONE STG.256 and read with ONE LDG.256.  Every sector carries three payload words
// and a check word  w = epoch ^ payload0 ^ payload1 ^ payload2  (bitwise), so a reader can tell a
// complete sector of THIS launch from a stale or torn one without any fence or flag: the hand-off
// between the reduce and apply halves of the cooperative kernel is "store the sectors / poll the
// sectors".  It relies only on 8-byte access atomicity; a torn or stale sector passes the check
// with probability 2^-64.  The common path of the combine reads sectors 0-2 (2 only for the
// thermostat); 3 is read by the one thread whose record holds the photon, 4 only when more than
// one particle of type 'L' exists.
// d is carried as unevaluated (hi, lo) pairs so that combining is (nearly) exact and therefore
// independent of how many CTAs / ranks took part up to the final rounding.
constexpr unsigned long long MULTI_L_BIT = 1ull << 63; // in first_L: "this record saw more than one 'L'"
struct __align__(32) Partial
    {
    double dhi[3];
    unsigned long long w0;
    double dlo[3];
    unsigned long long w1;
    double ke;                  // sum m |v|^2 (NOT halved)
    unsigned long long first_L; // GLOBAL index of the first 'L' particle seen (| MULTI_L_BIT), ~0ull if none
    unsigned long long n_L;     // number of 'L' particles seen (0, 1, or "2 = more than one" after a merge)
    unsigned long long w2;
    double q[3];                // unwrapped position of that first 'L' particle
    unsigned long long w3;
    double t[3];                // its dipole term charge*u (goes back into d if it is not the global first)
    unsigned long long w4;
    };
static_assert(sizeof(Partial) == CAVB200_SHARD_RECORD_BYTES, "record size is part of the ABI");

// Device-resident results of the last call; host getters copy this back lazily.
struct __align__(16) Scalars
    {
    // cavity force
    double energies[3];  // harmonic, coupling, dipole self
    double dipole[3];
    double Dq[2];
    double q[3];
    double FL[3];
    long long photon_idx; // global index, -1 if none
    unsigned int n_L;
    unsigned int pad0;
    // Bussi
    double ke;           // 1/2 sum m|v|^2 seen by the last call
    double alpha;
    double inst;         // instantaneous reservoir energy  KE (1 - alpha^2)
    double cumulative;   // running sum of inst
    double err;          // thermostat status of the LAST call that published KE / alpha: 0 ok, 1 = zero kinetic energy with dof != 0, 2 = hand-off timeout
    double err_force;    // cavity-force status of the LAST call that published a dipole: 0 ok, 2 = hand-off timeout
    // host-mapped (pinned) word a kernel sets when a hand-off between co-resident CTAs timed out; the host looks at it
    // at the top of every compute call without any synchronisation (api.cu check_fault)
    unsigned long long* fault;
    double pad1[1];
    };

struct Tuning
    {
    int variant;         // 0 = reduce kernel + apply kernel, 1 = fused persistent kernel, 2 = split-phase step kernel, 3 = split-phase with a folder CTA (default)
    int threads;         // CTA size of the streaming kernels (256 / 512 / 1024)
    int ctas_per_sm;     // resident CTAs per SM the grid is sized for
    int unroll;          // independent particle loads in flight per thread (1, 2 or 4)
    int pdl;             // 1: launch with programmatic stream serialization (hides the launch gap; co-residency of the persistent
                         //    grids by construction on a device this stream has to itself); 0: cooperative launch (the driver
                         //    guarantees co-residency, ~2 us per launch slower).  Switched to 0 by the library after a fault.
    int stamps;          // 1: debug, per-CTA phase timestamps of the persistent kernels; 2: per-launch {start, end} ring
    int md_shape;        // cavb200_md_step_fused launch shape: 0 = one 768-thread CTA per SM (default), 1 = two 384-thread CTAs
    int auto_threads;    // step kernel: pick 320 / 352 / 384 threads per CTA from the particle count (1) or use `threads` (0)
    int ke_first;        // folder step kernel: thermostat half first (1) or dipole half first (0)
    int small_n;         // calls over at most this many particles run as ONE CTA with no inter-CTA hand-off (0: off)
    int cluster_n;       // ... and, for calls that include the force, up to this many as ONE thread-block cluster of 16 CTAs:
                         //     hardware barrier instead of polled records (0: off; with a cluster of 8, half as many)
    int rhok_threads;    // k_rhok CTA size: 128 or 256; any other value (0 included) means 256
    int cluster_ctas;    // CTAs of that cluster (16 = non-portable size; the launcher falls back to 8 if the device refuses it)
    };

struct ShardState
    {
    int mode;            // 0 nccl, 1 nvlink mailbox
    int rank, nranks;
    void* nccl_comm;
    Partial* gather;     // device, nranks records (nccl all-gather target / local mailbox)
    Partial* peer_mailbox[16]; // IPC-mapped mailbox base of every rank (own entry = local)
    unsigned long long* flags;      // device, per-rank arrival sequence numbers (inside mailbox allocation)
    unsigned long long* peer_flags[16];
    void* mailbox_alloc;
    unsigned long long seq;
    };
    } // namespace cavb

#define CAVB_HOST_SLOTS 4

struct cavb200_handle
    {
    int device;
    int num_sms;
    int coop_supported;
    cavb::Partial* partials;          // MAX_PARTIALS records
    cavb::Scalars* scalars;           // 1 record
    unsigned long long* counters;     // [2] hand-off epoch, [4] reduce-pass ticket, [8..] Final (variant 0), [32..] Final (rank-1),
                                      // [48] cavb200_group_set check word, [49..51] cavb200_rank1_reindex {first, count, ticket},
                                      // [56..58] the photon's Langevin bath force bd[3] (double)
    uint64_t launches;
    uint64_t faults;                  // hand-off timeouts seen so far (each one switched the handle to cooperative launches)
    unsigned long long* fault_host;   // pinned + mapped: the word Scalars::fault points at
    unsigned long long* stamps;       // MAX_PARTIALS x 8 timestamps (debug)
    cavb::Tuning tune;
    cavb::ShardState shard;
    // host-buffer pipeline staging (grown on demand, owned)
    void* stage[CAVB_HOST_SLOTS][5];
    uint64_t stage_bytes[CAVB_HOST_SLOTS][5];
    cudaStream_t copy_streams[3];     // copy-in, kernels, copy-out
    cudaEvent_t copy_events[64];
    int copy_ready;
    int slot_used[CAVB_HOST_SLOTS];
    uint32_t slot_N[CAVB_HOST_SLOTS];  // particle count of the slot's last submit (KEEP_* flags)
    cavb::Scalars* slot_scalars;      // device, one per slot
    cavb::Scalars* slot_scalars_host; // pinned, one per slot
    // device-side tracker ring (track.cu): records | reference dipole | counter
    double* track_ring;
    uint64_t track_capacity;
    // F(k,t) workspace
    double* rhok_partials;
    uint64_t rhok_partials_bytes;
    void* rhok_table; // device, (cos, sin)(2 pi e / 512) as double2 (rhok.cu)
    // F(k,t) tracker (rhok.cu, cavb200_fkt_track_*): one allocation holding the wave vectors [3K] | rho slot [2K] |
    // stored references [max_refs][2K] | ring [capacity][2 + max_refs + 2K] | record counter; the reference count is
    // kept here on the host
    double* fkt_track;
    uint32_t fkt_K, fkt_max_refs, fkt_n_refs;
    uint64_t fkt_capacity;
    // thermostatted group as a bit mask (cavb200_group_set), used by the window entry points with CAVB200_GROUP_MASK
    uint32_t* group_mask;             // device, ceil(N / 32) words
    uint64_t group_mask_words;        // allocated words
    uint32_t group_n, group_N;        // members and particle count the mask was built for
    int group_ready;                  // the last cavb200_group_set succeeded
    };

namespace cavb
    {
// ---- 256-bit global accesses (PTX ISA 8.8, sm_100+): one LDG.E.256 / STG.E.256 per Scalar4 ----
__device__ __forceinline__ double4 ld256_stream(const double4* p)
    {
    double4 r;
    // read once per step: do not keep it in L1, and mark it first to leave L2 (the 126 MB L2 is wanted
    // for the charge / velocity lines the apply pass reads again and for the dirty output lines)
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w)
                 : "l"(p));
    return r;
    }
// streaming read of data that this kernel later overwrites (velocities): no L1 allocation, but not
// .nc (the non-coherent path requires the data to be read-only for the whole kernel)
__device__ __forceinline__ double4 ld256_na(const double4* p)
    {
    double4 r;
    // (an L2::evict_last hint here was measured and dropped: with several systems in flight the
    // pinned-but-dead velocity lines of earlier calls crowd L2; Bussi went from 17.8 to 19.5 us)
    asm volatile("ld.global.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w)
                 : "l"(p)
                 : "memory");
    return r;
    }
__device__ __forceinline__ double4 ld256(const double4* p)
    {
    double4 r;
    asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w)
                 : "l"(p)
                 : "memory");
    return r;
    }
__device__ __forceinline__ double4 ld256_cg(const double4* p)
    {
    double4 r;
    asm volatile("ld.relaxed.gpu.global.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w)
                 : "l"(p)
                 : "memory");
    return r;
    }
__device__ __forceinline__ double4 ld256_sys(const double4* p)
    {
    double4 r;
    asm volatile("ld.relaxed.sys.global.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w)
                 : "l"(p)
                 : "memory");
    return r;
    }
__device__ __forceinline__ void st256(double4* p, const double4& v)
    {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w)
                 : "memory");
    }
// output nobody in this library reads again (the force array)
__device__ __forceinline__ void st256_stream(double4* p, const double4& v)
    {
    asm volatile("st.global.L2::evict_first.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w)
                 : "memory");
    }
// Rescaled velocities.  Measured (profiles/cache_policy_r2a.txt): marking these dirty lines first-to-evict lets the
// write-back start early instead of competing with the next pass's reads -- 1M-particle step 30.9 -> 30.0 us, force +
// Bussi 38.9 -> 37.6 us, 4M Bussi call 62.7 -> 58.3 us.  When several systems that together fit in L2 are cycled
// through (262k particles x 4) it costs reuse instead (17.0 -> 18.3 us), so the launcher sets `ef` only when one
// system's arrays alone exceed half of L2.  (evict_last, and default / .cs / evict_last for the force stores: slower.)
__device__ __forceinline__ void st256_vel(double4* p, const double4& v, bool ef)
    {
    if (ef)
        asm volatile("st.global.L2::evict_first.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w)
                     : "memory");
    else
        asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w) : "memory");
    }
// image flags: read once per call
#ifndef CAVB_IMAGE_LD
#define CAVB_IMAGE_LD 1 // 0: __ldg, 1: evict_first cache policy (force call 22.1 -> 21.6 us at 1M, profiles/cache_policy_r2a.txt)
#endif
__device__ __forceinline__ int ld_image(const int* p)
    {
#if CAVB_IMAGE_LD == 1
    // (the L2::evict_first qualifier exists for 256-bit accesses only; narrower ones take a cache-policy operand)
    int r;
    asm volatile("{ .reg .b64 pol; createpolicy.fractional.L2::evict_first.b64 pol, 1.0;\n"
                 "ld.global.nc.L2::cache_hint.s32 %0, [%1], pol; }" : "=r"(r) : "l"(p));
    return r;
#else
    return __ldg(p);
#endif
    }
// charges of the apply pass (their second and last use in a call)
#ifndef CAVB_CHARGE2_LD
#define CAVB_CHARGE2_LD 1 // 0: __ldg, 1: evict_first cache policy (profiles/cache_policy_r2a.txt)
#endif
__device__ __forceinline__ double ld_charge_last(const double* p)
    {
#if CAVB_CHARGE2_LD == 1
    double r;
    asm volatile("{ .reg .b64 pol; createpolicy.fractional.L2::evict_first.b64 pol, 1.0;\n"
                 "ld.global.nc.L2::cache_hint.f64 %0, [%1], pol; }" : "=d"(r) : "l"(p));
    return r;
#else
    return __ldg(p);
#endif
    }

// programmatic dependent launch: wait for the previous kernel of the stream / let the next one start
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// thread-block cluster: rank and size of this CTA's cluster, and the hardware barrier over all its threads (release /
// acquire at cluster scope: what a thread wrote before it, to global memory too, is visible to every thread after it)
__device__ __forceinline__ unsigned int cluster_ctarank()
    {
    unsigned int r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
    }
__device__ __forceinline__ unsigned int cluster_nctarank()
    {
    unsigned int r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
    }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// store 8 bytes into the shared memory of CTA `peer` of this cluster, at the address `local` has in this CTA
__device__ __forceinline__ void st_dsmem_f64(const void* local, unsigned int peer, double v)
    {
    const unsigned int a = (unsigned int)__cvta_generic_to_shared(local);
    unsigned int dst;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(a), "r"(peer));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(dst), "d"(v) : "memory");
    }
__device__ __forceinline__ void cluster_sync()
    {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p)
    {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
    }
__device__ __forceinline__ unsigned long long atom_acq_rel_add_u64(unsigned long long* p, unsigned long long v)
    {
    unsigned long long old;
    asm volatile("atom.acq_rel.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
    }
// NOTE (measured, round 1): polling with a weak ld.global.cg does NOT work on sm_100 -- a thread
// whose first poll missed kept reading the stale value until the 2 s guard fired.  Polls and record
// reads therefore use strong (relaxed, gpu-scope) loads.
// a hand-off timed out: tell the host (system-scope store into pinned memory; cold path)
__device__ __forceinline__ void raise_fault(const Scalars* s)
    {
#ifdef CAVB_NO_FAULT // (A/B builds only, tools/build_exp.sh)
    return;
#endif
    unsigned long long* f = s->fault;
    if (f)
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(f), "l"(1ull) : "memory");
    }
__device__ __forceinline__ unsigned long long globaltimer_ns()
    {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
    }

// ---- compensated accumulation: (hi, lo) is an unevaluated sum; error-free transforms only ----
__device__ __forceinline__ void two_sum_acc(double& hi, double& lo, double t)
    {
    const double s = __dadd_rn(hi, t);
    const double bb = __dadd_rn(s, -hi);
    const double e = __dadd_rn(__dadd_rn(hi, -__dadd_rn(s, -bb)), __dadd_rn(t, -bb));
    hi = s;
    lo = __dadd_rn(lo, e);
    }
__device__ __forceinline__ void pair_add(double& hi, double& lo, double hi2, double lo2)
    {
    two_sum_acc(hi, lo, hi2);
    lo = __dadd_rn(lo, lo2);
    }

__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
    } // namespace cavb

// teardown hooks of the sharded and host-buffer paths (shard.cu, host.cu)
void cavb_shard_release(cavb200_handle* h);
void cavb_host_release(cavb200_handle* h);
void cavb_track_release(cavb200_handle* h);
void cavb_fkt_track_release(cavb200_handle* h);

// launch helpers implemented in the .cu files
namespace cavb
    {
struct ForceIn
    {
    const double4* pos;
    const double* charge;
    const int* image;
    double4* force;
    uint32_t N;
    unsigned long long index_offset; // global index of particle 0 (sharded mode)
    double Lx, Ly, Lz;
    uint32_t L_typeid;
    double g, K;
    // host-evaluated constants, same operation order as the reference (CavityForceCompute.cc:174-183)
    double gk;       // g / K
    double half_K;   // 0.5 * K
    double half_g2K; // 0.5 * (g*g / K)
    };
struct BussiIn
    {
    double4* vel;
    const uint32_t* gidx;
    uint32_t first, n;
    double kT, c /* exp(-dt/tau), host-evaluated */, dof, r_normal, r_gamma /* already doubled */;
    // host-evaluated pieces of compute_rescale_factor that do not depend on KE
    // (BussiReservoirThermostat.h:202-214, same operation order)
    double half_kT;  // kT / 2.0
    double omc;      // 1.0 - c
    double gR2;      // r_gamma + R*R
    double two_R;    // 2.0 * R
    double cdof;     // c * dof
    double den;      // (1.0 - c) * (kT * dof / 2.0)
    int rescale;         // 0: KE only
    int stream_st;       // rescaled velocities are stored first-to-evict (set by the launcher for systems larger than L2/2)
    };

void fill_force_constants(ForceIn& f);
inline bool misaligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; }
// ForceIn of one call from the entry point's arguments (api.cu): cudaErrorInvalidValue for a NULL pointer or params,
// cudaErrorMisalignedAddress for a pointer off its alignment (pos, force 32 B; charge 8 B; image 4 B)
int fill_force(ForceIn& f, const double* pos, const double* charge, const int32_t* image, double* force, uint32_t N,
               double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* p, uint64_t index_offset,
               bool need_force = true);
// device slot of the Final record cavb200_force_rank1 leaves for the rank-1 consumers (nve.cu); apart
// from the variant-0 slot at counters + 8, which every reduce-only launch overwrites
struct Final;
inline const Final* rank1_final(const cavb200_handle* h) { return reinterpret_cast<const Final*>(h->counters + 32); }
void fill_bussi_constants(BussiIn& b, const cavb200_bussi_args* a);
// The cavity mode's Langevin bath as the harness kernels take it (nve.cu, BATH): bd = cr - gamma v of the photon, with
// cr_c = coeff r_c and coeff = sqrt(6 gamma kT / dt) formed once on the host (api.cu fill_bath); bd points at the handle's
// slot that holds the bath force of the last step two
struct BathIn
    {
    double gamma;
    double cr[3];
    double* bd;
    };
// device slot of the bath force bd[3] (zero at cavb200_create)
inline double* bath_slot(const cavb200_handle* h) { return reinterpret_cast<double*>(h->counters + 56); }
// BathIn of one call: a = NULL gives the slot alone (step one reads the stored bd); cudaErrorInvalidValue for gamma < 0,
// kT < 0 or dt <= 0
int fill_bath(BathIn& b, const cavb200_handle* h, const cavb200_langevin_args* a, double dt);
int launch_hotpath(cavb200_handle* h, const ForceIn* f, const BussiIn* b, cudaStream_t s);
int cluster_kernels_init();
int launch_shard_step(cavb200_handle* h, const ForceIn* f, const BussiIn* b, cudaStream_t s);
// top of every compute entry point: a hand-off timeout reported by an earlier launch (Scalars::fault) switches the handle
// to cooperative launches for good and is returned ONCE as cudaErrorLaunchTimeout
int check_fault(cavb200_handle* h);
    } // namespace cavb
