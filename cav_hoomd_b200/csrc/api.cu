// api.cu -- the extern "C" surface of libcavb200.so: handle lifetime, argument checking and the
// translation of the C arguments into launches (include/cavb200.h documents every entry point and
// the reference interface it replaces).
#include "cavb200_internal.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

using namespace cavb;

namespace cavb
    {
// The constants the reference forms once per call on the host (CavityForceCompute.cc:174-183), in its
// operation order; IEEE double on both sides, so the device sees bit-identical values.
void fill_force_constants(ForceIn& f)
    {
    f.gk = f.g / f.K;
    f.half_K = 0.5 * f.K;
    f.half_g2K = 0.5 * (f.g * f.g / f.K);
    }

// BussiReservoirThermostat.h:186-214: everything that does not depend on the kinetic energy.
void fill_bussi_constants(BussiIn& b, const cavb200_bussi_args* a)
    {
    b.kT = a->kT;
    b.dof = a->dof;
    b.r_normal = a->r_normal;
    b.c = (a->tau != 0.0) ? exp(-a->deltaT / a->tau) : 0.0; // :186-190, host libm like the reference
    b.r_gamma = (a->dof > 1.0) ? 2.0 * a->gamma_draw : 0.0; // :195-200
    b.half_kT = a->kT / 2.0;                                // :202  set_T / 2.0 / K
    b.omc = 1.0 - b.c;
    b.gR2 = b.r_gamma + b.r_normal * b.r_normal;            // :203
    b.two_R = 2.0 * b.r_normal;                             // :204
    b.cdof = b.c * a->dof;                                  // :213  c * dof * K / ((1 - c) * K_bar)
    const double K_bar = a->kT * a->dof / 2.0;              // :212
    b.den = (1.0 - b.c) * K_bar;
    }

// HOOMD's TwoStepLangevin for one particle [HOOMD-upstream, not in the reference tree: restated from its definition]:
// coeff = sqrt(6 gamma kT / dt), left to right, host libm; the three products coeff * r_c are formed here too, so the
// device subtracts gamma v_c from bit-identical values
int fill_bath(BathIn& b, const cavb200_handle* h, const cavb200_langevin_args* a, double dt)
    {
    b = BathIn();
    b.bd = bath_slot(h);
    if (!a)
        return 0;
    if (!(a->gamma >= 0.0) || !(a->kT >= 0.0) || !(dt > 0.0))
        return (int)cudaErrorInvalidValue;
    const double coeff = sqrt(6.0 * a->gamma * a->kT / dt);
    b.gamma = a->gamma;
    for (int c = 0; c < 3; c++)
        b.cr[c] = coeff * a->r[c];
    return 0;
    }
    } // namespace cavb

namespace cavb
    {
int check_fault(cavb200_handle* h)
    {
    if (!h->fault_host || *(volatile unsigned long long*)h->fault_host == 0ull)
        return 0;
    // A persistent kernel of this handle gave up waiting for a CTA of its own grid: the grid was not co-resident,
    // i.e. something else (another stream, another process under MPS) held SM slots.  The outputs of that call were not
    // written.  From now on launch cooperatively -- the driver then guarantees co-residency -- and say so once.
    *(volatile unsigned long long*)h->fault_host = 0ull;
    h->tune.pdl = 0;
    h->faults += 1;
    return (int)cudaErrorLaunchTimeout;
    }

int fill_force(ForceIn& f, const double* pos, const double* charge, const int32_t* image, double* force, uint32_t N,
               double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* p, uint64_t index_offset,
               bool need_force)
    {
    if (!pos || !charge || !image || (need_force && !force) || !p)
        return (int)cudaErrorInvalidValue;
    if (misaligned(pos, 32) || misaligned(force, 32) || misaligned(charge, 8) || misaligned(image, 4))
        return (int)cudaErrorMisalignedAddress;
    f.pos = reinterpret_cast<const double4*>(pos);
    f.charge = charge;
    f.image = image;
    f.force = reinterpret_cast<double4*>(force);
    f.N = N;
    f.index_offset = index_offset;
    f.Lx = Lx;
    f.Ly = Ly;
    f.Lz = Lz;
    f.L_typeid = L_typeid;
    f.g = p->couplstr;
    f.K = p->K;
    fill_force_constants(f);
    return 0;
    }
    } // namespace cavb

namespace
    {
int fill_bussi(BussiIn& b, double* vel, const uint32_t* gidx, uint32_t first, uint32_t n, const cavb200_bussi_args* a,
               int rescale)
    {
    if ((n && !vel) || (rescale && !a))
        return (int)cudaErrorInvalidValue;
    if (n && (misaligned(vel, 32) || misaligned(gidx, 4)))
        return (int)cudaErrorMisalignedAddress;
    b.vel = reinterpret_cast<double4*>(vel);
    b.gidx = gidx;
    b.first = first;
    b.n = n;
    b.rescale = rescale;
    // rescaled velocities first-to-evict when one system's arrays (116 B/particle) exceed half of the 126 MB L2
    // (cavb200_internal.cuh st256_vel)
    b.stream_st = (uint64_t)n * 116ull > (63ull << 20);
    b.kT = b.c = b.dof = b.r_normal = b.r_gamma = 0.0;
    b.half_kT = b.omc = b.gR2 = b.two_R = b.cdof = b.den = 0.0;
    if (a)
        fill_bussi_constants(b, a);
    return 0;
    }
    } // namespace

extern "C"
    {
int cavb200_version(void) { return CAVB200_VERSION; }

const char* cavb200_error_string(int err) { return cudaGetErrorString((cudaError_t)err); }

int cavb200_device_count(int* n)
    {
    if (!n)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaGetDeviceCount(n));
    return 0;
    }

int cavb200_create(cavb200_handle** out, int device)
    {
    if (!out)
        return (int)cudaErrorInvalidValue;
    *out = nullptr;
    CAVB_CHECK(cudaSetDevice(device));
    cavb200_handle* h = (cavb200_handle*)calloc(1, sizeof(cavb200_handle));
    if (!h)
        return (int)cudaErrorMemoryAllocation;
    h->device = device;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess)
        {
        free(h);
        return (int)e;
        }
    h->num_sms = prop.multiProcessorCount;
    h->coop_supported = prop.cooperativeLaunch;
    if ((e = cudaMalloc((void**)&h->partials, sizeof(Partial) * MAX_PARTIALS)) != cudaSuccess
        || (e = cudaMalloc((void**)&h->scalars, sizeof(Scalars))) != cudaSuccess
        || (e = cudaMalloc((void**)&h->counters, 1024)) != cudaSuccess
        || (e = cudaMalloc((void**)&h->stamps, 8 * sizeof(unsigned long long) * MAX_PARTIALS)) != cudaSuccess
        || (e = cudaMemset(h->scalars, 0, sizeof(Scalars))) != cudaSuccess
        || (e = cudaMemset(h->counters, 0, 1024)) != cudaSuccess
        || (e = cudaMemset(h->partials, 0, sizeof(Partial) * MAX_PARTIALS)) != cudaSuccess)
        {
        cavb200_destroy(h);
        return (int)e;
        }
    // the fault word: pinned host memory the kernels can store to (Scalars::fault), read by check_fault without a sync
    if ((e = cudaHostAlloc((void**)&h->fault_host, 64, cudaHostAllocMapped | cudaHostAllocPortable)) != cudaSuccess)
        {
        cavb200_destroy(h);
        return (int)e;
        }
    *h->fault_host = 0ull;
        {
        unsigned long long* dptr = nullptr;
        if ((e = cudaHostGetDevicePointer((void**)&dptr, h->fault_host, 0)) != cudaSuccess
            || (e = cudaMemcpy(&h->scalars->fault, &dptr, sizeof(dptr), cudaMemcpyHostToDevice)) != cudaSuccess)
            {
            cavb200_destroy(h);
            return (int)e;
            }
        }
    h->tune.variant = 3; // split-phase step kernel with a folder CTA; force-only / Bussi-only calls use the fused kernel (variant 1)
    h->tune.threads = 384;
    h->tune.ctas_per_sm = 2;
    h->tune.unroll = 2;
    h->tune.pdl = 1;
    h->tune.auto_threads = 1;
    h->tune.small_n = 768;
    h->tune.cluster_n = 8192;
    h->tune.cluster_ctas = cluster_kernels_init();
    h->shard.mode = 0;
    h->shard.nranks = 1;
    *out = h;
    return 0;
    }

int cavb200_destroy(cavb200_handle* h)
    {
    if (!h)
        return 0;
    cudaSetDevice(h->device);
    cavb_shard_release(h);
    cavb_host_release(h);
    cavb_track_release(h);
    cavb_fkt_track_release(h);
    cudaFree(h->partials);
    cudaFree(h->scalars);
    cudaFree(h->counters);
    cudaFree(h->stamps);
    cudaFree(h->rhok_partials);
    cudaFree(h->rhok_table);
    cudaFree(h->group_mask);
    if (h->fault_host)
        cudaFreeHost(h->fault_host);
    free(h);
    return 0;
    }

uint64_t cavb200_launch_count(const cavb200_handle* h) { return h ? h->launches : 0; }
uint64_t cavb200_fault_count(const cavb200_handle* h) { return h ? h->faults : 0; }

int cavb200_debug_stamps(cavb200_handle* h, uint64_t* out, uint32_t n_ctas)
    {
    if (!h || !out || n_ctas > (uint32_t)MAX_PARTIALS)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaMemcpy(out, h->stamps, 8ull * sizeof(unsigned long long) * n_ctas, cudaMemcpyDeviceToHost));
    return 0;
    }

static int* tuning_slot(cavb::Tuning* t, const char* key)
    {
    if (!strcmp(key, "variant")) return &t->variant;
    if (!strcmp(key, "threads")) return &t->threads;
    if (!strcmp(key, "ctas_per_sm")) return &t->ctas_per_sm;
    if (!strcmp(key, "unroll")) return &t->unroll;
    if (!strcmp(key, "stamps")) return &t->stamps;
    if (!strcmp(key, "pdl")) return &t->pdl;
    if (!strcmp(key, "ke_first")) return &t->ke_first;
    if (!strcmp(key, "auto_threads")) return &t->auto_threads;
    if (!strcmp(key, "md_shape")) return &t->md_shape;
    if (!strcmp(key, "small_n")) return &t->small_n;
    if (!strcmp(key, "cluster_n")) return &t->cluster_n;
    if (!strcmp(key, "cluster_ctas")) return &t->cluster_ctas;
    if (!strcmp(key, "rhok_threads")) return &t->rhok_threads;
    return nullptr;
    }

int cavb200_set_tuning(cavb200_handle* h, const char* key, int value)
    {
    if (!h || !key)
        return (int)cudaErrorInvalidValue;
    int* slot = tuning_slot(&h->tune, key);
    if (!slot)
        return (int)cudaErrorInvalidValue;
    if (!strcmp(key, "threads") && (value < 32 || value > 1024 || (value & 31)))
        return (int)cudaErrorInvalidValue;
    if (!strcmp(key, "ctas_per_sm") && (value < 1 || value > 32))
        return (int)cudaErrorInvalidValue;
    if (!strcmp(key, "unroll") && value != 2 && value != 4 && value != 8)
        return (int)cudaErrorInvalidValue;
    *slot = value;
    if (!strcmp(key, "threads"))
        h->tune.auto_threads = 0; // an explicit CTA size switches the automatic choice off (set auto_threads = 1 to re-enable)
    return 0;
    }

int cavb200_get_tuning(const cavb200_handle* h, const char* key, int* value)
    {
    if (!h || !key || !value)
        return (int)cudaErrorInvalidValue;
    int* slot = tuning_slot(const_cast<cavb::Tuning*>(&h->tune), key);
    if (!slot)
        return (int)cudaErrorInvalidValue;
    *value = *slot;
    return 0;
    }

// ---- cavity force ----------------------------------------------------------------------------
int cavb200_force(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image, double* force,
                  uint32_t N, double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params,
                  void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (const int fault = check_fault(h))
        return fault;
    if (N == 0)
        return 0;
    ForceIn f;
    int rc = fill_force(f, pos, charge, image, force, N, Lx, Ly, Lz, L_typeid, params, 0);
    if (rc)
        return rc;
    h->index_offset = 0;
    return launch_hotpath(h, &f, nullptr, (cudaStream_t)stream);
    }

int cavb200_force_rank1(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image, uint32_t N,
                        double Lx, double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (const int fault = check_fault(h))
        return fault;
    if (N == 0)
        return 0;
    ForceIn f;
    int rc = fill_force(f, pos, charge, image, nullptr, N, Lx, Ly, Lz, L_typeid, params, 0, false);
    if (rc)
        return rc;
    h->index_offset = 0;
    return launch_hotpath(h, &f, nullptr, (cudaStream_t)stream);
    }

int cavb200_rank1_read(cavb200_handle* h, double Dq[2], double F_L[3], int32_t* photon_idx, uint32_t* n_L, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    Scalars s;
    CAVB_CHECK(cudaMemcpyAsync(&s, h->scalars, sizeof(Scalars), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CAVB_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    for (int k = 0; k < 3; k++)
        {
        if (Dq && k < 2)
            Dq[k] = s.Dq[k];
        if (F_L)
            F_L[k] = s.FL[k];
        }
    if (photon_idx)
        *photon_idx = (int32_t)s.photon_idx;
    if (n_L)
        *n_L = s.n_L;
    return 0;
    }

int cavb200_force_read(cavb200_handle* h, double energies[3], double dipole[3], int32_t* photon_idx, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    Scalars s;
    CAVB_CHECK(cudaMemcpyAsync(&s, h->scalars, sizeof(Scalars), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CAVB_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    if (s.err_force == 2.0)
        return (int)cudaErrorLaunchTimeout;
    for (int k = 0; k < 3; k++)
        {
        if (energies)
            energies[k] = s.energies[k];
        if (dipole)
            dipole[k] = s.dipole[k];
        }
    if (photon_idx)
        *photon_idx = (int32_t)s.photon_idx;
    return 0;
    }

// ---- Bussi -----------------------------------------------------------------------------------
int cavb200_bussi(cavb200_handle* h, double* vel, const uint32_t* group_idx, uint32_t group_first, uint32_t n,
                  const cavb200_bussi_args* args, void* stream)
    {
    if (!h || !args)
        return (int)cudaErrorInvalidValue;
    if (const int fault = check_fault(h))
        return fault;
    if (args->deltaT == 0.0) // BussiReservoirThermostat.h:45-48: {1,1}, nothing else happens
        return 0;
    BussiIn b;
    int rc = fill_bussi(b, vel, group_idx, group_first, n, args, 1);
    if (rc)
        return rc;
    return launch_hotpath(h, nullptr, &b, (cudaStream_t)stream);
    }

int cavb200_bussi_ke(cavb200_handle* h, const double* vel, const uint32_t* group_idx, uint32_t group_first, uint32_t n,
                     void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (const int fault = check_fault(h))
        return fault;
    BussiIn b;
    int rc = fill_bussi(b, const_cast<double*>(vel), group_idx, group_first, n, nullptr, 0);
    if (rc)
        return rc;
    return launch_hotpath(h, nullptr, &b, (cudaStream_t)stream);
    }

int cavb200_bussi_read(cavb200_handle* h, double out[5], void* stream)
    {
    if (!h || !out)
        return (int)cudaErrorInvalidValue;
    Scalars s;
    CAVB_CHECK(cudaMemcpyAsync(&s, h->scalars, sizeof(Scalars), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CAVB_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    out[0] = s.ke;
    out[1] = s.alpha;
    out[2] = s.inst;
    out[3] = s.cumulative;
    out[4] = s.err;
    return 0;
    }

int cavb200_bussi_reset(cavb200_handle* h, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    // zero {inst, cumulative, err}: BussiReservoirThermostat.h:153-159
    CAVB_CHECK(cudaMemsetAsync(&h->scalars->inst, 0, 3 * sizeof(double), (cudaStream_t)stream));
    return 0;
    }

// ---- fused step ------------------------------------------------------------------------------
int cavb200_step(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image, double* force,
                 double* vel, uint32_t N, double Lx, double Ly, double Lz, uint32_t L_typeid,
                 const cavb200_params* params, uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                 void* stream)
    {
    if (!h || !bussi)
        return (int)cudaErrorInvalidValue;
    if (const int fault = check_fault(h))
        return fault;
    if (N == 0)
        return 0;
    if ((unsigned long long)group_first + n_group > N)
        return (int)cudaErrorInvalidValue;
    ForceIn f;
    int rc = fill_force(f, pos, charge, image, force, N, Lx, Ly, Lz, L_typeid, params, 0);
    if (rc)
        return rc;
    h->index_offset = 0;
    if (bussi->deltaT == 0.0)
        return launch_hotpath(h, &f, nullptr, (cudaStream_t)stream);
    BussiIn b;
    rc = fill_bussi(b, vel, nullptr, group_first, n_group, bussi, 1);
    if (rc)
        return rc;
    return launch_hotpath(h, &f, &b, (cudaStream_t)stream);
    }

// ---- memory / stream / event / graph helpers ---------------------------------------------------
int cavb200_dev_alloc(void** ptr, uint64_t bytes)
    {
    if (!ptr)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaMalloc(ptr, bytes ? bytes : 1));
    return 0;
    }
int cavb200_dev_free(void* ptr) { return (int)cudaFree(ptr); }
int cavb200_host_alloc(void** ptr, uint64_t bytes)
    {
    if (!ptr)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaMallocHost(ptr, bytes ? bytes : 1));
    return 0;
    }
int cavb200_host_free(void* ptr) { return (int)cudaFreeHost(ptr); }
int cavb200_memcpy_h2d(void* dst, const void* src, uint64_t bytes, void* stream)
    {
    return (int)cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
    }
int cavb200_memcpy_d2h(void* dst, const void* src, uint64_t bytes, void* stream)
    {
    return (int)cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    }
int cavb200_memcpy_d2d(void* dst, const void* src, uint64_t bytes, void* stream)
    {
    return (int)cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    }
int cavb200_memset(void* dst, int value, uint64_t bytes, void* stream)
    {
    return (int)cudaMemsetAsync(dst, value, bytes, (cudaStream_t)stream);
    }
int cavb200_stream_create(void** stream)
    {
    if (!stream)
        return (int)cudaErrorInvalidValue;
    cudaStream_t s;
    CAVB_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = (void*)s;
    return 0;
    }
int cavb200_stream_destroy(void* stream) { return (int)cudaStreamDestroy((cudaStream_t)stream); }
int cavb200_stream_sync(void* stream) { return (int)cudaStreamSynchronize((cudaStream_t)stream); }
int cavb200_device_sync(void) { return (int)cudaDeviceSynchronize(); }

int cavb200_event_create(void** ev)
    {
    if (!ev)
        return (int)cudaErrorInvalidValue;
    cudaEvent_t e;
    CAVB_CHECK(cudaEventCreate(&e));
    *ev = (void*)e;
    return 0;
    }
int cavb200_event_destroy(void* ev) { return (int)cudaEventDestroy((cudaEvent_t)ev); }
int cavb200_event_record(void* ev, void* stream) { return (int)cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)stream); }
int cavb200_event_elapsed_ms(void* start, void* stop, float* ms)
    {
    CAVB_CHECK(cudaEventSynchronize((cudaEvent_t)stop));
    return (int)cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop);
    }

int cavb200_graph_begin(void* stream)
    {
    return (int)cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal);
    }
int cavb200_graph_end(void* stream, void** graph_exec)
    {
    if (!graph_exec)
        return (int)cudaErrorInvalidValue;
    cudaGraph_t g;
    CAVB_CHECK(cudaStreamEndCapture((cudaStream_t)stream, &g));
    cudaGraphExec_t ge;
    cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess)
        return (int)e;
    *graph_exec = (void*)ge;
    return 0;
    }
int cavb200_graph_launch(void* graph_exec, void* stream)
    {
    return (int)cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream);
    }
int cavb200_graph_destroy(void* graph_exec) { return (int)cudaGraphExecDestroy((cudaGraphExec_t)graph_exec); }
    }
