// track.cu -- device-side trackers (SURVEY.md 8f.4).
//
// The reference's per-step trackers each take a full device->host snapshot of the system every step
// (sim.state.cpu_local_snapshot: reference src/cavitymd/analysis.py:188,234 dipole autocorrelation,
// :1327 cavity mode, :535,578 energies) only to form a handful of scalars the force / thermostat kernels
// have already produced: the total dipole d (compute_total_dipole_moment, :18-31), the photon
// coordinate, the three cavity energies, the group's kinetic energy.  Here one 1-warp kernel per step
// appends a 128-byte record built from the handle's device-resident Scalars (plus the photon's
// velocity, the only per-particle datum needed) to a ring in device memory; the host reads the ring
// once per output period.  No snapshot, no synchronisation inside the step.
#include "hotpath.cuh"

namespace cavb
    {
// One record = CAVB200_TRACK_WORDS doubles (include/cavb200.h documents the layout).  sc: the Scalars of the handle that
// holds the force result; sb: those of the handle that ran the thermostat (nullptr: unknown, [12..14] are NaN); offset:
// the global index of vel[0], so that the photon's (global) index finds its row in a rank's local array.
__global__ void k_track_record(const Scalars* __restrict__ sc, const Scalars* __restrict__ sb, const double4* __restrict__ vel,
                               uint32_t N, unsigned long long offset, uint32_t flags, double timestep,
                               const double* __restrict__ ref, double* __restrict__ ring,
                               unsigned long long* __restrict__ count, unsigned long long capacity)
    {
    if (threadIdx.x != 0)
        return;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const bool pending = flags & CAVB200_TRACK_VELOCITIES_PENDING;
    const unsigned long long n = *count;
    double* r = ring + (n % capacity) * CAVB200_TRACK_WORDS;
    r[0] = timestep;
    double dd = 0.0;
    for (int k = 0; k < 3; k++)
        {
        const double d = sc->dipole[k];
        r[1 + k] = d;
        r[4 + k] = sc->q[k];
        r[7 + k] = sc->energies[k];
        // C(t) = d(0) . d(t), np.dot order x, y, z (analysis.py:222-224)
        dd = __dadd_rn(dd, __dmul_rn(ref[k], d));
        }
    r[10] = dd;
    // cavity-mode kinetic energy 1/2 m |v|^2 of the photon (analysis.py:1352-1354)
    double ke_ph = 0.0;
    const long long ph = sc->photon_idx;
    const unsigned long long local = (unsigned long long)ph - offset;
    if (vel && ph >= 0 && (unsigned long long)ph >= offset && local < N)
        {
        const double4 v = vel[local];
        const double v2 = __dadd_rn(__dadd_rn(__dmul_rn(v.x, v.x), __dmul_rn(v.y, v.y)), __dmul_rn(v.z, v.z));
        ke_ph = __dmul_rn(__dmul_rn(0.5, v.w), v2);
        }
    r[11] = pending ? nan : ke_ph;
    r[12] = sb && !pending ? sb->ke : nan;
    r[13] = sb ? sb->alpha : nan;
    r[14] = sb ? sb->cumulative : nan;
    r[15] = (double)ph;
    *count = n + 1;
    }

__global__ void k_track_set_reference(const Scalars* __restrict__ sc, double* __restrict__ ref)
    {
    if (threadIdx.x < 3)
        ref[threadIdx.x] = sc->dipole[threadIdx.x];
    }
    } // namespace cavb

using namespace cavb;

void cavb_track_release(cavb200_handle* h)
    {
    cudaFree(h->track_ring);
    h->track_ring = nullptr;
    h->track_capacity = 0;
    }

extern "C" int cavb200_track_open(cavb200_handle* h, uint32_t capacity)
    {
    if (!h || capacity == 0)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaSetDevice(h->device));
    cavb_track_release(h);
    // ring | reference dipole (4 doubles) | record counter
    const size_t bytes = (size_t)capacity * CAVB200_TRACK_WORDS * sizeof(double) + 4 * sizeof(double) + sizeof(unsigned long long);
    CAVB_CHECK(cudaMalloc((void**)&h->track_ring, bytes));
    CAVB_CHECK(cudaMemset(h->track_ring, 0, bytes));
    h->track_capacity = capacity;
    return 0;
    }

static double* track_ref(cavb200_handle* h) { return h->track_ring + (size_t)h->track_capacity * CAVB200_TRACK_WORDS; }
static unsigned long long* track_counter(cavb200_handle* h) { return reinterpret_cast<unsigned long long*>(track_ref(h) + 4); }

extern "C" int cavb200_track_set_reference_from(cavb200_handle* h, const cavb200_handle* src, void* stream)
    {
    if (!h || !h->track_ring || !src)
        return (int)cudaErrorInvalidValue;
    k_track_set_reference<<<1, 32, 0, (cudaStream_t)stream>>>(src->scalars, track_ref(h));
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

extern "C" int cavb200_track_set_reference(cavb200_handle* h, void* stream)
    {
    return cavb200_track_set_reference_from(h, h, stream);
    }

extern "C" int cavb200_track_record_from(cavb200_handle* h, const cavb200_handle* force_src, const cavb200_handle* bussi_src,
                                         uint64_t timestep, const double* vel, uint32_t N, uint32_t flags, void* stream)
    {
    if (!h || !h->track_ring || !force_src || (flags & ~CAVB200_TRACK_VELOCITIES_PENDING))
        return (int)cudaErrorInvalidValue;
    if (vel && (reinterpret_cast<uintptr_t>(vel) & 31))
        return (int)cudaErrorMisalignedAddress;
    k_track_record<<<1, 32, 0, (cudaStream_t)stream>>>(force_src->scalars, bussi_src ? bussi_src->scalars : nullptr,
                                                        reinterpret_cast<const double4*>(vel), N, force_src->index_offset,
                                                        flags, (double)timestep, track_ref(h), h->track_ring,
                                                        track_counter(h), h->track_capacity);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

extern "C" int cavb200_track_record(cavb200_handle* h, uint64_t timestep, const double* vel, uint32_t N, void* stream)
    {
    return cavb200_track_record_from(h, h, h, timestep, vel, N, 0, stream);
    }

extern "C" int cavb200_track_read(cavb200_handle* h, double* out, uint32_t max_records, uint32_t* n_out, uint64_t* total,
                                  void* stream)
    {
    if (!h || !h->track_ring || (!out && max_records) || !n_out)
        return (int)cudaErrorInvalidValue;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long cnt = 0;
    CAVB_CHECK(cudaMemcpyAsync(&cnt, track_counter(h), sizeof(cnt), cudaMemcpyDeviceToHost, s));
    CAVB_CHECK(cudaStreamSynchronize(s));
    const unsigned long long cap = h->track_capacity;
    unsigned long long have = cnt < cap ? cnt : cap; // records still in the ring
    if (have > max_records)
        have = max_records;
    // the newest `have` records, oldest first; the ring wraps at most once inside that span
    const unsigned long long first = cnt - have;
    const size_t rec = CAVB200_TRACK_WORDS * sizeof(double);
    unsigned long long done = 0;
    while (done < have)
        {
        const unsigned long long at = (first + done) % cap;
        unsigned long long run = cap - at;
        if (run > have - done)
            run = have - done;
        CAVB_CHECK(cudaMemcpyAsync(out + done * CAVB200_TRACK_WORDS, h->track_ring + at * CAVB200_TRACK_WORDS, run * rec,
                                   cudaMemcpyDeviceToHost, s));
        done += run;
        }
    CAVB_CHECK(cudaStreamSynchronize(s));
    *n_out = (uint32_t)have;
    if (total)
        *total = cnt;
    return 0;
    }
